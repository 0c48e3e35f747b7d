// visual_inertial_pnp on the GPU: the whole ceres::Solve of pvio/src/pvio/estimation/pnp.cpp:32-100
// in ONE kernel launch (SURVEY.md 8f rank 2, the other ceres::Solve of PVIO's per-frame loop).
//
// The problem is tiny -- 15 unknowns (pose + v, bg, ba of the new frame; 6 without inertial), one
// PreIntegrationPriorCost (estimation/ceres/preintegration_error_cost.h:167-206) and ~150
// PoseOnly reprojection blocks on constant world points
// (estimation/ceres/reprojection_error_cost.h:128-203, CauchyLoss(1.0)) -- so it is launch- and
// latency-bound: a single CTA keeps the state, the 15x15 normal equations and the trust-region
// variables in shared memory and runs every iteration of TrustRegionMinimizer + TRADITIONAL_DOGLEG
// (Ceres 1.14 defaults as PVIO sets them, solver_options.h:26-33) on the device; the host sees one
// launch and one read-back.  All arithmetic is fp64.
#include <cstring>
#include "api_internal.h"
#include "ba_lin.cuh"
#include "ba_solve.cuh"

namespace pvio {

struct PnpArgs {
    const double *pts;      // [n][3]
    const double *z;        // [n][2]
    int n, inertial, max_iter;
    double radius0;
    WinConst wc;            // extrinsics, sqrt_inv_cov, cauchy_a
    double last[16];
    const double *imu_rec;  // [288] device
    double *frame;          // [16] in/out (device)
    double *out;            // [8] iterations, accepted, termination, usable, initial_cost, final_cost, radius, mu
};

constexpr int kPnpThreads = 256;

// residual (whitened) and local Jacobian of one pose-only reprojection block, fp64
__device__ __forceinline__ void pnp_point(const double *R, const double *p, const double *Rcs, const double *pcs,
                                          const double *W, const double *xw, const double *z, bool jac, double *r,
                                          double *J /*[2][6]*/) {
    double d[3] = {xw[0] - p[0], xw[1] - p[1], xw[2] - p[2]}, yc[3], t[3], y[3];
    mat3_tvec(R, d, yc);                                       // q^-1 (x - p)            :174
    for (int k = 0; k < 3; ++k) t[k] = yc[k] - pcs[k];
    mat3_tvec(Rcs, t, y);                                      //                         :175
    const double iz = 1.0 / y[2];
    const double u0 = y[0] * iz - z[0], u1 = y[1] * iz - z[1];
    r[0] = W[0] * u0 + W[1] * u1;
    r[1] = W[2] * u0 + W[3] * u1;
    if (!jac) return;
    const double dp[6] = {iz, 0, -y[0] * iz * iz, 0, iz, -y[1] * iz * iz};
    double A[6], Dc[6];
    for (int k = 0; k < 3; ++k) { A[k] = W[0] * dp[k] + W[1] * dp[3 + k]; A[3 + k] = W[2] * dp[k] + W[3] * dp[3 + k]; }
    for (int i = 0; i < 2; ++i)                                 // A * Rcs^T
        for (int k = 0; k < 3; ++k) Dc[3 * i + k] = A[3 * i] * Rcs[3 * k] + A[3 * i + 1] * Rcs[3 * k + 1] + A[3 * i + 2] * Rcs[3 * k + 2];
    for (int i = 0; i < 2; ++i) {
        const double a0 = Dc[3 * i], a1 = Dc[3 * i + 1], a2 = Dc[3 * i + 2];
        J[6 * i + 0] = a1 * yc[2] - a2 * yc[1];               // Dc * hat(yc)             :188
        J[6 * i + 1] = a2 * yc[0] - a0 * yc[2];
        J[6 * i + 2] = a0 * yc[1] - a1 * yc[0];
        for (int k = 0; k < 3; ++k)                             // -Dc * R^T                :192
            J[6 * i + 3 + k] = -(a0 * R[3 * k] + a1 * R[3 * k + 1] + a2 * R[3 * k + 2]);
    }
}

struct PnpShared {
    double x[16], xc[16];
    double H[225], g[15];
    double Jraw[450], rraw[16], Jw[225], rw[16];
    double scale[15], diag[15], grad[15], gn[15], dx[15];
    double red[32];
    double cost, cand_cost, radius, mu, alpha, x_norm, model_change, step_norm;
    int done, term, usable, it, accepted, reuse, action, nd;
};

// all threads: H, g, cost at state xs (jac) or only the cost
__device__ void pnp_evaluate(const PnpArgs &a, PnpShared &S, const double *xs, bool jac, double *cost_out) {
    const int tid = threadIdx.x;
    __shared__ double R[9], Rcs[9];
    if (tid == 0) { quat_to_mat(xs, R); quat_to_mat(a.wc.cam_q, Rcs); }
    if (jac) for (int i = tid; i < 225 + 15; i += kPnpThreads) S.H[i] = 0.0;     // H and g are contiguous
    if (tid < 32) S.red[tid] = 0.0;
    __syncthreads();
    const double cb = a.wc.cauchy_a * a.wc.cauchy_a;
    double acc[28];
    for (int i = 0; i < 28; ++i) acc[i] = 0.0;
    for (int i = tid; i < a.n; i += kPnpThreads) {
        double r[2], J[12];
        pnp_point(R, xs + 4, Rcs, a.wc.cam_p, a.wc.sic, a.pts + 3 * i, a.z + 2 * i, jac, r, J);
        const double s = r[0] * r[0] + r[1] * r[1], t = 1.0 + s / cb;
        acc[27] += 0.5 * cb * log(t);
        if (jac) {
            const double sc = sqrt(1.0 / t);                   // corrector (rho'' < 0)
            r[0] *= sc; r[1] *= sc;
            for (int k = 0; k < 12; ++k) J[k] *= sc;
            int e = 0;
            for (int p = 0; p < 6; ++p)
                for (int q = p; q < 6; ++q) acc[e++] += J[p] * J[q] + J[6 + p] * J[6 + q];
            for (int p = 0; p < 6; ++p) acc[21 + p] += J[p] * r[0] + J[6 + p] * r[1];
        }
    }
    for (int k = jac ? 0 : 27; k < 28; ++k) {
        double v = acc[k];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((tid & 31) == 0 && v != 0.0) atomicAdd(&S.red[k], v);
    }
    // IMU prior factor: frame_i = last frame (constant), Jacobian columns of frame_j only
    if (a.inertial) {
        if (tid == 32) imu_factor_raw(a.last, xs, a.imu_rec, a.wc, 1, S.rraw, jac ? S.Jraw : nullptr);
        __syncthreads();
        for (int e = tid; e < 15 * 16; e += kPnpThreads) {
            const int row = e / 16, col = e - row * 16;
            const double *Wm = a.imu_rec + 11 + row * 15;
            double s = 0.0;
            if (col < 15) { if (jac) { for (int k = 0; k < 15; ++k) s += Wm[k] * S.Jraw[k * 30 + 15 + col]; S.Jw[row * 15 + col] = s; } }
            else { for (int k = 0; k < 15; ++k) s += Wm[k] * S.rraw[k]; S.rw[row] = s; }
        }
    }
    __syncthreads();
    if (jac) {
        // scatter the 6x6 vision block, then add the IMU block
        for (int e = tid; e < 225; e += kPnpThreads) {
            const int i = e / 15, j = e - i * 15;
            double v = 0.0;
            if (i < 6 && j < 6) { const int p = min(i, j), q = max(i, j); v = S.red[p * 6 - p * (p - 1) / 2 + (q - p)]; }
            if (a.inertial) for (int k = 0; k < 15; ++k) v += S.Jw[k * 15 + i] * S.Jw[k * 15 + j];
            S.H[e] = v;
        }
        if (tid < 15) {
            double v = tid < 6 ? S.red[21 + tid] : 0.0;
            if (a.inertial) for (int k = 0; k < 15; ++k) v += S.Jw[k * 15 + tid] * S.rw[k];
            S.g[tid] = v;
        }
    }
    if (tid == 0) {
        double c = S.red[27];
        if (a.inertial) for (int k = 0; k < 15; ++k) c += 0.5 * S.rw[k] * S.rw[k];
        *cost_out = c;
    }
    __syncthreads();
}

__device__ double pnp_ambient_norm2(const double *x, const double *y, int inertial) {   // |x - y|^2 or |x|^2 (y = null)
    double s = 0.0;
    const int n = inertial ? 16 : 7;
    for (int i = 0; i < n; ++i) { const double d = y ? x[i] - y[i] : x[i]; s += d * d; }
    return s;
}

// thread 0: regularised GN solve (Hs + mu diag^2) xs = gs by dense Cholesky; returns false if not SPD
__device__ bool pnp_chol_solve(const double *Hs, const double *lm2, const double *rhs, int n, double *xs) {
    double L[225];
    for (int i = 0; i < n; ++i)
        for (int j = 0; j <= i; ++j) {
            double s = Hs[i * 15 + j] + (i == j ? lm2[i] : 0.0);
            for (int k = 0; k < j; ++k) s -= L[i * 15 + k] * L[j * 15 + k];
            if (i == j) { if (!(s > 0.0) || !isfinite(s)) return false; L[i * 15 + i] = sqrt(s); }
            else L[i * 15 + j] = s / L[j * 15 + j];
        }
    for (int i = 0; i < n; ++i) { double s = rhs[i]; for (int k = 0; k < i; ++k) s -= L[i * 15 + k] * xs[k]; xs[i] = s / L[i * 15 + i]; }
    for (int i = n - 1; i >= 0; --i) { double s = xs[i]; for (int k = i + 1; k < n; ++k) s -= L[k * 15 + i] * xs[k]; xs[i] = s / L[i * 15 + i]; }
    for (int i = 0; i < n; ++i) if (!isfinite(xs[i])) return false;
    return true;
}

__global__ void __launch_bounds__(kPnpThreads) pnp_kernel(PnpArgs a) {
    __shared__ PnpShared S;
    const int tid = threadIdx.x;
    if (tid < 16) S.x[tid] = a.frame[tid];
    if (tid == 0) {
        S.done = 0; S.term = PVIO_B200_TERM_NO_CONVERGENCE; S.usable = 1; S.it = 0; S.accepted = 0; S.reuse = 0;
        S.radius = a.radius0; S.mu = 1e-8; S.nd = a.inertial ? 15 : 6;
    }
    __syncthreads();
    pnp_evaluate(a, S, S.x, true, &S.cost);
    if (tid == 0) {
        a.out[4] = S.cost;
        double gmax = 0.0;
        for (int i = 0; i < S.nd; ++i) {
            S.scale[i] = 1.0 / (1.0 + sqrt(fmax(S.H[i * 15 + i], 0.0)));     // Jacobi scaling, fixed at iteration 0
            gmax = fmax(gmax, fabs(S.g[i]));
        }
        if (gmax <= 1e-10) { S.done = 1; S.term = PVIO_B200_TERM_CONVERGENCE; }
        S.x_norm = sqrt(pnp_ambient_norm2(S.x, nullptr, a.inertial));
    }
    __syncthreads();
    for (;;) {
        __syncthreads();                 // everybody has consumed the flags of the previous round
        if (S.done) break;
        __syncthreads();
        // ---------------- thread 0: DoglegStrategy::ComputeStep
        if (tid == 0) {
            S.action = 0;
            if (S.it >= a.max_iter) { S.done = 1; }
            else {
                ++S.it;
                const int n = S.nd;
                double Hs[225], gs[15], step[15];
                for (int i = 0; i < n; ++i) { gs[i] = S.g[i] * S.scale[i]; for (int j = 0; j < n; ++j) Hs[i * 15 + j] = S.H[i * 15 + j] * S.scale[i] * S.scale[j]; }
                if (!S.reuse) {
                    double sg[15], g2 = 0.0, q = 0.0;
                    for (int i = 0; i < n; ++i) {
                        S.diag[i] = sqrt(fmin(fmax(Hs[i * 15 + i], 1.0e-6), 1.0e32));
                        S.grad[i] = gs[i] / S.diag[i];
                        sg[i] = S.grad[i] / S.diag[i];
                        g2 += S.grad[i] * S.grad[i];
                    }
                    for (int i = 0; i < n; ++i) { double t = 0.0; for (int j = 0; j < n; ++j) t += Hs[i * 15 + j] * sg[j]; q += sg[i] * t; }
                    S.alpha = g2 / q;
                    double xs[15], lm2[15];
                    for (;;) {
                        for (int i = 0; i < n; ++i) lm2[i] = S.diag[i] * S.diag[i] * S.mu;
                        if (pnp_chol_solve(Hs, lm2, gs, n, xs)) break;
                        S.mu *= 10.0;
                        if (S.mu > 1.0) { S.done = 1; S.term = PVIO_B200_TERM_FAILURE; S.usable = 0; break; }
                    }
                    for (int i = 0; i < n; ++i) S.gn[i] = -S.diag[i] * xs[i];
                }
                if (!S.done) {
                    double gn2 = 0.0, g2 = 0.0, gdot = 0.0;
                    for (int i = 0; i < n; ++i) { gn2 += S.gn[i] * S.gn[i]; g2 += S.grad[i] * S.grad[i]; gdot += S.grad[i] * S.gn[i]; }
                    const double gn_norm = sqrt(gn2), g_norm = sqrt(g2), rad = S.radius;
                    if (gn_norm <= rad) { for (int i = 0; i < n; ++i) step[i] = S.gn[i]; S.step_norm = gn_norm; }
                    else if (g_norm * S.alpha >= rad) { for (int i = 0; i < n; ++i) step[i] = -(rad / g_norm) * S.grad[i]; S.step_norm = rad; }
                    else {
                        const double b_dot_a = -S.alpha * gdot, a2 = (S.alpha * g_norm) * (S.alpha * g_norm);
                        const double bma2 = a2 - 2.0 * b_dot_a + gn2, c = b_dot_a - a2;
                        const double d = sqrt(c * c + bma2 * (rad * rad - a2));
                        const double beta = c <= 0 ? (d - c) / bma2 : (rad * rad - a2) / (d + c);
                        for (int i = 0; i < n; ++i) step[i] = (-S.alpha * (1.0 - beta)) * S.grad[i] + beta * S.gn[i];
                        S.step_norm = rad;
                    }
                    double sg_ = 0.0, sHs = 0.0;
                    for (int i = 0; i < n; ++i) step[i] /= S.diag[i];
                    for (int i = 0; i < n; ++i) { double t = 0.0; for (int j = 0; j < n; ++j) t += Hs[i * 15 + j] * step[j]; sHs += step[i] * t; sg_ += step[i] * gs[i]; }
                    S.model_change = -(sg_ + 0.5 * sHs);
                    if (S.model_change < 0.0) { S.radius *= 0.5; S.reuse = 1; S.action = 0; }       // invalid step
                    else {
                        for (int i = 0; i < 15; ++i) S.dx[i] = i < n ? step[i] * S.scale[i] : 0.0;
                        quat_plus(S.x, S.dx, S.xc);
                        for (int i = 0; i < 12; ++i) S.xc[4 + i] = S.x[4 + i] + S.dx[3 + i];
                        S.action = 1;
                    }
                }
            }
        }
        __syncthreads();
        if (S.done) break;
        if (S.action == 0) continue;
        // ---------------- all threads: candidate cost
        pnp_evaluate(a, S, S.xc, false, &S.cand_cost);
        if (tid == 0) {
            S.action = 0;
            const double step_amb = sqrt(pnp_ambient_norm2(S.xc, S.x, a.inertial));
            if (step_amb <= 1e-8 * (S.x_norm + 1e-8)) { S.done = 1; S.term = PVIO_B200_TERM_CONVERGENCE; }
            else if (fabs(S.cost - S.cand_cost) <= 1e-6 * S.cost) { S.done = 1; S.term = PVIO_B200_TERM_CONVERGENCE; }
            else {
                const double rel = (S.cost - S.cand_cost) / S.model_change;
                if (rel > 1e-3) {
                    for (int i = 0; i < 16; ++i) S.x[i] = S.xc[i];
                    S.x_norm = sqrt(pnp_ambient_norm2(S.x, nullptr, a.inertial));
                    ++S.accepted;
                    if (rel < 0.25) S.radius *= 0.5;
                    if (rel > 0.75) S.radius = fmax(S.radius, 3.0 * S.step_norm);
                    S.mu = fmax(1e-8, 2.0 * S.mu / 10.0);
                    S.reuse = 0;
                    S.action = 2;                                   // re-linearise
                } else { S.radius *= 0.5; S.reuse = 1; }
                if (S.radius <= 1e-32) { S.done = 1; S.term = PVIO_B200_TERM_CONVERGENCE; }
            }
        }
        __syncthreads();
        if (S.action == 2) {
            pnp_evaluate(a, S, S.x, true, &S.cost);
            if (tid == 0) {
                double gmax = 0.0;
                for (int i = 0; i < S.nd; ++i) gmax = fmax(gmax, fabs(S.g[i]));
                if (gmax <= 1e-10) { S.done = 1; S.term = PVIO_B200_TERM_CONVERGENCE; }
            }
            __syncthreads();
        }
    }
    if (tid < 16) a.frame[tid] = S.x[tid];
    if (tid == 0) {
        a.out[0] = S.it; a.out[1] = S.accepted; a.out[2] = S.term; a.out[3] = S.usable;
        a.out[5] = S.cost; a.out[6] = S.radius; a.out[7] = S.mu;
    }
}

int pnp_solve_impl(Handle *h, const pvio_b200_pnp_problem *pb, double *frame, const pvio_b200_options *opt,
                   pvio_b200_summary *summary) {
    const int n = pb->n_points;
    if (n < 0 || !frame || !pb->last_frame || (pb->use_inertial && !pb->imu_data))
        return fail(h, PVIO_B200_EINVAL, "pnp: bad arguments");
    const size_t words = (size_t)5 * n + 16 + 8 + kImuStride;
    if (words > h->pnp_words) {                       // this runs on every frame: no allocation in the steady state
        if (h->pnp_dev) cudaFree(h->pnp_dev);
        if (h->pnp_host) cudaFreeHost(h->pnp_host);
        h->pnp_dev = nullptr; h->pnp_host = nullptr; h->pnp_words = 0;
        const size_t cap = std::max<size_t>(words, (size_t)5 * 512 + 16 + 8 + kImuStride);
        CK(h, cudaMalloc(&h->pnp_dev, sizeof(double) * cap));
        CK(h, cudaMallocHost(&h->pnp_host, sizeof(double) * cap));
        h->pnp_words = cap;
    }
    double *d = h->pnp_dev, *stage = h->pnp_host;
    memset(stage, 0, sizeof(double) * words);
    if (n > 0) { memcpy(stage, pb->points, sizeof(double) * 3 * n); memcpy(stage + 3 * n, pb->z, sizeof(double) * 2 * n); }
    memcpy(stage + 5 * n, frame, sizeof(double) * 16);
    if (pb->use_inertial) memcpy(stage + 5 * n + 24, pb->imu_data, sizeof(double) * kImuStride);
    CK(h, cudaMemcpyAsync(d, stage, sizeof(double) * words, cudaMemcpyHostToDevice, h->stream));
    PnpArgs a;
    memset(&a, 0, sizeof(a));
    a.pts = d; a.z = d + 3 * n; a.frame = d + 5 * n; a.out = d + 5 * n + 16; a.imu_rec = d + 5 * n + 24;
    a.n = n; a.inertial = pb->use_inertial ? 1 : 0;
    const SolveOpts o = solve_opts(opt);
    a.max_iter = o.max_iter;
    a.radius0 = o.radius0;
    memcpy(a.wc.cam_q, pb->cam_q_cs, 32); memcpy(a.wc.cam_p, pb->cam_p_cs, 24);
    memcpy(a.wc.imu_q, pb->imu_q_cs, 32); memcpy(a.wc.imu_p, pb->imu_p_cs, 24);
    memcpy(a.wc.sic, pb->sqrt_inv_cov, 32);
    a.wc.cauchy_a = pb->cauchy_a > 0 ? pb->cauchy_a : 1.0;
    memcpy(a.last, pb->last_frame, sizeof(double) * 16);
    CK(h, cudaEventRecord(h->ev0, h->stream));
    pnp_kernel<<<1, kPnpThreads, 0, h->stream>>>(a);
    CK(h, cudaEventRecord(h->ev1, h->stream));
    ++h->launches;
    double *back = stage + 5 * n;                     // the frame + summary words come back into the pinned staging
    CK(h, cudaMemcpyAsync(back, d + 5 * n, sizeof(double) * 24, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    CK(h, cudaGetLastError());
    memcpy(frame, back, sizeof(double) * 16);
    if (summary) {
        memset(summary, 0, sizeof(*summary));
        summary->iterations = (int)back[16]; summary->accepted_steps = (int)back[17];
        summary->termination = (int)back[18]; summary->usable = (int)back[19];
        summary->initial_cost = back[20]; summary->final_cost = back[21];
        summary->final_radius = back[22]; summary->final_mu = back[23];
        float ms = 0.f;
        cudaEventElapsedTime(&ms, h->ev0, h->ev1);
        summary->solve_seconds = ms * 1e-3;
    }
    return 0;
}

}  // namespace pvio
