// Frame marginalisation: BundleAdjustor::marginalize_frame (estimation/bundle_adjustor.cpp:348-599).
//
//   prior J^T J                                   :369-413   marg_assemble_kernel
//   IMU factors adjacent to the victim            :416-450   marg_assemble_kernel
//   reprojection factors of victim-seen tracks    :453-533   lin_obs_kernel<false, double> (no loss, quirk Q3; ba_linearize.cuh)
//   landmark Schur (1/mat, isfinite skip)         :536-545   schur_kernel<double> (ba_schur.cuh)
//   frame Schur with the explicit 15x15 inverse   :547-581   marg_reduce_kernel
//   eigen factorisation, clamp lambda <= 1e-8     :583-590   marg_eig_kernel (Householder tridiagonalisation + implicit QL)
// All dense algebra is fp64.  Runs once per keyframe (not per iteration): latency, not bandwidth.
#include <cstring>
#include <vector>
#include "api_internal.h"
#include "ba_lin.cuh"
#include "ba_solve.cuh"

namespace pvio {

struct MargArgs {
    const WinHdr *hdr;
    const WinConst *cst;
    const double *frames;
    const double *Hred, *gred;         // vision part (xi coordinates) from the linearise + Schur stage
    const int32_t *imu_idx;
    const double *imu_data;
    const int32_t *prior_frames;
    const double *prior_S, *prior_L, *prior_e, *prior_x0;
    int Ncap;
    int index;                         // victim frame
    double *H;                         // [(15N)^2] row-major, full symmetric
    double *b;                         // [15N]
    double *scratch;                   // >= 4*(15*30+16) + 4*15*Ncap doubles
};

__global__ void __launch_bounds__(256) marg_assemble_kernel(MargArgs a) {
    const WinHdr &Hh = a.hdr[0];
    const WinConst &wc = a.cst[0];
    const int N = Hh.N, n = 15 * N;
    const int tid = threadIdx.x, nt = blockDim.x;
    const double *frames = a.frames;
    __shared__ double T[kMaxFrames * 36];
    for (int i = tid; i < n * n; i += nt) a.H[i] = 0.0;
    for (int i = tid; i < n; i += nt) a.b[i] = 0.0;
    if (tid < N) {
        const double *fs = frames + tid * kFrameStride;
        double R[9], Hp[9], B[9];
        quat_to_mat(fs, R);
        const double p[3] = {fs[4] - wc.origin[0], fs[5] - wc.origin[1], fs[6] - wc.origin[2]};
        hat(p, Hp);
        mat3_mul(Hp, R, B);
        double *Tf = T + tid * 36;
        for (int r_ = 0; r_ < 3; ++r_)
            for (int c_ = 0; c_ < 3; ++c_) {
                Tf[r_ * 6 + c_] = R[3 * r_ + c_];
                Tf[r_ * 6 + 3 + c_] = 0.0;
                Tf[(3 + r_) * 6 + c_] = -B[3 * r_ + c_];
                Tf[(3 + r_) * 6 + 3 + c_] = (r_ == c_) ? -1.0 : 0.0;
            }
    }
    __syncthreads();
    // ---- vision: H_delta[f,g] = T_f^T X T_g  (reprojection + landmark Schur, :453-545)
    const int npairs = N * (N + 1) / 2;
    for (int e = tid; e < npairs * 36; e += nt) {
        const int p = e / 36, ij = e - p * 36, i = ij / 6, j = ij - i * 6;
        int f = 0;
        while ((f + 1) * (f + 2) / 2 <= p) ++f;
        const int gf = p - f * (f + 1) / 2;
        const double *X = a.Hred + p * 36;
        const double *Tf = T + f * 36, *Tg = T + gf * 36;
        double s = 0.0;
        for (int aa = 0; aa < 6; ++aa) {
            double t = 0.0;
            for (int bb = 0; bb < 6; ++bb) t += X[aa * 6 + bb] * Tg[bb * 6 + j];
            s += Tf[aa * 6 + i] * t;
        }
        const int gi = f * 15 + i, gj = gf * 15 + j;
        a.H[(size_t)gi * n + gj] = s;
        if (f != gf) a.H[(size_t)gj * n + gi] = s;
    }
    for (int e = tid; e < N * 6; e += nt) {
        const int f = e / 6, i = e - f * 6;
        double s = 0.0;
        for (int aa = 0; aa < 6; ++aa) s += T[f * 36 + aa * 6 + i] * a.gred[f * 6 + aa];
        a.b[f * 15 + i] = s;
    }
    __syncthreads();
    // ---- prior :369-413  (H += E^T Lambda E, b += E^T S^T (S r0 + e))
    if (Hh.n_prior > 0) {
        const int np = Hh.n_prior, d = 15 * np;
        double *r0 = a.scratch, *rr = r0 + d, *vv = rr + d, *Ji = vv + d;
        if (tid < np) prior_frame_raw(frames + a.prior_frames[tid] * kFrameStride, a.prior_x0 + tid * kFrameStride,
                                      r0 + 15 * tid, Ji + 9 * tid);
        __syncthreads();
        for (int i = tid; i < d; i += nt) {
            double s = a.prior_e[i];
            for (int k = 0; k < d; ++k) s += a.prior_S[(size_t)i * d + k] * r0[k];
            rr[i] = s;
        }
        __syncthreads();
        for (int i = tid; i < d; i += nt) {
            double s = 0.0;
            for (int k = 0; k < d; ++k) s += a.prior_S[(size_t)k * d + i] * rr[k];
            vv[i] = s;
        }
        __syncthreads();
        for (int i = tid; i < d; i += nt) {
            const int fi = i / 15, ci = i - fi * 15;
            double s;
            if (ci < 3) { s = 0.0; for (int k = 0; k < 3; ++k) s += Ji[9 * fi + 3 * k + ci] * vv[15 * fi + k]; }
            else s = vv[i];
            a.b[a.prior_frames[fi] * 15 + ci] += s;
        }
        const double *L = a.prior_L;
        for (int e = tid; e < d * d; e += nt) {
            const int i = e / d, j = e - i * d;
            const int fi = i / 15, ci = i - fi * 15, fj = j / 15, cj = j - fj * 15;
            double s = 0.0;
            if (ci < 3 && cj < 3) {
                for (int k = 0; k < 3; ++k)
                    for (int m = 0; m < 3; ++m)
                        s += Ji[9 * fi + 3 * k + ci] * L[(size_t)(15 * fi + k) * d + 15 * fj + m] * Ji[9 * fj + 3 * m + cj];
            } else if (ci < 3) {
                for (int k = 0; k < 3; ++k) s += Ji[9 * fi + 3 * k + ci] * L[(size_t)(15 * fi + k) * d + j];
            } else if (cj < 3) {
                for (int m = 0; m < 3; ++m) s += L[(size_t)i * d + 15 * fj + m] * Ji[9 * fj + 3 * m + cj];
            } else {
                s = L[(size_t)i * d + j];
            }
            a.H[(size_t)(a.prior_frames[fi] * 15 + ci) * n + a.prior_frames[fj] * 15 + cj] += s;
        }
        __syncthreads();
    }
    // ---- IMU factors with j == index or j == index + 1  :416-450.  The functor reads the bias
    // linearisation point from the very memory passed as the parameter, so dbg = dba = 0.
    for (int m = 0; m < Hh.n_imu; ++m) {
        const int fi = a.imu_idx[2 * m], fj = a.imu_idx[2 * m + 1];
        if (fj != a.index && fj != a.index + 1) continue;
        double *Jraw = a.scratch, *rraw = Jraw + 450, *Jw = rraw + 16, *rw = Jw + 450;
        const double *rec = a.imu_data + (size_t)m * kImuStride;
        if (tid == 0) imu_factor_raw(frames + fi * kFrameStride, frames + fj * kFrameStride, rec, wc, 1, rraw, Jraw);
        __syncthreads();
        for (int e = tid; e < 15 * 31; e += nt) {
            const int row = e / 31, col = e - row * 31;
            const double *Wm = rec + 11 + row * 15;
            double s = 0.0;
            if (col < 30) { for (int k = 0; k < 15; ++k) s += Wm[k] * Jraw[k * 30 + col]; Jw[row * 30 + col] = s; }
            else { for (int k = 0; k < 15; ++k) s += Wm[k] * rraw[k]; rw[row] = s; }
        }
        __syncthreads();
        for (int e = tid; e < 30 * 31; e += nt) {
            const int ra = e / 31, cb_ = e - ra * 31;
            const int ga = (ra < 15 ? fi * 15 + ra : fj * 15 + ra - 15);
            double s = 0.0;
            if (cb_ < 30) {
                const int gb = (cb_ < 15 ? fi * 15 + cb_ : fj * 15 + cb_ - 15);
                for (int k = 0; k < 15; ++k) s += Jw[k * 30 + ra] * Jw[k * 30 + cb_];
                a.H[(size_t)ga * n + gb] += s;
            } else {
                for (int k = 0; k < 15; ++k) s += Jw[k * 30 + ra] * rw[k];
                a.b[ga] += s;
            }
        }
        __syncthreads();
    }
}

// Frame Schur complement :547-581.  inv = H[vv]^-1 by Gauss-Jordan with partial pivoting
// (Eigen's dynamic .inverse() is PartialPivLU based), then Hk = H[kk] - H[kv] inv H[vk].
__global__ void __launch_bounds__(256) marg_reduce_kernel(const double *H, const double *b, int N, int index,
                                                         double *Hk, double *bk) {
    const int n = 15 * N, dk = n - 15, v0 = 15 * index;
    const int tid = threadIdx.x, nt = blockDim.x;
    __shared__ double M[15][31];
    __shared__ int piv_sm;
    for (int e = tid; e < 15 * 30; e += nt) {
        const int i = e / 30, j = e - i * 30;
        M[i][j] = (j < 15) ? H[(size_t)(v0 + i) * n + v0 + j] : ((j - 15 == i) ? 1.0 : 0.0);
    }
    __syncthreads();
    for (int c = 0; c < 15; ++c) {
        if (tid == 0) {
            int p = c;
            double best = fabs(M[c][c]);
            for (int i = c + 1; i < 15; ++i) if (fabs(M[i][c]) > best) { best = fabs(M[i][c]); p = i; }
            piv_sm = p;
        }
        __syncthreads();
        const int p = piv_sm;
        if (p != c && tid < 30) { const double t = M[c][tid]; M[c][tid] = M[p][tid]; M[p][tid] = t; }
        __syncthreads();
        const double ip = 1.0 / M[c][c];
        __syncthreads();
        if (tid < 30) M[c][tid] *= ip;
        __syncthreads();
        // eliminate column c from the other rows (compute, barrier, write: no read/write race)
        double newv[2] = {0.0, 0.0};
        int cnt = 0;
        for (int e = tid; e < 15 * 30; e += nt, ++cnt) {
            const int i = e / 30, jx = e - i * 30;
            newv[cnt] = (i != c) ? M[i][jx] - M[i][c] * M[c][jx] : M[i][jx];
        }
        __syncthreads();
        cnt = 0;
        for (int e = tid; e < 15 * 30; e += nt, ++cnt) M[e / 30][e % 30] = newv[cnt];
        __syncthreads();
    }
    // keep index list: all coordinates except the victim's 15
    // W = H[kv] * inv  (dk x 15) streamed through registers per thread
    for (int e = tid; e < dk * (dk + 1); e += nt) {
        const int i = e / (dk + 1), j = e - i * (dk + 1);
        const int gi = i < v0 ? i : i + 15;
        // row vector H[gi, v] * inv
        double acc = 0.0;
        if (j < dk) {
            const int gj = j < v0 ? j : j + 15;
            for (int k = 0; k < 15; ++k) {
                double wk = 0.0;
                for (int m = 0; m < 15; ++m) wk += H[(size_t)gi * n + v0 + m] * M[m][15 + k];
                acc += wk * H[(size_t)(v0 + k) * n + gj];
            }
            Hk[(size_t)i * dk + j] = H[(size_t)gi * n + gj] - acc;
        } else {
            for (int k = 0; k < 15; ++k) {
                double wk = 0.0;
                for (int m = 0; m < 15; ++m) wk += H[(size_t)gi * n + v0 + m] * M[m][15 + k];
                acc += wk * b[v0 + k];
            }
            bk[i] = b[gi] - acc;
        }
    }
}

// Symmetric eigen-decomposition for the factorisation :583-590 (Eigen::SelfAdjointEigenSolver in the reference): Householder
// tridiagonalisation + implicit QL with eigenvector accumulation (the EISPACK tred2 / tql2 pair), one CTA, the matrix
// in SHARED memory (odd leading dimension: conflict-free rows and columns).  Every O(n^2) inner loop is spread over the
// CTA; the scalar QL recurrence runs on one thread, which hands a batch of rotations to the CTA (thread k owns row k of
// the eigenvector matrix and applies the batch in order: no barrier inside a sweep).
// Then S = sqrt(max(lambda, 0 if <= 1e-8)) V^T and e = sqrt(1 / lambda) V^T b.
// (The first version was a parallel cyclic Jacobi on global memory: 32 ms for d = 120, profiles/r02_latency.md.)
__device__ __forceinline__ double block_sum(double v, double *red, int tid, int nt) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((tid & 31) == 0) red[tid >> 5] = v;
    __syncthreads();
    double s = 0.0;
    for (int k = 0; k < (nt >> 5); ++k) s += red[k];
    return s;
}

#ifdef PVIO_MARG_STAMPS            // tuning builds of tools/ only: phase times of the eigen-solver
__device__ long long g_marg_stamps[8];
#define MARG_STAMP(k) do { __syncthreads(); if (threadIdx.x == 0) g_marg_stamps[k] = clock64(); } while (0)
#else
#define MARG_STAMP(k) do { } while (0)
#endif

__global__ void __launch_bounds__(256) marg_eig_kernel(const double *Ain, const double *bvec, int n, int ring, double *S, double *evec) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, nt = blockDim.x;
    const int ld = n | 1;
    double *a = reinterpret_cast<double *>(smem_raw);       // [n][ld]: matrix -> eigenvectors (columns)
    double *d = a + (size_t)n * ld;                         // [n]
    double *e = d + n;                                      // [n]
    double *rot = e + n;                                    // [ring][2][n] rotation cosines / sines of the QL sweeps in flight
    __shared__ double red[8];
    __shared__ double sc_sm[4];
    __shared__ int ctl[2 + 2 * 4];                          // produced, consumed, index range of each ring slot
    for (int idx = tid; idx < n * n; idx += nt) a[(idx / n) * ld + idx % n] = Ain[idx];
    __syncthreads();
    MARG_STAMP(0);
    // ---- tred2
    for (int i = n - 1; i > 0; --i) {
        const int l = i - 1;
        double *ai = a + (size_t)i * ld;
        if (l > 0) {
            double sa = 0.0;
            for (int k = tid; k <= l; k += nt) sa += fabs(ai[k]);
            const double scale = block_sum(sa, red, tid, nt);
            if (scale == 0.0) {
                if (tid == 0) { e[i] = ai[l]; d[i] = 0.0; }
                __syncthreads();
                continue;
            }
            double sh = 0.0;
            for (int k = tid; k <= l; k += nt) { const double v = ai[k] / scale; ai[k] = v; sh += v * v; }
            double h = block_sum(sh, red, tid, nt);
            if (tid == 0) {
                const double f = ai[l], g = f >= 0 ? -sqrt(h) : sqrt(h);
                e[i] = scale * g;
                sc_sm[0] = h - f * g;
                ai[l] = f - g;
            }
            __syncthreads();
            h = sc_sm[0];
            double sf = 0.0;
            for (int j = tid; j <= l; j += nt) {             // e[j] = (A u)_j / h, u = row i
                a[(size_t)j * ld + i] = ai[j] / h;
                double g = 0.0;
                const double *aj = a + (size_t)j * ld;
                for (int k = 0; k <= j; ++k) g += aj[k] * ai[k];
                for (int k = j + 1; k <= l; ++k) g += a[(size_t)k * ld + j] * ai[k];
                e[j] = g / h;
                sf += e[j] * ai[j];
            }
            const double f = block_sum(sf, red, tid, nt);
            const double hh = f / (h + h);
            for (int j = tid; j <= l; j += nt) e[j] -= hh * ai[j];
            __syncthreads();
            const int tri = (l + 1) * (l + 2) / 2;          // rank-2 update of the lower triangle
            for (int idx = tid; idx < tri; idx += nt) {
                int j = (int)((sqrtf(8.0f * idx + 1.0f) - 1.0f) * 0.5f);
                while ((j + 1) * (j + 2) / 2 <= idx) ++j;
                while (j * (j + 1) / 2 > idx) --j;
                const int k = idx - j * (j + 1) / 2;
                a[(size_t)j * ld + k] -= ai[j] * e[k] + e[j] * ai[k];
            }
            if (tid == 0) d[i] = h;
        } else if (tid == 0) { e[i] = ai[l]; d[i] = 0.0; }
        __syncthreads();
    }
    if (tid == 0) { d[0] = 0.0; e[0] = 0.0; }
    __syncthreads();
    MARG_STAMP(1);
    for (int i = 0; i < n; ++i) {                            // accumulate the transformations
        const int l = i - 1;
        double *ai = a + (size_t)i * ld;
        if (d[i] != 0.0) {
            for (int j = tid; j <= l; j += nt) {
                double g = 0.0;
                for (int k = 0; k <= l; ++k) g += ai[k] * a[(size_t)k * ld + j];
                for (int k = 0; k <= l; ++k) a[(size_t)k * ld + j] -= g * a[(size_t)k * ld + i];
            }
        }
        __syncthreads();
        if (tid == 0) { d[i] = ai[i]; ai[i] = 1.0; }
        for (int j = tid; j <= l; j += nt) { a[(size_t)j * ld + i] = 0.0; ai[j] = 0.0; }
        __syncthreads();
    }
    MARG_STAMP(2);
    // ---- tql2, producer / consumer: the scalar recurrence of the implicit QL sweeps touches only d and e -- it does not
    // depend on the eigenvector matrix -- so ONE thread (lane 0 of warp 0) runs ahead through all sweeps, publishing each
    // sweep's rotations (cosines, sines, index range) in a ring of `ring` slots, while warps 1..7 apply the batches in
    // order, row k of the matrix per thread.  The sweep time was scalar chain + application + three CTA barriers
    // (13 K cycles per sweep, ~220 sweeps at n = 120); it is now the longer of the two.
    if (tid == 0) { for (int i = 1; i < n; ++i) e[i - 1] = e[i]; e[n - 1] = 0.0; }
    volatile int *vctl = ctl;                                // [0] batches produced, [1] batches consumed
    if (tid == 0) { vctl[0] = 0; vctl[1] = 0; }
    int *rng = ctl + 2;                                      // [ring][2] index range of each slot (i_hi, i_lo); i_hi = -2: the end
    __syncthreads();
    if (tid < 32) {
        if (tid == 0) {
            int prod = 0;
            for (int l = 0; l < n; ++l) {
                for (int iter = 0; iter < 64; ++iter) {
                    int m = l;
                    for (; m < n - 1; ++m) { const double dd = fabs(d[m]) + fabs(d[m + 1]); if (fabs(e[m]) <= 2.3e-16 * dd) break; }
                    if (m == l) break;
                    while (prod - vctl[1] >= ring) __nanosleep(40);       // every slot still in use
                    double *rc = rot + (size_t)(prod % ring) * 2 * n, *rs = rc + n;
                    // (sqrt(f^2 + g^2) instead of hypot, one reciprocal instead of two divisions: this scalar chain is the
                    // critical path of the kernel -- ~60 dependent rotations per sweep, ~200 sweeps; the magnitudes here
                    // (<= 1e15 from the gauge prior) are far from the range where hypot's rescaling matters)
                    double g = (d[l + 1] - d[l]) / (2.0 * e[l]), r = sqrt(g * g + 1.0);
                    g = d[m] - d[l] + e[l] / (g + (g >= 0 ? fabs(r) : -fabs(r)));
                    double s = 1.0, c = 1.0, p = 0.0;
                    int i = m - 1;
                    bool broke = false;
                    // e[i] and d[i] of the NEXT rotation are loaded ahead (they are untouched originals: off the dependent
                    // chain s, c, g, p), and d[i + 1] is the d[i] of the rotation before
                    double e_i = e[i], d_i = d[i], d_i1 = d[m];
                    for (; i >= l; --i) {
                        const double e_nx = i > l ? e[i - 1] : 0.0, d_nx = i > l ? d[i - 1] : 0.0;
                        const double f = s * e_i, b = c * e_i;
                        const double q2 = f * f + g * g;
                        if (q2 == 0.0) { e[i + 1] = 0.0; d[i + 1] -= p; e[m] = 0.0; broke = true; break; }
                        const double ir = rsqrt(q2);            // one reciprocal square root gives both r and 1 / r
                        e[i + 1] = r = q2 * ir;
                        s = f * ir; c = g * ir; g = d_i1 - p; r = (d_i - g) * s + 2.0 * c * b; p = s * r; d[i + 1] = g + p; g = c * r - b;
                        rc[i] = c; rs[i] = s;
                        d_i1 = d_i; e_i = e_nx; d_i = d_nx;
                    }
                    if (!broke) { d[l] -= p; e[l] = g; e[m] = 0.0; }
                    rng[2 * (prod % ring)] = m - 1;                      // rotations i = m - 1 .. i_lo, in this order
                    rng[2 * (prod % ring) + 1] = broke ? i + 1 : l;
                    __threadfence_block();
                    vctl[0] = ++prod;
                }
            }
            while (prod - vctl[1] >= ring) __nanosleep(40);
            rng[2 * (prod % ring)] = -2;
            __threadfence_block();
            vctl[0] = prod + 1;
        }
    } else {
        const int ct = tid - 32, nct = nt - 32;
        for (int k = 0;; ++k) {
            while (vctl[0] <= k) __nanosleep(20);
            __threadfence_block();
            const int i_hi = rng[2 * (k % ring)], i_lo = rng[2 * (k % ring) + 1];
            if (i_hi == -2) break;
            const double *rc = rot + (size_t)(k % ring) * 2 * n, *rs = rc + n;
            for (int row = ct; row < n; row += nct) {        // row `row` of the eigenvector matrix takes the whole batch
                double *zk = a + (size_t)row * ld;
                double zi1 = zk[i_hi + 1];
                for (int i = i_hi; i >= i_lo; --i) {
                    const double zi = zk[i], c = rc[i], s = rs[i];
                    zk[i + 1] = s * zi + c * zi1;
                    zi1 = c * zi - s * zi1;
                }
                zk[i_lo] = zi1;
            }
            asm volatile("bar.sync 1, %0;" ::"r"(nct) : "memory");       // the consumers are done with the slot
            if (ct == 0) { vctl[1] = k + 1; }
        }
    }
    __syncthreads();
    MARG_STAMP(3);
    // S = sqrt(lambda_clamped) V^T ; e = sqrt(1 / lambda) V^T b
    for (int i = tid; i < n; i += nt) {
        const double lam = d[i];
        const bool pos = lam > 1.0e-8;
        const double sl = pos ? sqrt(lam) : 0.0, il = pos ? sqrt(1.0 / lam) : 0.0;
        double dot = 0.0;
        for (int k = 0; k < n; ++k) {
            const double v = a[(size_t)k * ld + i];
            S[(size_t)i * n + k] = sl * v;
            dot += v * bvec[k];
        }
        evec[i] = il * dot;
    }
    MARG_STAMP(4);
}

#ifdef PVIO_MARG_STAMPS
extern "C" int pvio_b200_debug_marg_stamps(long long *out) {
    return cudaMemcpyFromSymbol(out, g_marg_stamps, sizeof(long long) * 8) == cudaSuccess ? 0 : -1;
}
#endif

// Persistent device scratch of the marginaliser (it runs at every keyframe: nothing is allocated in the steady state).
struct MargScratch {
    double *buf = nullptr;
    size_t words = 0;
};

void marg_free(Handle *h) {
    if (h->marg) {
        if (h->marg->buf) cudaFree(h->marg->buf);
        delete h->marg;
        h->marg = nullptr;
    }
}

// keep_on_device (index 0 only): the new prior -- S, e and its linearisation point, the CURRENT states of the frames that
// stay -- is written straight into slot 0's prior arrays on the device; the next solve of the shifted window names it
// with prior_S == NULL (pack_window) and nothing of it crosses PCIe.
int marginalize_impl(Handle *h, const pvio_b200_window *w, const pvio_b200_state *s, int index, bool keep_on_device,
                     double *S_out, double *e_out, double *H_out, double *b_out) {
    const int N = w->n_frames;
    if (index < 0 || index >= N || N < 2) return fail(h, PVIO_B200_EINVAL, "marginalize: bad frame index");
    if (!w->use_inertial) return fail(h, PVIO_B200_EINVAL, "marginalize: the window must carry motion states");
    const int n = 15 * N, dk = n - 15;
    if (keep_on_device && index != 0) return fail(h, PVIO_B200_EINVAL, "marginalize: the resident prior is defined for index 0");
    if ((S_out || e_out || keep_on_device) && sizeof(double) * ((size_t)dk * (dk | 1) + 6 * (size_t)dk) > 226 * 1024)
        return fail(h, PVIO_B200_EINVAL, "marginalize: window too large for the shared-memory eigen-solver (15 (N - 1) <= 165)");
    int rc = pack_and_upload(h, w, s);
    if (rc != 0) return rc;
    // dense buffers: sized once from the handle's frame capacity
    const size_t ncap = 15 * (size_t)h->Ncap, dcap = ncap - 15;
    const size_t words = ncap * ncap + ncap + 3 * dcap * dcap + 2 * dcap + 2048 + 64 * (size_t)h->Ncap;
    if (!h->marg) h->marg = new MargScratch();
    if (h->marg->words < words) {
        if (h->marg->buf) cudaFree(h->marg->buf);
        h->marg->buf = nullptr; h->marg->words = 0;
        CK(h, cudaMalloc(&h->marg->buf, sizeof(double) * words));
        h->marg->words = words;
    }
    double *dH = h->marg->buf, *db = dH + ncap * ncap, *dHk = db + ncap, *dV = dHk + dcap * dcap, *dS = dV + dcap * dcap,
           *dbk = dS + dcap * dcap, *de = dbk + dcap, *dscr = de + dcap;
    // vision part: no loss, victim-seen landmarks only, mu = 0, fp64 (lin_obs_kernel<false, double> + schur_kernel<double>)
    rc = run_marg_vision(h);
    if (rc != 0) return rc;
    MargArgs m;
    m.hdr = h->hdr.d; m.cst = h->cst.d; m.frames = h->frames.d; m.Hred = h->Hred.d; m.gred = h->gred;
    m.imu_idx = h->imu_idx.d; m.imu_data = h->imu_data.d; m.prior_frames = h->prior_frames.d;
    m.prior_S = h->prior_S.d; m.prior_L = h->prior_L.d; m.prior_e = h->prior_e.d; m.prior_x0 = h->prior_x0.d;
    m.Ncap = h->Ncap; m.index = index; m.H = dH; m.b = db; m.scratch = dscr;
    marg_assemble_kernel<<<1, 256, 0, h->stream>>>(m);
    marg_reduce_kernel<<<1, 256, 0, h->stream>>>(dH, db, N, index, dHk, dbk);
    h->launches += 2;
    if (H_out) CK(h, cudaMemcpyAsync(H_out, dHk, sizeof(double) * dk * dk, cudaMemcpyDeviceToHost, h->stream));
    if (b_out) CK(h, cudaMemcpyAsync(b_out, dbk, sizeof(double) * dk, cudaMemcpyDeviceToHost, h->stream));
    if (S_out || e_out || keep_on_device) {
        // matrix + d, e + the ring of rotation batches (4 slots; 2 when the matrix leaves no room: dk = 165)
        const size_t esm4 = sizeof(double) * ((size_t)dk * (dk | 1) + 10 * (size_t)dk);
        const int ring = esm4 <= 226 * 1024 ? 4 : 2;
        const size_t esm = sizeof(double) * ((size_t)dk * (dk | 1) + (2 + 2 * (size_t)ring) * dk);
        static bool attr_set = false;
        if (!attr_set) { CK(h, cudaFuncSetAttribute(marg_eig_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024)); attr_set = true; }
        marg_eig_kernel<<<1, 256, esm, h->stream>>>(dHk, dbk, dk, ring, dS, de);
        ++h->launches;
        if (S_out) CK(h, cudaMemcpyAsync(S_out, dS, sizeof(double) * dk * dk, cudaMemcpyDeviceToHost, h->stream));
        if (e_out) CK(h, cudaMemcpyAsync(e_out, de, sizeof(double) * dk, cudaMemcpyDeviceToHost, h->stream));
        if (keep_on_device) {       // slot 0: dense dk x dk S, e, x0 = states of frames 1 .. N - 1 (read by the kernels above: stream order)
            CK(h, cudaMemcpyAsync(h->prior_S.d, dS, sizeof(double) * dk * dk, cudaMemcpyDeviceToDevice, h->stream));
            CK(h, cudaMemcpyAsync(h->prior_e.d, de, sizeof(double) * dk, cudaMemcpyDeviceToDevice, h->stream));
            CK(h, cudaMemcpyAsync(h->prior_x0.d, h->frames.d + kFrameStride, sizeof(double) * (N - 1) * kFrameStride, cudaMemcpyDeviceToDevice, h->stream));
        }
    }
    CK(h, cudaStreamSynchronize(h->stream));
    CK(h, cudaGetLastError());
    if (keep_on_device) { h->prior_resident = true; h->prior_resident_n = N - 1; }
    return 0;
}

}  // namespace pvio
