// libpvio_b200: C-ABI entry points (include/pvio_b200.h), host-side packing and launch
// orchestration of the bundle-adjustment kernels.  No torch types, no CPU fallback, no environment switches:
// one pipeline (frame-major table -> linearise -> Schur -> solve -> back-substitution / candidate), in fp32
// Jacobians for visual-only windows and fp64 for windows with motion states.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include "api_internal.h"
#include "ba_fobs.cuh"
#include "ba_linearize.cuh"
#include "ba_schur.cuh"
#include "ba_solve.cuh"
#include "ba_tr.cuh"
#include "ba_update.cuh"

namespace pvio {

int fail(Handle *h, int code, const char *what, cudaError_t e) {
    if (h) {
        h->err = what ? what : "";
        if (e != cudaSuccess) { h->err += ": "; h->err += cudaGetErrorString(e); }
    }
    return code;
}

// (re)allocates b: n zeroed elements on the device and, if pinned, in pinned host staging; what b held is freed first
template <typename T>
static int alloc(Handle *h, DevBuf<T> &b, size_t n, bool pinned) {
    b = DevBuf<T>();
    b.n = n;
    if (n == 0) return 0;
    CK(h, cudaMalloc(&b.d, n * sizeof(T)));
    CK(h, cudaMemset(b.d, 0, n * sizeof(T)));
    if (pinned) {
        CK(h, cudaMallocHost(&b.h, n * sizeof(T)));
        memset(b.h, 0, n * sizeof(T));
    }
    return 0;
}

SolveOpts solve_opts(const pvio_b200_options *opt) {
    SolveOpts o;
    if (opt) {
        o.max_iter = opt->max_iterations;
        if (opt->initial_trust_region_radius > 0) o.radius0 = opt->initial_trust_region_radius;
        o.alias_bias = opt->alias_bias;
        o.max_time = opt->max_time;
    }
    return o;
}

void drop_graphs(Handle *h) {
    for (auto &kv : h->graphs) cudaGraphExecDestroy(kv.second.first);
    h->graphs.clear();
}

// The per-window input arrays: pack_window fills their pinned staging, upload_range copies it to the device.
// f(m, n, g) is called for each array h->*m, with n elements per window and the array's group g, skipping the
// groups the handle has not allocated.  The prior arrays are allocated with the inertial ones; they are a group of
// their own because a device-resident prior is not uploaded.
enum InputGroup { kVision, kInertial, kPrior, kPlanes };

template <class F>
static int for_each_input(const Handle *h, F f) {
    const size_t N = h->Ncap, dcap = 15 * N;
    TRY(f(&Handle::hdr, 1, kVision));
    TRY(f(&Handle::cst, 1, kVision));
    TRY(f(&Handle::obs, h->Kcap, kVision));
    TRY(f(&Handle::lms, h->Mcap, kVision));
    TRY(f(&Handle::rho, h->Mcap, kVision));
    TRY(f(&Handle::frames, N * kFrameStride, kVision));
    if (h->have_inertial) {
        TRY(f(&Handle::imu_idx, N * 2, kInertial));
        TRY(f(&Handle::imu_data, N * kImuStride, kInertial));
        TRY(f(&Handle::prior_frames, N, kInertial));
        TRY(f(&Handle::prior_S, dcap * dcap, kPrior));
        TRY(f(&Handle::prior_e, dcap, kPrior));
        TRY(f(&Handle::prior_x0, N * kFrameStride, kPrior));
    }
    if (h->have_planes) {
        TRY(f(&Handle::plane_param, (size_t)h->Pcap * 4, kPlanes));
        TRY(f(&Handle::pt_plane, h->Tcap, kPlanes));
        TRY(f(&Handle::pt_begin, h->Tcap + 1, kPlanes));
        TRY(f(&Handle::pt_frame, h->Ocap, kPlanes));
        TRY(f(&Handle::pt_z, 2 * (size_t)h->Ocap, kPlanes));
    }
    return 0;
}

static int alloc_inertial(Handle *h) {
    const size_t W = h->W, N = h->Ncap, M = h->Mcap, dcap = 15 * N;
    TRY(for_each_input(h, [&](auto m, size_t per, InputGroup g) {
        return g == kInertial || g == kPrior ? alloc(h, h->*m, W * per, true) : 0;
    }));
    TRY(alloc(h, h->prior_L, W * dcap * dcap, false));
    // windows with motion states run the fp64 pipeline: h records of 8-byte elements
    TRY(alloc(h, h->hs, 2 * W * N * M * 6 * sizeof(double), false));      // two buffer sets (LinBufs)
    TRY(alloc(h, h->jr, 2 * W * N * M * 2 * sizeof(double), false));
    TRY(alloc(h, h->lm_w, 2 * W * M * 2 * sizeof(double), false));
    h->hs_double = true;
    return 0;
}

static int ensure_inertial(Handle *h) {
    if (h->have_inertial) return 0;
    cudaStreamSynchronize(h->stream);
    drop_graphs(h);                                 // the record array is reallocated below: pointers in cached graphs go stale
    h->have_inertial = true;                        // for_each_input visits the inertial arrays from here on
    const int rc = alloc_inertial(h);
    if (rc != 0) h->have_inertial = false;          // the next inertial window allocates again
    return rc;
}

// Plane buffers grow on demand WITHOUT losing the slots already packed into the pinned staging area
// (the device copies are refreshed by the next upload anyway).  The grown arrays replace the old ones only once all
// of them are allocated, so a failed allocation leaves the handle as it was.
static int ensure_planes(Handle *h, int T, int O) {
    if (h->have_planes && T <= h->Tcap && O <= h->Ocap) return 0;
    const size_t W = h->W;
    cudaStreamSynchronize(h->stream);
    drop_graphs(h);
    Handle g;                                       // capacities and arrays after the growth
    g.W = h->W; g.Pcap = h->Pcap; g.have_planes = true;
    g.Tcap = std::max({T, h->Tcap, 256}); g.Ocap = std::max({O, h->Ocap, 256 * 8});
    TRY(for_each_input(&g, [&](auto m, size_t per, InputGroup grp) {
        if (grp != kPlanes) return 0;
        auto &to = g.*m;
        const auto &from = h->*m;                   // empty before the first plane window
        TRY(alloc(h, to, W * per, true));
        const size_t old = from.n / W;              // old stride -> new stride, slot by slot
        for (size_t i = 0; i < W && old > 0; ++i) memcpy(to.h + i * per, from.h + i * old, sizeof(*to.h) * old);
        return 0;
    }));
    TRY(alloc(h, g.pt_J, W * g.Tcap * (6 * (size_t)h->Ncap + 2), false));      // device scratch of solve_kernel's plane block
    for_each_input(&g, [&](auto m, size_t, InputGroup grp) { if (grp == kPlanes) (h->*m).swap(g.*m); return 0; });
    h->pt_J.swap(g.pt_J);
    h->Tcap = g.Tcap; h->Ocap = g.Ocap;
    h->have_planes = true;
    return 0;
}

// ------------------------------------------------------------------------ small kernels
// Lambda = S^T S of the marginalisation prior (once per upload; constant across iterations)
__global__ void prior_lambda_kernel(const WinHdr *hdr, const double *S, double *L, int Ncap, int w0) {
    const int w = blockIdx.x + w0;
    const int d = 15 * hdr[w].n_prior, dcap = 15 * Ncap;
    const double *Sw = S + (size_t)w * dcap * dcap;
    double *Lw = L + (size_t)w * dcap * dcap;
    // gridDim.y CTAs share a window (a single window would otherwise leave 147 SMs idle for 0.29 ms)
    for (int e = blockIdx.y * blockDim.x + threadIdx.x; e < d * d; e += blockDim.x * gridDim.y) {
        const int i = e / d, j = e - i * d;
        double s = 0.0;
        for (int k = 0; k < d; ++k) s += Sw[(size_t)k * d + i] * Sw[(size_t)k * d + j];
        Lw[e] = s;
    }
}

// Landmark post-pass (bundle_adjustor.cpp:277-296): depth test in every observing camera
// (anchor included) and mean pixel reprojection error.  One group of 16 lanes per landmark.
__global__ void postpass_kernel(const WinHdr *hdr, const WinConst *cst, const ObsRec *obs, const LmRec *lms,
                                const double *rho, const double *frames, uint8_t *valid, double *quality,
                                double *err_acc, int Ncap, int Mcap, int Kcap, int w0) {
    const int w = blockIdx.y + w0;
    const WinHdr &H = hdr[w];
    const WinConst &wc = cst[w];
    __shared__ FrameSm F[kMaxFrames];
    if (threadIdx.x < H.N) make_frame(frames + ((size_t)w * Ncap + threadIdx.x) * kFrameStride, wc, F[threadIdx.x]);
    __syncthreads();
    const int lane = threadIdx.x & (kGroup - 1);
    const int gid = (blockIdx.x * blockDim.x + threadIdx.x) / kGroup;
    const int ngrp = gridDim.x * blockDim.x / kGroup;
    for (int l0 = 0; l0 < H.M; l0 += ngrp) {
        const int l = l0 + gid;
        const bool ok = l < H.M;
        const LmRec lr = lms[(size_t)w * Mcap + (ok ? l : 0)];
        const int n_obs = ok ? lm_nobs(lr.meta) : 0;
        const int anchor = lm_anchor(lr.meta);
        const unsigned fmask = ok ? lm_mask(lr.meta) : 0u;
        double x[3];
        float xf[3], cl[3];
        world_point(F[anchor], lr.zrx, lr.zry, ok ? rho[(size_t)w * Mcap + l] : 1.0, x, xf, cl);
        // lane = frame: its observation is record popc(mask below the lane); the anchor lane uses z_ref
        int frame = -1;
        float zx = 0.f, zy = 0.f;
        if ((fmask >> lane) & 1u) {
            const ObsRec o = obs[(size_t)w * Kcap + lr.obs_begin + __popc(fmask & ((1u << lane) - 1u))];
            frame = lane; zx = o.zx; zy = o.zy;
        } else if (lane == anchor && ok) {
            frame = anchor; zx = lr.zrx; zy = lr.zry;
        }
        double e = 0.0;
        int bad = 0;
        if (frame >= 0) {
            const FrameSm &Ft = F[frame];
            const double d0 = x[0] - Ft.c[0], d1 = x[1] - Ft.c[1], d2 = x[2] - Ft.c[2];
            const double y0 = Ft.Rwc[0] * d0 + Ft.Rwc[3] * d1 + Ft.Rwc[6] * d2;
            const double y1 = Ft.Rwc[1] * d0 + Ft.Rwc[4] * d1 + Ft.Rwc[7] * d2;
            const double y2 = Ft.Rwc[2] * d0 + Ft.Rwc[5] * d1 + Ft.Rwc[8] * d2;
            if (y2 <= 1.0e-3 || y2 > 50.0) bad = 1;                        // :286
            const double ex = (y0 / y2 - (double)zx) * wc.fx, ey = (y1 / y2 - (double)zy) * wc.fy;
            e = sqrt(ex * ex + ey * ey);                                   // :291
        }
        const unsigned badm = __ballot_sync(0xffffffffu, bad);
        const int grp_bad = (badm >> (threadIdx.x & 16)) & 0xffff;
#pragma unroll
        for (int off = kGroup / 2; off > 0; off >>= 1) e += __shfl_xor_sync(0xffffffffu, e, off, kGroup);
        if (ok && lane == 0) {
            const bool v = grp_bad == 0;
            if (valid) valid[(size_t)w * Mcap + l] = v ? 1 : 0;
            if (quality) quality[(size_t)w * Mcap + l] = v ? e / fmax((double)(n_obs + 1), 1.0) : 0.0;
            if (err_acc) { atomicAdd(&err_acc[2 * w], e); atomicAdd(&err_acc[2 * w + 1], (double)(n_obs + 1)); }
        }
    }
}

// ------------------------------------------------------------------------ packing
static int pack_window(Handle *h, int slot, const pvio_b200_window *w, const pvio_b200_state *s) {
    const int N = w->n_frames, M = w->n_landmarks, K = w->n_obs;
    if (slot < 0 || slot >= h->W) return fail(h, PVIO_B200_EINVAL, "slot out of range");
    if (N < 1 || N > h->Ncap || N > kMaxFrames || M > h->Mcap || K > h->Kcap || M < 0 || K < 0)
        return fail(h, PVIO_B200_EINVAL, "window exceeds the handle's capacity");
    if (!s->frames || (M > 0 && (!s->inv_depth || !w->lm_anchor || !w->lm_z_ref || !w->lm_obs_begin)) ||
        (K > 0 && (!w->obs_frame || !w->obs_z)))
        return fail(h, PVIO_B200_EINVAL, "null array in window / state");
    // every index array of the caller is range-checked here: bad indices would become device-side out-of-bounds accesses
    if (M > 0 && (w->lm_obs_begin[0] != 0 || w->lm_obs_begin[M] != K))
        return fail(h, PVIO_B200_EINVAL, "lm_obs_begin must start at 0 and end at n_obs");
    const bool inertial = w->use_inertial != 0;
    const int n_imu = inertial ? w->n_imu : 0, n_prior = inertial ? w->n_prior : 0;
    if (n_imu < 0 || n_prior < 0 || n_imu > h->Ncap || n_prior > h->Ncap || n_prior > N)
        return fail(h, PVIO_B200_EINVAL, "too many IMU / prior frames");
    for (int n = 0; n < n_imu; ++n) {
        const int i = w->imu_frame_i[n], j = w->imu_frame_j[n];
        if (i < 0 || i >= N || j < 0 || j >= N || i == j) return fail(h, PVIO_B200_EINVAL, "IMU factor with bad frame indices");
    }
    {
        unsigned seen = 0;
        for (int n = 0; n < n_prior; ++n) {
            const int f = w->prior_frames[n];
            if (f < 0 || f >= N || ((seen >> f) & 1u)) return fail(h, PVIO_B200_EINVAL, "prior_frames must be distinct window indices");
            seen |= 1u << f;
        }
    }
    if (w->n_plane_tracks < 0 || w->n_planes < 0 || w->n_planes > h->Pcap) return fail(h, PVIO_B200_EINVAL, "too many planes");
    if (w->n_plane_tracks > 0) {
        if (!w->pt_obs_begin || !w->pt_plane || !w->pt_obs_frame || !w->pt_obs_z || !w->plane_param || w->pt_obs_begin[0] != 0)
            return fail(h, PVIO_B200_EINVAL, "null / malformed plane-track arrays");
        for (int t = 0; t < w->n_plane_tracks; ++t) {
            const int len = w->pt_obs_begin[t + 1] - w->pt_obs_begin[t];
            if (len < 0 || len > kMaxFrames) return fail(h, PVIO_B200_EINVAL, "plane track too long / CSR offsets not monotone");
            if (w->pt_plane[t] < 0 || w->pt_plane[t] >= w->n_planes) return fail(h, PVIO_B200_EINVAL, "pt_plane out of range");
        }
        const int O = w->pt_obs_begin[w->n_plane_tracks];
        for (int i = 0; i < O; ++i)
            if (w->pt_obs_frame[i] < 0 || w->pt_obs_frame[i] >= N) return fail(h, PVIO_B200_EINVAL, "pt_obs_frame out of range");
    }
    if (n_imu > 0 || n_prior > 0 || inertial) TRY(ensure_inertial(h));
    WinHdr &H = h->hdr.h[slot];
    WinConst &C = h->cst.h[slot];
    memset(&H, 0, sizeof(H));
    H.N = N; H.M = M; H.K = K; H.use_inertial = inertial ? 1 : 0;
    for (int f = 0; f < N; ++f) if (w->frame_fixed && w->frame_fixed[f]) H.fixed_mask |= 1 << f;
    memcpy(C.cam_q, w->cam_q_cs, 32); memcpy(C.cam_p, w->cam_p_cs, 24);
    memcpy(C.imu_q, w->imu_q_cs, 32); memcpy(C.imu_p, w->imu_p_cs, 24);
    memcpy(C.sic, w->sqrt_inv_cov, 32);
    C.fx = w->fx; C.fy = w->fy; C.cauchy_a = w->cauchy_a > 0 ? w->cauchy_a : 1.0; C.plane_sic = w->plane_sqrt_inv_cov;
    // frames + origin (mean frame position keeps |x_l| ~ depth in the fp32 Jacobian arithmetic)
    double *fr = h->frames.h + (size_t)slot * h->Ncap * kFrameStride;
    memcpy(fr, s->frames, sizeof(double) * N * kFrameStride);
    double o[3] = {0, 0, 0};
    for (int f = 0; f < N; ++f) for (int k = 0; k < 3; ++k) o[k] += fr[f * kFrameStride + 4 + k];
    for (int k = 0; k < 3; ++k) C.origin[k] = o[k] / N;
    // landmarks sorted by anchor (the reference's first-visit order already is, bundle_adjustor.cpp:92-103)
    std::vector<int32_t> &perm = h->perm[slot];
    perm.resize(M);
    std::iota(perm.begin(), perm.end(), 0);
    bool sorted = true;
    for (int l = 0; l < M; ++l) {
        const int a = w->lm_anchor[l];
        if (a < 0 || a >= N) return fail(h, PVIO_B200_EINVAL, "landmark with bad anchor");
        if (l > 0 && a < w->lm_anchor[l - 1]) sorted = false;
    }
    if (!sorted) std::stable_sort(perm.begin(), perm.end(), [&](int a, int b) { return w->lm_anchor[a] < w->lm_anchor[b]; });
    ObsRec *ob = h->obs.h + (size_t)slot * h->Kcap;
    LmRec *lm = h->lms.h + (size_t)slot * h->Mcap;
    double *rh = h->rho.h + (size_t)slot * h->Mcap;
    int k_out = 0, nch = 0;
    for (int lp = 0; lp < M; ++lp) {
        const int l = perm[lp];
        const int a = w->lm_anchor[l];
        const int b0 = w->lm_obs_begin[l], b1 = w->lm_obs_begin[l + 1];
        const int n = b1 - b0;
        if (b0 < 0 || b1 > K || n < 0 || n >= kGroup) return fail(h, PVIO_B200_EINVAL, "landmark with bad observation range / too many observations");
        lm[lp].zrx = (float)w->lm_z_ref[2 * l];
        lm[lp].zry = (float)w->lm_z_ref[2 * l + 1];
        lm[lp].obs_begin = k_out;
        rh[lp] = s->inv_depth[l];
        // records in increasing frame order: the frame index lives in the landmark's mask, not in the record
        unsigned seen = 0;
        for (int k = b0; k < b1; ++k) {
            const int f = w->obs_frame[k];
            if (f <= a || f >= N || (seen >> f) & 1)
                return fail(h, PVIO_B200_EINVAL, "observation frames must be distinct and later than the anchor (Track::first_frame is the lowest id)");
            seen |= 1u << f;
        }
        if (k_out + n > h->Kcap) return fail(h, PVIO_B200_EINVAL, "observation table overflow");
        for (int k = b0; k < b1; ++k) {
            const int f = w->obs_frame[k];
            const int pos = k_out + __builtin_popcount(seen & ((1u << f) - 1u));
            ob[pos].zx = (float)w->obs_z[2 * k];
            ob[pos].zy = (float)w->obs_z[2 * k + 1];
        }
        k_out += n;
        lm[lp].meta = lm_meta(a, (w->lm_in_victim && w->lm_in_victim[l]) ? 1 : 0, n, seen);
        // chunks: <= kChunk landmarks of one anchor
        if (nch == 0 || (H.chunk_meta[nch - 1] >> 8) != a || (H.chunk_meta[nch - 1] & 0xff) == kChunk) {
            if (nch == kMaxChunks) return fail(h, PVIO_B200_EINVAL, "too many landmark chunks");
            H.chunk_begin[nch] = lp;
            H.chunk_meta[nch] = (a << 8);
            ++nch;
        }
        H.chunk_meta[nch - 1] += 1;
    }
    H.n_chunks = nch;
    H.K = k_out;
    h->slot_M[slot] = M; h->slot_N[slot] = N; h->slot_K[slot] = k_out;
    h->perm_identity[slot] = sorted ? 1 : 0;
    // inertial part
    H.n_imu = n_imu;
    H.n_prior = n_prior;
    if (n_imu > 0 || n_prior > 0) {
        int32_t *ii = h->imu_idx.h + (size_t)slot * h->Ncap * 2;
        for (int n = 0; n < n_imu; ++n) { ii[2 * n] = w->imu_frame_i[n]; ii[2 * n + 1] = w->imu_frame_j[n]; }
        if (n_imu > 0) memcpy(h->imu_data.h + (size_t)slot * h->Ncap * kImuStride, w->imu_data, sizeof(double) * n_imu * kImuStride);
        const size_t dcap = 15 * (size_t)h->Ncap, d = 15 * (size_t)n_prior;
        for (int n = 0; n < n_prior; ++n) h->prior_frames.h[(size_t)slot * h->Ncap + n] = w->prior_frames[n];
        if (d > 0 && !w->prior_S) {         // prior left on the device by marginalize_impl(keep_on_device): slot 0 only
            if (slot != 0 || !h->prior_resident || h->prior_resident_n != n_prior)
                return fail(h, PVIO_B200_EINVAL, "prior_S == NULL: no device-resident prior of that size");
        } else if (d > 0) {
            if (slot == 0) h->prior_resident = false;
            memcpy(h->prior_S.h + (size_t)slot * dcap * dcap, w->prior_S, sizeof(double) * d * d);   // dense d x d, row-major
            memcpy(h->prior_e.h + (size_t)slot * dcap, w->prior_e, sizeof(double) * d);
            memcpy(h->prior_x0.h + (size_t)slot * h->Ncap * kFrameStride, w->prior_state0, sizeof(double) * n_prior * kFrameStride);
        }
    }
    // planes
    H.n_planes = w->n_planes; H.n_ptracks = w->n_plane_tracks;
    if (H.n_ptracks > 0) {
        const int O = w->pt_obs_begin[H.n_ptracks];
        TRY(ensure_planes(h, H.n_ptracks, O));
        memcpy(h->plane_param.h + (size_t)slot * h->Pcap * 4, w->plane_param, sizeof(double) * 4 * H.n_planes);
        memcpy(h->pt_plane.h + (size_t)slot * h->Tcap, w->pt_plane, sizeof(int32_t) * H.n_ptracks);
        memcpy(h->pt_begin.h + (size_t)slot * (h->Tcap + 1), w->pt_obs_begin, sizeof(int32_t) * (H.n_ptracks + 1));
        memcpy(h->pt_frame.h + (size_t)slot * h->Ocap, w->pt_obs_frame, sizeof(int32_t) * O);
        float *z = h->pt_z.h + (size_t)slot * h->Ocap * 2;
        for (int i = 0; i < 2 * O; ++i) z[i] = (float)w->pt_obs_z[i];
    }
    return 0;
}

template <typename T>
static int h2d(Handle *h, DevBuf<T> &b, size_t per, int w0, int n, cudaStream_t st) {
    if (!b.d || !b.h || per == 0) return 0;
    CK(h, cudaMemcpyAsync(b.d + per * w0, b.h + per * w0, per * n * sizeof(T), cudaMemcpyHostToDevice, st));
    return 0;
}

// Host -> device copy of windows [w0, w0 + n) on stream st, then the device-side preparation that is constant
// across the iterations of a solve: the frame-major table and Lambda = S^T S of the priors.
static int upload_range(Handle *h, int w0, int n, cudaStream_t st) {
    if (n < 1 || w0 < 0 || w0 + n > h->W) return fail(h, PVIO_B200_EINVAL, "bad window range");
    const bool resident = w0 == 0 && n == 1 && h->prior_resident;     // a device-resident prior (marginalize_impl) is never re-uploaded
    TRY(for_each_input(h, [&](auto m, size_t per, InputGroup g) {
        return g == kPrior && resident ? 0 : h2d(h, h->*m, per, w0, n, st);
    }));
    bool any_prior = false;
    if (h->have_inertial) for (int i = w0; i < w0 + n; ++i) any_prior |= h->hdr.h[i].n_prior > 0;
    if (any_prior) {
        prior_lambda_kernel<<<dim3(n, n < 64 ? 32 : 1), 256, 0, st>>>(h->hdr.d, h->prior_S.d, h->prior_L.d, h->Ncap, w0);
        ++h->launches;
    }
    FobsArgs fa;
    fa.hdr = h->hdr.d; fa.obs = h->obs.d; fa.lms = h->lms.d; fa.fobs = h->fobs.d; fa.seg = h->seg.d;
    fa.Mcap = h->Mcap; fa.Kcap = h->Kcap; fa.w0 = w0;
    fobs_build_kernel<<<n, 256, 0, st>>>(fa);
    ++h->launches;
    CK(h, cudaGetLastError());
    return 0;
}

static int upload(Handle *h, int n) {
    TRY(upload_range(h, 0, n, h->stream));
    h->n_uploaded = n;
    return 0;
}

int pack_and_upload(Handle *h, const pvio_b200_window *w, const pvio_b200_state *s) {
    TRY(pack_window(h, 0, w, s));
    return upload(h, 1);
}

// ------------------------------------------------------------------------ launches
struct StepCfg {
    double mu = -1.0;              // < 0: per-window WinCtrl::mu
    double beta = 1.0;             // truncated Gauss-Newton step: step = beta * dx_gn
    int apply = 0;                 // plain GN step: the candidate becomes the state
    int compute_scale = 1;
    int alias_bias = 0;
    int dump = 0;
    int loop = 0;                  // kernels obey the per-window trust-region flags
    int w0 = 0;                    // first window (sub-batch pipelining)
    int fork_aux = 0;              // latency path: the non-vision candidate cost runs beside the candidate's linearisation sweep
    cudaStream_t stream = nullptr; // nullptr: the handle's stream
};

// what the windows [w0, w0 + n) need from the launch: worst case over the batch
struct BatchShape {
    int N = 1, M = 1, nfree = 1, D = 0;
    bool inertial = false, planes = false;
    size_t solve_smem_full = 0, solve_smem_lean = 0;
};

static size_t solve_smem_one(const WinHdr &H, bool lean) {
    size_t D = (H.use_inertial ? 15 : 6) * (size_t)H.N;
    if (lean) {                       // the lean kernel drops constant frames from the system
        const int nfree = H.N - __builtin_popcount((unsigned)H.fixed_mask & ((1u << H.N) - 1u));
        if (nfree > 0) D = 6 * (size_t)nfree;
    }
    const size_t nb = (D + 3) / 4, Dp = nb * 4;
    const size_t np_ = (size_t)H.N * (H.N + 1) / 2;
    size_t scr = lean ? Dp + 10 * 36 + 36 : std::max<size_t>(Dp, 2 * np_ * 36 + (size_t)H.N * 36 + (size_t)H.N * 12);   // X blocks, X T_g, diagonal, gradients
    if (H.use_inertial) scr = std::max<size_t>(scr, 8 * 450 + 8 * 16 + 8 * 480 + 8 * 225);      // kImuRound factors: raw J, r; whitened [J | r]; their W
    if (H.n_prior > 0) scr = std::max<size_t>(scr, 3 * 15 * (size_t)H.n_prior + 9 * (size_t)H.n_prior + 8 * 225);   // + one 15 x 15 block per warp
    return sizeof(double) * ((nb + 1) * (nb + 2) / 2 * 18 + 4 * Dp + (size_t)H.N * 36 + scr);   // tiles of kTP = 18 doubles (ba_solve.cuh)
}

static BatchShape batch_shape(Handle *h, int w0, int n, bool by_capacity) {
    BatchShape b;
    for (int i = w0; i < w0 + n; ++i) {
        const WinHdr &H = h->hdr.h[i];
        b.N = std::max(b.N, H.N); b.M = std::max(b.M, H.M);
        const unsigned allm = (1u << H.N) - 1u, freem = ~(unsigned)H.fixed_mask & allm;
        b.nfree = std::max(b.nfree, __builtin_popcount(freem));
        b.inertial |= H.use_inertial != 0;
        b.planes |= H.n_ptracks > 0;
        b.solve_smem_full = std::max(b.solve_smem_full, solve_smem_one(H, false));
        b.solve_smem_lean = std::max(b.solve_smem_lean, solve_smem_one(H, true));
    }
    if (by_capacity) {                 // graph-cached launches: shapes depend on the frame count (part of the graph key) only
        b.M = h->Mcap; b.nfree = b.N;
        WinHdr H;
        memset(&H, 0, sizeof(H));
        H.N = b.N; H.use_inertial = b.inertial ? 1 : 0; H.n_prior = b.inertial ? b.N : 0;
        b.solve_smem_full = solve_smem_one(H, false);
    }
    return b;
}

static LinBufs lin_bufs(Handle *h) {
    const size_t W = h->W, N = h->Ncap, M = h->Mcap, es = h->hs_double ? sizeof(double) : sizeof(float);
    LinBufs b;
    b.hs = W * N * M * 6 * es; b.jr = W * N * M * 2 * es; b.lm_w = W * M * 2 * es;
    b.lm_msk = W * M; b.lm_aux = W * M;
    b.Hred = h->sys_set; b.Hdd = h->sys_set; b.g = h->sys_set; b.cost = h->sys_set;
    return b;
}

static PipeArgs make_pipe_args(Handle *h, const StepCfg &c) {
    PipeArgs a;
    memset(&a, 0, sizeof(a));
    a.bufs = lin_bufs(h); a.frames_cand = h->frames_cand.d; a.rho_cand = h->rho_cand.d;
    a.hdr = h->hdr.d; a.cst = h->cst.d; a.fobs = h->fobs.d; a.seg = h->seg.d; a.lms = h->lms.d;
    a.rho = h->rho.d; a.frames = h->frames.d; a.ctrl = h->ctrl.d; a.lm_scale = h->lm_scale.d; a.lm_aux = h->lm_aux.d;
    a.jr = h->jr.d; a.hs = h->hs.d; a.lm_w = h->lm_w.d; a.lm_msk = h->lm_msk.d;
    a.Hred = h->Hred.d; a.Hdd = h->Hdd; a.gdir = h->gdir; a.gred = h->gred; a.cost_vis = h->cost_vis;
    a.Ncap = h->Ncap; a.Mcap = h->Mcap; a.Kcap = h->Kcap;
    a.compute_scale = c.compute_scale; a.victim_only = 0; a.mu_override = c.mu; a.w0 = c.w0; a.loop = c.loop;
    return a;
}

// CTAs per window of the sweeps: one once the batch fills the machine, otherwise a window is cut into row ranges
static int sweep_grid_x(Handle *h, int n) { return n * 2 < h->sm_count ? 16 : 1; }

// CTA shapes of the sweeps (fp32 pipeline): warps per CTA and resident CTAs per SM the register allocation targets.
// Compile-time constants, chosen by measurement (profiles/r02*.md); -D overrides exist for tuning builds only.
#ifndef PVIO_LIN_BLOCKS
#define PVIO_LIN_BLOCKS 4
#endif
#ifndef PVIO_SCHUR_BLOCKS
#define PVIO_SCHUR_BLOCKS 4
#endif
#ifndef PVIO_UPD_BLOCKS
#define PVIO_UPD_BLOCKS 8
#endif
constexpr int kLinWarps = 4, kLinBlocks = PVIO_LIN_BLOCKS;
constexpr int kSchurThreads = 128, kSchurBlocks = PVIO_SCHUR_BLOCKS;
constexpr int kUpdWarps = 4, kUpdBlocks = PVIO_UPD_BLOCKS;

template <typename real>
static size_t schur_launch_smem(int N, int nfree) { return schur_smem_bytes<real>(N, kSchurThreads, nfree); }

#define LAUNCH_CK(h, what)                                                                        \
    do {                                                                                          \
        cudaError_t e__ = cudaGetLastError();                                                     \
        if (e__ != cudaSuccess) return fail((h), PVIO_B200_ECUDA, "launch of " what, e__);        \
    } while (0)

// linearise + Schur stage of windows [w0, w0 + n)
// zeroes the direct / reduced system of the buffer set a sweep is about to accumulate into with atomics (several CTAs
// per window: the latency path)
static __global__ void zero_system_kernel(PipeArgs a_in, int npairs_cap) {
    PipeArgs a = a_in;
    const int w = blockIdx.x + a.w0;
    const int bsel = pipe_buffer(a, w);
    if (bsel < 0) return;
    pipe_select(a, bsel);
    double *Hred = a.Hred + (size_t)w * npairs_cap * 36, *Hdd = a.Hdd + (size_t)w * a.Ncap * 36;
    double *gdir = a.gdir + (size_t)w * a.Ncap * 6, *gred = a.gred + (size_t)w * a.Ncap * 6;
    for (int i = threadIdx.x; i < npairs_cap * 36; i += blockDim.x) Hred[i] = 0.0;
    for (int i = threadIdx.x; i < a.Ncap * 36; i += blockDim.x) Hdd[i] = 0.0;
    for (int i = threadIdx.x; i < a.Ncap * 6; i += blockDim.x) { gdir[i] = 0.0; gred[i] = 0.0; }
    if (threadIdx.x == 0) a.cost_vis[w] = 0.0;
}

// linearise sweep (+ per-landmark completion as its own launch when several CTAs share a window).  spec: the
// speculative sweep of the trust-region loop over the CANDIDATE, into the window's other buffer set (ba_tr.cuh).
static int launch_lin(Handle *h, int n, const StepCfg &c, const BatchShape &b, bool loss, bool victim_only, bool spec) {
    cudaStream_t st = c.stream ? c.stream : h->stream;
    const int gx = sweep_grid_x(h, n);
    PipeArgs a = make_pipe_args(h, c);
    a.victim_only = victim_only ? 1 : 0;
    a.spec = spec ? 1 : 0;
    if (gx > 1) {
        zero_system_kernel<<<n, 256, 0, st>>>(a, h->Ncap * (h->Ncap + 1) / 2);
        ++h->launches;
        LAUNCH_CK(h, "zero_system_kernel");
    }
    const int Mp = (b.M + 31) & ~31;
    if (!h->hs_double) {
        if (!loss) return fail(h, PVIO_B200_EINVAL, "the loss-free sweep runs in fp64");
        lin_obs_kernel<true, float, kLinWarps, kLinBlocks><<<dim3(gx, n), kLinWarps * 32, lin_smem_bytes<float>(b.N, Mp, kLinWarps), st>>>(a);
        LAUNCH_CK(h, "lin_obs_kernel<float>");
        if (gx > 1) { lm_finish_kernel<float><<<dim3((b.M + 127) / 128, n), 128, 0, st>>>(a); ++h->launches; LAUNCH_CK(h, "lm_finish_kernel<float>"); }
    } else {
        if (loss) lin_obs_kernel<true, double, kLinWarps, 2><<<dim3(gx, n), kLinWarps * 32, lin_smem_bytes<double>(b.N, Mp, kLinWarps), st>>>(a);
        else lin_obs_kernel<false, double, kLinWarps, 2><<<dim3(gx, n), kLinWarps * 32, lin_smem_bytes<double>(b.N, Mp, kLinWarps), st>>>(a);
        LAUNCH_CK(h, "lin_obs_kernel<double>");
        if (gx > 1) { lm_finish_kernel<double><<<dim3((b.M + 127) / 128, n), 128, 0, st>>>(a); ++h->launches; LAUNCH_CK(h, "lm_finish_kernel<double>"); }
    }
    ++h->launches;
    return 0;
}

static int launch_schur(Handle *h, int n, const StepCfg &c, const BatchShape &b, bool victim_only) {
    cudaStream_t st = c.stream ? c.stream : h->stream;
    const int gx = sweep_grid_x(h, n);
    PipeArgs a = make_pipe_args(h, c);
    a.victim_only = victim_only ? 1 : 0;
    const int sgx = std::min(gx, std::max(1, (b.M + kSlab - 1) / kSlab));
    if (!h->hs_double) {
        schur_kernel<float, kSchurThreads, kSchurBlocks><<<dim3(sgx, n), kSchurThreads, schur_launch_smem<float>(b.N, b.nfree), st>>>(a);
        LAUNCH_CK(h, "schur_kernel<float>");
    } else {
        schur_kernel<double, kSchurThreads, 1><<<dim3(sgx, n), kSchurThreads, schur_launch_smem<double>(b.N, b.nfree), st>>>(a);
        LAUNCH_CK(h, "schur_kernel<double>");
    }
    ++h->launches;
    return 0;
}

// the linearise + Schur stage at the state; its two halves are timed by events when it is the plain batched step
static int run_linearize(Handle *h, int n, const StepCfg &c, const BatchShape &b, bool loss = true, bool victim_only = false) {
    cudaStream_t st = c.stream ? c.stream : h->stream;
    if (h->kev.empty()) {
        h->kev.resize(3 * 256);
        for (auto &e : h->kev) CK(h, cudaEventCreate(&e));
    }
    const int slot = (h->kev_count % 256) * 3;
    const bool timed = !h->capturing && !c.loop && st == h->stream;   // stage times are a property of the plain batched step
    if (timed) CK(h, cudaEventRecord(h->kev[slot], st));
    TRY(launch_lin(h, n, c, b, loss, victim_only, false));
    if (timed) CK(h, cudaEventRecord(h->kev[slot + 1], st));
    TRY(launch_schur(h, n, c, b, victim_only));
    if (timed) { CK(h, cudaEventRecord(h->kev[slot + 2], st)); ++h->kev_count; }
    return 0;
}

int run_marg_vision(Handle *h) {
    StepCfg c;
    c.mu = 0.0; c.compute_scale = 1;
    const BatchShape b = batch_shape(h, 0, 1, false);
    return run_linearize(h, 1, c, b, false, true);
}

static int run_solve(Handle *h, int n, const StepCfg &c, const BatchShape &b) {
    SolveArgs a;
    memset(&a, 0, sizeof(a));
    a.hdr = h->hdr.d; a.cst = h->cst.d; a.frames = h->frames.d; a.ctrl = h->ctrl.d;
    a.Hred = h->Hred.d; a.Hdd = h->Hdd; a.gdir = h->gdir; a.gred = h->gred; a.cost_vis = h->cost_vis;
    a.imu_idx = h->imu_idx.d; a.imu_data = h->imu_data.d; a.alias_bias = c.alias_bias;
    a.prior_frames = h->prior_frames.d; a.prior_S = h->prior_S.d; a.prior_L = h->prior_L.d; a.prior_e = h->prior_e.d;
    a.prior_x0 = h->prior_x0.d;
    a.plane_param = h->plane_param.d; a.pt_plane = h->pt_plane.d; a.pt_begin = h->pt_begin.d; a.pt_frame = h->pt_frame.d;
    a.pt_z = h->pt_z.d; a.Pcap = h->Pcap; a.Tcap = h->Tcap; a.Ocap = h->Ocap; a.pt_J = h->pt_J.d;
    a.pose_scale = h->pose_scale.d; a.dx_pose = h->dx_pose.d; a.v_pose = h->v_pose.d;
    a.Hfull = c.dump ? h->Hfull.d : nullptr; a.gfull = c.dump ? h->gfull.d : nullptr;
    a.Ncap = h->Ncap; a.compute_scale = c.compute_scale; a.mu_override = c.mu; a.w0 = c.w0; a.loop = c.loop;
    a.bufs = lin_bufs(h);
    cudaStream_t st = c.stream ? c.stream : h->stream;
    // visual-only batches: the lean kernel (no IMU / prior / plane code, no full staging), a narrow CTA
    // per window so that many windows are resident per SM; otherwise the full kernel with a wide CTA
    const bool visual = n >= 64 && !b.inertial && !b.planes && b.solve_smem_lean <= 48 * 1024;
    const size_t smem = visual ? b.solve_smem_lean : b.solve_smem_full;
    if (smem > 220 * 1024) return fail(h, PVIO_B200_EINVAL, "reduced system too large for shared memory");
    if (visual) solve_kernel_visual<<<n, 64, smem, st>>>(a);
    else solve_kernel<<<n, 256, smem, st>>>(a);
    ++h->launches;
    LAUNCH_CK(h, "solve_kernel");
    return 0;
}

static CostArgs make_cost_args(Handle *h, const StepCfg &c) {
    CostArgs k;
    memset(&k, 0, sizeof(k));
    k.hdr = h->hdr.d; k.cst = h->cst.d; k.frames_cand = h->frames_cand.d; k.frames_cur = h->frames.d;
    k.imu_idx = h->imu_idx.d; k.imu_data = h->imu_data.d; k.alias_bias = c.alias_bias;
    k.prior_frames = h->prior_frames.d; k.prior_S = h->prior_S.d; k.prior_e = h->prior_e.d; k.prior_x0 = h->prior_x0.d;
    k.plane_param = h->plane_param.d; k.pt_plane = h->pt_plane.d; k.pt_begin = h->pt_begin.d; k.pt_frame = h->pt_frame.d;
    k.pt_z = h->pt_z.d; k.Pcap = h->Pcap; k.Tcap = h->Tcap; k.Ocap = h->Ocap; k.Ncap = h->Ncap; k.out = h->aux_cost.d;
    k.w0 = c.w0;
    k.ctrl = h->ctrl.d; k.acc = h->acc.d; k.frames_state = h->frames.d; k.rho_state = h->rho.d; k.rho_cand = h->rho_cand.d;
    k.Mcap = h->Mcap; k.loop = c.loop; k.apply = c.apply; k.beta = c.beta;
    k.cost_vis = h->cost_vis; k.cost_stride = h->sys_set;
    return k;
}

static UpdArgs make_upd_args(Handle *h, const StepCfg &c) {
    UpdArgs u;
    memset(&u, 0, sizeof(u));
    u.hdr = h->hdr.d; u.cst = h->cst.d; u.obs = h->obs.d; u.lms = h->lms.d; u.rho = h->rho.d; u.frames = h->frames.d;
    u.ctrl = h->ctrl.d; u.lm_scale = h->lm_scale.d; u.lm_aux = h->lm_aux.d; u.hs = h->hs.d;
    u.fobs = h->fobs.d; u.seg = h->seg.d; u.dx_pose = h->dx_pose.d;
    u.rho_cand = h->rho_cand.d; u.frames_cand = h->frames_cand.d; u.dx_lm = h->dx_lm.d; u.lm_v = h->lm_v.d; u.acc = h->acc.d;
    u.Ncap = h->Ncap; u.Mcap = h->Mcap; u.Kcap = h->Kcap; u.mu_override = c.mu; u.w0 = c.w0;
    u.step_a = 0.0; u.step_b = c.beta; u.v_pose = h->v_pose.d; u.loop = c.loop;
    u.bufs = lin_bufs(h);
    return u;
}

template <int kMode>
static int launch_update(Handle *h, int n, const StepCfg &c, const BatchShape &b, int gx) {
    cudaStream_t st = c.stream ? c.stream : h->stream;
    const UpdArgs u = make_upd_args(h, c);
    const int Mp = (b.M + 31) & ~31;
    constexpr int kW = kUpdWarps;
    constexpr int kB = 4, kBf = kUpdBlocks;
    if (kMode == 1 && n * 2 < h->sm_count) {        // latency path: one wide CTA per window for the back-substitution
        if (!h->hs_double) update_obs_kernel<true, float, 8, 2, 1><<<dim3(gx, n), 256, upd_smem_bytes<float>(b.N, Mp, 8), st>>>(u);
        else update_obs_kernel<true, double, 8, 2, 1><<<dim3(gx, n), 256, upd_smem_bytes<double>(b.N, Mp, 8), st>>>(u);
    }
    else if (!h->hs_double) update_obs_kernel<true, float, kW, kBf, kMode><<<dim3(gx, n), kW * 32, upd_smem_bytes<float>(b.N, Mp, kW), st>>>(u);
    else update_obs_kernel<true, double, kW, kB, kMode><<<dim3(gx, n), kW * 32, upd_smem_bytes<double>(b.N, Mp, kW), st>>>(u);
    ++h->launches;
    LAUNCH_CK(h, "update_obs_kernel");
    return 0;
}

// part 0: cost + decision in one launch; 1: cost only, on stream `on`; 2: decision only (aux_cost_kernel)
static int launch_aux_cost(Handle *h, int n, const StepCfg &c, const BatchShape &b, int part = 0, cudaStream_t on = nullptr) {
    cudaStream_t st = on ? on : (c.stream ? c.stream : h->stream);
    const CostArgs k = make_cost_args(h, c);
    // inertial windows: 8 warps share the prior's S r0 product; reprojection-only batches only need the acceptance copy
    const int threads = (b.inertial && part != 2) ? 256 : 64;
    const size_t smem = sizeof(double) * 2 * 15 * kMaxFrames;
    if (part == 1) aux_cost_kernel<1><<<n, threads, smem, st>>>(k);
    else if (part == 2) aux_cost_kernel<2><<<n, threads, smem, st>>>(k);
    else aux_cost_kernel<0><<<n, threads, smem, st>>>(k);
    ++h->launches;
    LAUNCH_CK(h, "aux_cost_kernel");
    return 0;
}

// One plain Gauss-Newton iteration (fixed mu, step beta * dx_gn): linearise, Schur, solve, back-substitution +
// candidate in one sweep, non-vision cost + optional acceptance.  5 launches.
static int run_gn_step(Handle *h, int n, const StepCfg &c, const BatchShape &b) {
    cudaStream_t st = c.stream ? c.stream : h->stream;
    TRY(run_linearize(h, n, c, b));
    TRY(run_solve(h, n, c, b));
    CK(h, cudaMemsetAsync(h->acc.d + (size_t)kAcc * c.w0, 0, sizeof(double) * kAcc * n, st));
    TRY(launch_update<0>(h, n, c, b, sweep_grid_x(h, n)));
    TRY(launch_aux_cost(h, n, c, b));
    return 0;
}

// One iteration of the device-side trust-region loop (ba_tr.cuh): 8 launches (9 in the first body), no host decision.
// The linearisation of the STATE is launched in the first body only: afterwards the state's linearisation is either the
// accepted candidate's (buffer swap) or still valid (rejected step), and the one case that invalidates it -- a failed
// linear solve, retried with mu * 10 -- is relinearised by the candidate sweep of the same body (pipe_buffer).
static int iteration_body(Handle *h, int n, const StepCfg &c, const BatchShape &b, bool first) {
    cudaStream_t st = c.stream ? c.stream : h->stream;
    if (first) TRY(launch_lin(h, n, c, b, true, false, false));
    TRY(launch_schur(h, n, c, b, false));
    TRY(run_solve(h, n, c, b));
    TRY(launch_update<1>(h, n, c, b, 1));
    {
        const UpdArgs u = make_upd_args(h, c);
        jv_vision_kernel<true><<<dim3(sweep_grid_x(h, n), n), kLinThreads, 0, st>>>(u);
        LAUNCH_CK(h, "jv_vision_kernel");
        JvAuxArgs ja;
        ja.c = make_cost_args(h, c);
        ja.v_pose = h->v_pose.d; ja.acc = h->acc.d;
        jv_aux_kernel<<<n, 64, sizeof(double) * 15 * kMaxFrames, st>>>(ja);
        LAUNCH_CK(h, "jv_aux_kernel");
        h->launches += 2;
    }
    TRY(launch_update<2>(h, n, c, b, 1));
    const bool fork = c.fork_aux && (b.inertial || b.planes);   // the candidate's IMU / prior / plane cost on a parallel branch
    if (fork) {
        CK(h, cudaEventRecord(h->ev_aux_fork, st));
        CK(h, cudaStreamWaitEvent(h->stream_aux, h->ev_aux_fork, 0));
        TRY(launch_aux_cost(h, n, c, b, 1, h->stream_aux));
        CK(h, cudaEventRecord(h->ev_aux_join, h->stream_aux));
    }
    TRY(launch_lin(h, n, c, b, true, false, true));      // the candidate's linearisation: its cost decides, its Jacobians stay
    if (fork) {
        CK(h, cudaStreamWaitEvent(st, h->ev_aux_join, 0));
        TRY(launch_aux_cost(h, n, c, b, 2));
    } else {
        TRY(launch_aux_cost(h, n, c, b));
    }
    return 0;
}

// The whole trust-region solve of the uploaded windows [w0, w0 + n) on stream st: init + max_iter (+ spare) identical
// bodies.  For the latency path (few windows from 0 on the handle's stream) the sequence is captured once into a CUDA
// graph keyed by (n, max_iter, flags) with capacity-sized launch shapes, and replayed: ONE launch per solve, no
// device -> host traffic inside.
static int run_solve_loop(Handle *h, int w0, int n, cudaStream_t st, const SolveOpts &o) {
    StepCfg c;
    c.mu = -1.0; c.loop = 1; c.alias_bias = o.alias_bias; c.compute_scale = 0; c.w0 = w0; c.stream = st;
    const bool graphable = w0 == 0 && st == h->stream && n * 2 < h->sm_count;
    const BatchShape b = batch_shape(h, w0, n, graphable);
    const int bodies = o.max_iter + 2;               // spare bodies absorb retries of a failed linear solve (mu *= 10)
    init_ctrl_kernel<<<n, 32, 0, st>>>(h->ctrl.d, 1e-8, o.radius0, o.max_iter, o.max_time, w0);
    ++h->launches;
    LAUNCH_CK(h, "init_ctrl_kernel");
    if (!graphable) {
        for (int it = 0; it < bodies; ++it) TRY(iteration_body(h, n, c, b, it == 0));
        return 0;
    }
    const Handle::GraphKey key(1, n, o.max_iter, (o.alias_bias ? 1 : 0) | (b.inertial ? 2 : 0) | (b.planes ? 4 : 0) | (h->hs_double ? 8 : 0) | (b.N << 4));
    auto it = h->graphs.find(key);
    if (it == h->graphs.end()) {
        if (h->graphs.size() >= 16) drop_graphs(h);
        const int64_t l0 = h->launches;
        cudaGraph_t g = nullptr;
        cudaGraphExec_t ge = nullptr;
        if (!h->stream_aux) {
            CK(h, cudaStreamCreateWithFlags(&h->stream_aux, cudaStreamNonBlocking));
            CK(h, cudaEventCreateWithFlags(&h->ev_aux_fork, cudaEventDisableTiming));
            CK(h, cudaEventCreateWithFlags(&h->ev_aux_join, cudaEventDisableTiming));
        }
        c.fork_aux = 1;                // a second branch of the graph (captured through h->stream_aux)
        CK(h, cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
        h->capturing = true;
        int rc = 0;
        for (int i = 0; i < bodies && rc == 0; ++i) rc = iteration_body(h, n, c, b, i == 0);
        h->capturing = false;
        const cudaError_t e = cudaStreamEndCapture(h->stream, &g);
        if (rc != 0) { if (g) cudaGraphDestroy(g); return rc; }
        if (e != cudaSuccess) return fail(h, PVIO_B200_ECUDA, "cudaStreamEndCapture", e);
        CK(h, cudaGraphInstantiate(&ge, g, 0));
        cudaGraphDestroy(g);
        const int nl = (int)(h->launches - l0);
        h->launches = l0;
        it = h->graphs.emplace(key, std::make_pair(ge, nl)).first;
    }
    CK(h, cudaGraphLaunch(it->second.first, h->stream));
    h->launches += it->second.second;
    return 0;
}

static int run_postpass(Handle *h, int n, bool want_flags, double *err_acc) {
    postpass_kernel<<<dim3(n * 2 < h->sm_count ? 8 : 1, n), 256, 0, h->stream>>>(
        h->hdr.d, h->cst.d, h->obs.d, h->lms.d, h->rho.d, h->frames.d, want_flags ? h->valid.d : nullptr,
        want_flags ? h->quality.d : nullptr, err_acc, h->Ncap, h->Mcap, h->Kcap, 0);
    ++h->launches;
    CK(h, cudaGetLastError());
    return 0;
}

// pinned staging -> caller arrays (landmark order un-permuted), windows [w0, w0 + n)
static int scatter_dx(Handle *h, int w0, int n, double *dx, int64_t dx_stride, double *costs) {
    for (int i = w0; i < w0 + n; ++i) {
        const int N = h->slot_N[i], M = h->slot_M[i];
        if (dx) {
            double *o = dx + (size_t)i * dx_stride;
            memcpy(o, h->dx_pose.h + (size_t)i * h->Ncap * 15, sizeof(double) * N * 15);
            const double *dl = h->dx_lm.h + (size_t)i * h->Mcap;
            if (h->perm_identity[i]) memcpy(o + N * 15, dl, sizeof(double) * M);
            else { const std::vector<int32_t> &perm = h->perm[i]; for (int lp = 0; lp < M; ++lp) o[N * 15 + perm[lp]] = dl[lp]; }
        }
        if (costs) { costs[2 * i] = h->ctrl.h[i].cost; costs[2 * i + 1] = h->ctrl.h[i].cand_cost; }
        if (h->ctrl.h[i].solve_failed) return fail(h, PVIO_B200_ENUMERIC, "reduced system not positive definite");
    }
    return 0;
}

// device -> host of the steps + control records of windows [w0, w0 + n) on stream st (async)
static int download_dx_async(Handle *h, int w0, int n, cudaStream_t st) {
    const size_t N = h->Ncap;
    CK(h, cudaMemcpyAsync(h->dx_pose.h + (size_t)w0 * N * 15, h->dx_pose.d + (size_t)w0 * N * 15, sizeof(double) * N * 15 * n,
                          cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemcpyAsync(h->dx_lm.h + (size_t)w0 * h->Mcap, h->dx_lm.d + (size_t)w0 * h->Mcap, sizeof(double) * h->Mcap * n,
                          cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemcpyAsync(h->ctrl.h + w0, h->ctrl.d + w0, sizeof(WinCtrl) * n, cudaMemcpyDeviceToHost, st));
    return 0;
}

static int download_dx(Handle *h, int n, double *dx, int64_t dx_stride, double *costs) {
    if (n < 1 || n > h->W) return fail(h, PVIO_B200_EINVAL, "bad window count");
    TRY(download_dx_async(h, 0, n, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    return scatter_dx(h, 0, n, dx, dx_stride, costs);
}

// device -> host of the solved state + summaries of windows [w0, w0 + n) on stream st (async)
static int download_state_async(Handle *h, int w0, int n, cudaStream_t st) {
    const size_t N = h->Ncap;
    CK(h, cudaMemcpyAsync(h->frames_out.h + (size_t)w0 * N * kFrameStride, h->frames.d + (size_t)w0 * N * kFrameStride,
                          sizeof(double) * N * kFrameStride * n, cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemcpyAsync(h->rho_out.h + (size_t)w0 * h->Mcap, h->rho.d + (size_t)w0 * h->Mcap, sizeof(double) * h->Mcap * n,
                          cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemcpyAsync(h->ctrl.h + w0, h->ctrl.d + w0, sizeof(WinCtrl) * n, cudaMemcpyDeviceToHost, st));
    return 0;
}

static void fill_summary(const WinCtrl &c, pvio_b200_summary *sm) {
    memset(sm, 0, sizeof(*sm));
    sm->iterations = c.iteration; sm->accepted_steps = c.accepted; sm->termination = c.termination; sm->usable = c.usable;
    sm->initial_cost = c.initial_cost; sm->final_cost = c.cost; sm->final_radius = c.radius; sm->final_mu = c.mu;
}

// downloaded states -> caller arrays (landmark order un-permuted) and summaries, windows [w0, w0 + n)
static void scatter_states(Handle *h, int w0, int n, double *frames, int64_t frames_stride, double *inv_depth,
                           int64_t inv_depth_stride, pvio_b200_summary *summaries) {
    for (int i = w0; i < w0 + n; ++i) {
        const int N = h->slot_N[i], M = h->slot_M[i];
        if (frames)
            memcpy(frames + (size_t)i * frames_stride, h->frames_out.h + (size_t)i * h->Ncap * kFrameStride, sizeof(double) * N * kFrameStride);
        if (inv_depth) {
            double *o = inv_depth + (size_t)i * inv_depth_stride;
            const double *r = h->rho_out.h + (size_t)i * h->Mcap;
            const std::vector<int32_t> &perm = h->perm[i];
            if (h->perm_identity[i]) memcpy(o, r, sizeof(double) * M);
            else for (int lp = 0; lp < M; ++lp) o[perm[lp]] = r[lp];
        }
        if (summaries) fill_summary(h->ctrl.h[i], &summaries[i]);
    }
}

// sub-batch schedule of the pipelined host paths: small batches first and last (the first upload and the last
// kernels + download are the only parts of the pipeline that nothing overlaps), 512-window batches in between
#ifndef PVIO_PIPE_STREAMS
#define PVIO_PIPE_STREAMS 6
#endif
#ifndef PVIO_PIPE_CHUNK
#define PVIO_PIPE_CHUNK 512
#endif
static constexpr int kPipeStreams = PVIO_PIPE_STREAMS;   // sub-batches in flight on the SMs at once (each alone is latency-bound: one wave)
static std::vector<int> sub_batches(int n) {
    std::vector<int> sizes;
    if (n < 1024) { sizes.push_back(n); return sizes; }
    int mid = n - 2 * (128 + 256);
    sizes.push_back(128); sizes.push_back(256);
    while (mid > 0) { const int m = std::min(PVIO_PIPE_CHUNK, mid); sizes.push_back(m); mid -= m; }
    sizes.push_back(256); sizes.push_back(128);
    return sizes;
}

static int ensure_pipeline_streams(Handle *h, int nsub) {
    if (!h->stream_up) {
        CK(h, cudaStreamCreateWithFlags(&h->stream_up, cudaStreamNonBlocking));
        CK(h, cudaStreamCreateWithFlags(&h->stream_down, cudaStreamNonBlocking));
    }
    while ((int)h->ev_up.size() < nsub) {
        cudaEvent_t a, b, c_;
        CK(h, cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
        CK(h, cudaEventCreateWithFlags(&b, cudaEventDisableTiming));
        CK(h, cudaEventCreateWithFlags(&c_, cudaEventDisableTiming));
        h->ev_up.push_back(a); h->ev_done.push_back(b); h->ev_down.push_back(c_);
    }
    if (h->stream_c.empty()) {
        h->stream_c.resize(kPipeStreams);
        for (auto &st : h->stream_c) CK(h, cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        CK(h, cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    }
    return 0;
}

// Upload, compute and download of windows [0, n) with HOST buffers.  Large batches are cut into sub-batches and
// pipelined over three streams: host->device copy of sub-batch i+1 overlaps the kernels of sub-batch i and the
// device->host copy of sub-batch i-1 (PCIe is full duplex), so the call costs max(copy, compute) instead of their sum.
// The kernels of sub-batch i run on compute stream i % kPipeStreams (a sub-batch is at most one wave of CTAs, so alone
// it runs at the latency of its kernel chain; several in flight fill the SMs); the windows of different sub-batches
// share nothing on the device.  compute(w0, m, stream) and download(w0, m, stream) enqueue, scatter(w0, m) copies a
// landed sub-batch to the caller while the GPU works on the later ones.
template <class Compute, class Download, class Scatter>
static int run_pipelined(Handle *h, int n, Compute compute, Download download, Scatter scatter) {
    if (n < 1 || n > h->W) return fail(h, PVIO_B200_EINVAL, "bad window count");
    const std::vector<int> sizes = sub_batches(n);
    const int nsub = (int)sizes.size();
    if (nsub == 1) {
        TRY(upload(h, n));
        TRY(compute(0, n, h->stream));
        TRY(download(0, n, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
        return scatter(0, n);
    }
    std::vector<int> starts(nsub, 0);
    for (int i = 1; i < nsub; ++i) starts[i] = starts[i - 1] + sizes[i - 1];
    TRY(ensure_pipeline_streams(h, nsub));
    CK(h, cudaEventRecord(h->ev_fork, h->stream));
    CK(h, cudaStreamWaitEvent(h->stream_up, h->ev_fork, 0));
    for (auto &sc : h->stream_c) CK(h, cudaStreamWaitEvent(sc, h->ev_fork, 0));
    for (int i = 0; i < nsub; ++i) {
        const int w0 = starts[i], m = sizes[i];
        cudaStream_t sc = h->stream_c[i % kPipeStreams];
        TRY(upload_range(h, w0, m, h->stream_up));
        CK(h, cudaEventRecord(h->ev_up[i], h->stream_up));
        CK(h, cudaStreamWaitEvent(sc, h->ev_up[i], 0));
        TRY(compute(w0, m, sc));
        CK(h, cudaEventRecord(h->ev_done[i], sc));
        CK(h, cudaStreamWaitEvent(h->stream_down, h->ev_done[i], 0));
        CK(h, cudaStreamWaitEvent(h->stream, h->ev_done[i], 0));      // later calls on the handle's stream see the result
        TRY(download(w0, m, h->stream_down));
        CK(h, cudaEventRecord(h->ev_down[i], h->stream_down));
    }
    h->n_uploaded = n;
    for (int i = 0; i < nsub; ++i) {
        CK(h, cudaEventSynchronize(h->ev_down[i]));
        TRY(scatter(starts[i], sizes[i]));
    }
    CK(h, cudaStreamSynchronize(h->stream));
    return 0;
}

}  // namespace pvio

using namespace pvio;

// ======================================================================== C ABI
extern "C" {

const char *pvio_b200_version(void) { return "pvio_b200 0.2 (sm_100a)"; }

int pvio_b200_create(int device, int max_windows, int max_frames, int max_landmarks, int max_obs,
                     pvio_b200_handle *out) {
    if (!out) return PVIO_B200_EINVAL;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device >= ndev || device < 0) return PVIO_B200_ENODEV;
    if (max_windows < 1 || max_frames < 1 || max_frames > kMaxFrames || max_landmarks < 1 || max_landmarks > 65534 || max_obs < 1)
        return PVIO_B200_EINVAL;
    Handle *h = new Handle();
    h->device = device; h->W = max_windows; h->Ncap = max_frames;
    h->Mcap = (max_landmarks + 3) & ~3;                      // the Schur kernel's bulk copies move 16-byte granules (4 masks)
    h->Kcap = max_obs;
    if (cudaSetDevice(device) != cudaSuccess) { delete h; return PVIO_B200_ENODEV; }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    h->sm_count = prop.multiProcessorCount;
    *out = reinterpret_cast<pvio_b200_handle>(h);
    CK(h, cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CK(h, cudaEventCreate(&h->ev0)); CK(h, cudaEventCreate(&h->ev1));
    const size_t W = h->W, N = h->Ncap, M = h->Mcap, K = h->Kcap, npc = N * (N + 1) / 2;
    TRY(for_each_input(h, [&](auto m, size_t per, InputGroup) { return alloc(h, h->*m, W * per, true); }));
    TRY(alloc(h, h->fobs, W * K, false)); TRY(alloc(h, h->seg, W * kSegTab, false));
    TRY(alloc(h, h->ctrl, W, true));
    TRY(alloc(h, h->rho_cand, W * M, false)); TRY(alloc(h, h->frames_cand, W * N * kFrameStride, false));
    // the linearisation lives in two buffer sets (LinBufs, ba_types.h): everything below up to the reduced system is doubled
    TRY(alloc(h, h->lm_scale, W * M, false)); TRY(alloc(h, h->lm_aux, 2 * W * M, false));
    TRY(alloc(h, h->hs, 2 * W * N * M * 6 * sizeof(float), false)); TRY(alloc(h, h->jr, 2 * W * N * M * 2 * sizeof(float), false));
    TRY(alloc(h, h->lm_w, 2 * W * M * 2 * sizeof(float), false)); TRY(alloc(h, h->lm_msk, 2 * W * M, false));
    {   // landing area of downloaded states: host only
        CK(h, cudaMallocHost(&h->frames_out.h, sizeof(double) * W * N * kFrameStride));
        CK(h, cudaMallocHost(&h->rho_out.h, sizeof(double) * W * M));
    }
    TRY(alloc(h, h->dx_lm, W * M, true)); TRY(alloc(h, h->lm_v, W * M, false)); TRY(alloc(h, h->dx_pose, W * N * 15, true));
    TRY(alloc(h, h->pose_scale, W * N * 15, false)); TRY(alloc(h, h->v_pose, W * N * 15, false));
    TRY(alloc(h, h->valid, W * M, true)); TRY(alloc(h, h->quality, W * M, true));
    {   // the reduced-system outputs of the linearise kernel live in ONE allocation so that the
        // multi-CTA-per-window mode (atomic accumulation) needs a single memset per launch
        const size_t n_sys = W * (npc * 36 + N * 36 + N * 6 + N * 6 + 1);
        TRY(alloc(h, h->Hred, 2 * n_sys, false));
        h->Hdd = h->Hred.d + W * npc * 36;
        h->gdir = h->Hdd + W * N * 36;
        h->gred = h->gdir + W * N * 6;
        h->cost_vis = h->gred + W * N * 6;
        h->sys_set = n_sys;                                   // set 1 of each array lies n_sys elements behind set 0
    }
    TRY(alloc(h, h->acc, W * kAcc, true)); TRY(alloc(h, h->aux_cost, W, false));
    TRY(alloc(h, h->Hfull, (15 * N) * (15 * N), true)); TRY(alloc(h, h->gfull, 15 * N, true));
    h->perm.resize(W); h->perm_identity.assign(W, 1); h->slot_M.assign(W, 0); h->slot_N.assign(W, 0); h->slot_K.assign(W, 0);
    {   // opt in to large dynamic shared memory ONCE per kernel with the device limit: the attribute is process-wide, so a
        // per-handle value would be overwritten by the next handle with other capacities
        const int lim = (int)prop.sharedMemPerBlockOptin - 2048;
        CK(h, cudaFuncSetAttribute(lin_obs_kernel<true, float, kLinWarps, kLinBlocks>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CK(h, cudaFuncSetAttribute(lin_obs_kernel<true, double, kLinWarps, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CK(h, cudaFuncSetAttribute(lin_obs_kernel<false, double, kLinWarps, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CK(h, cudaFuncSetAttribute(schur_kernel<float, kSchurThreads, kSchurBlocks>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CK(h, cudaFuncSetAttribute(schur_kernel<double, kSchurThreads, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CK(h, cudaFuncSetAttribute(update_obs_kernel<true, float, kUpdWarps, kUpdBlocks, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CK(h, cudaFuncSetAttribute(update_obs_kernel<true, float, kUpdWarps, kUpdBlocks, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CK(h, cudaFuncSetAttribute(update_obs_kernel<true, float, 8, 2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CK(h, cudaFuncSetAttribute(update_obs_kernel<true, double, kUpdWarps, 4, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CK(h, cudaFuncSetAttribute(update_obs_kernel<true, float, kUpdWarps, kUpdBlocks, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CK(h, cudaFuncSetAttribute(update_obs_kernel<true, double, kUpdWarps, 4, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CK(h, cudaFuncSetAttribute(update_obs_kernel<true, double, 8, 2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CK(h, cudaFuncSetAttribute(update_obs_kernel<true, double, kUpdWarps, 4, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CK(h, cudaFuncSetAttribute(solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        CK(h, cudaFuncSetAttribute(solve_kernel_visual, cudaFuncAttributeMaxDynamicSharedMemorySize, 48 * 1024));
    }
    init_ctrl_kernel<<<(int)W, 32, 0, h->stream>>>(h->ctrl.d, 1e-8, 1e4, 10, 0.0, 0);
    ++h->launches;
    CK(h, cudaStreamSynchronize(h->stream));
    return 0;
}

void pvio_b200_destroy(pvio_b200_handle hh) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->pnp_dev) cudaFree(h->pnp_dev);
    if (h->pnp_host) cudaFreeHost(h->pnp_host);
    klt_free(h);
    marg_free(h);
    resident_free(h);
    detect_free(h);
    fm_free(h);
    drop_graphs(h);
    for (auto &e : h->kev) cudaEventDestroy(e);
    cudaEventDestroy(h->ev0); cudaEventDestroy(h->ev1);
    for (auto &e : h->ev_up) cudaEventDestroy(e);
    for (auto &e : h->ev_done) cudaEventDestroy(e);
    for (auto &e : h->ev_down) cudaEventDestroy(e);
    if (h->stream_up) cudaStreamDestroy(h->stream_up);
    if (h->stream_down) cudaStreamDestroy(h->stream_down);
    for (auto &st : h->stream_c) cudaStreamDestroy(st);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->stream_aux) { cudaStreamDestroy(h->stream_aux); cudaEventDestroy(h->ev_aux_fork); cudaEventDestroy(h->ev_aux_join); }
    cudaStreamDestroy(h->stream);
    delete h;
}

const char *pvio_b200_last_error(pvio_b200_handle hh) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    return h ? h->err.c_str() : "null handle";
}

int64_t pvio_b200_kernel_launches(pvio_b200_handle hh) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    return h ? h->launches : 0;
}

int pvio_b200_sync(pvio_b200_handle hh) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h) return PVIO_B200_EINVAL;
    CK(h, cudaStreamSynchronize(h->stream));
    return 0;
}

int pvio_b200_timer_start(pvio_b200_handle hh) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h) return PVIO_B200_EINVAL;
    CK(h, cudaEventRecord(h->ev0, h->stream));
    return 0;
}

int pvio_b200_timer_stop(pvio_b200_handle hh, float *ms) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || !ms) return PVIO_B200_EINVAL;
    CK(h, cudaEventRecord(h->ev1, h->stream));
    CK(h, cudaEventSynchronize(h->ev1));
    CK(h, cudaEventElapsedTime(ms, h->ev0, h->ev1));
    return 0;
}

// Device time of the linearise + Schur stage from the CUDA events recorded around its launches:
// which = 0 the most recent stage; 1 the MEAN stage over the launches since the last reset (at most the latest 256);
// 2 / 3 the mean of the linearise / the Schur kernel alone; -1 resets the accumulation.
int pvio_b200_last_kernel_ms(pvio_b200_handle hh, int which, float *ms) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h) return PVIO_B200_EINVAL;
    if (which < 0) { h->kev_count = 0; if (ms) *ms = 0.f; return 0; }
    if (!ms) return PVIO_B200_EINVAL;
    if (h->kev_count == 0) { *ms = 0.f; return 0; }     // graph-replayed launches are not individually timed
    CK(h, cudaStreamSynchronize(h->stream));
    const int n = which == 0 ? 1 : std::min(h->kev_count, 256);
    double tot = 0.0;
    for (int i = 0; i < n; ++i) {
        const int slot = ((h->kev_count - 1 - i) % 256) * 3;
        float t = 0.f;
        const int e0 = which == 3 ? 1 : 0, e1 = which == 2 ? 1 : 2;
        CK(h, cudaEventElapsedTime(&t, h->kev[slot + e0], h->kev[slot + e1]));
        tot += t;
    }
    *ms = (float)(tot / n);
    return 0;
}

int pvio_b200_batch_set_window(pvio_b200_handle hh, int slot, const pvio_b200_window *w, const pvio_b200_state *s) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || !w || !s) return PVIO_B200_EINVAL;
    return pack_window(h, slot, w, s);
}

int pvio_b200_batch_replicate(pvio_b200_handle hh, int n) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h) return PVIO_B200_EINVAL;
    if (n < 1 || n > h->W) return fail(h, PVIO_B200_EINVAL, "bad window count");
    for_each_input(h, [&](auto m, size_t per, InputGroup) {
        auto &b = h->*m;
        for (int i = 1; i < n; ++i) memcpy(b.h + (size_t)i * per, b.h, sizeof(*b.h) * per);
        return 0;
    });
    for (int i = 1; i < n; ++i) {
        h->perm[i] = h->perm[0]; h->perm_identity[i] = h->perm_identity[0]; h->slot_M[i] = h->slot_M[0]; h->slot_N[i] = h->slot_N[0]; h->slot_K[i] = h->slot_K[0];
    }
    return 0;
}

int pvio_b200_batch_upload(pvio_b200_handle hh, int n) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h) return PVIO_B200_EINVAL;
    return upload(h, n);
}

int pvio_b200_batch_gn_step(pvio_b200_handle hh, int n, double mu, int apply) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h) return PVIO_B200_EINVAL;
    if (n < 1 || n > h->n_uploaded) return fail(h, PVIO_B200_EINVAL, "windows not uploaded");
    StepCfg c;
    c.mu = mu; c.apply = apply; c.compute_scale = 1;
    return run_gn_step(h, n, c, batch_shape(h, 0, n, false));
}

int pvio_b200_batch_download(pvio_b200_handle hh, int n, double *dx, int64_t dx_stride, double *costs) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h) return PVIO_B200_EINVAL;
    return download_dx(h, n, dx, dx_stride, costs);
}

// End-to-end Gauss-Newton step with HOST buffers (run_pipelined).
int pvio_b200_batch_gn_step_host(pvio_b200_handle hh, int n, double mu, double *dx, int64_t dx_stride, double *costs) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h) return PVIO_B200_EINVAL;
    return run_pipelined(h, n,
        [&](int w0, int m, cudaStream_t st) {
            StepCfg c;
            c.mu = mu; c.apply = 0; c.compute_scale = 1; c.w0 = w0; c.stream = st;
            return run_gn_step(h, m, c, batch_shape(h, w0, m, false));
        },
        [&](int w0, int m, cudaStream_t st) { return download_dx_async(h, w0, m, st); },
        [&](int w0, int m) { return scatter_dx(h, w0, m, dx, dx_stride, costs); });
}

// Full trust-region solve (device-side loop, per-window termination) of the first n uploaded windows; the states on
// the device are overwritten with the solutions.
int pvio_b200_batch_solve(pvio_b200_handle hh, int n, const pvio_b200_options *opt) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h) return PVIO_B200_EINVAL;
    if (n < 1 || n > h->n_uploaded) return fail(h, PVIO_B200_EINVAL, "windows not uploaded");
    return run_solve_loop(h, 0, n, h->stream, solve_opts(opt));
}

int pvio_b200_batch_download_state(pvio_b200_handle hh, int n, double *frames, int64_t frames_stride, double *inv_depth,
                                   int64_t inv_depth_stride, pvio_b200_summary *summaries) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h) return PVIO_B200_EINVAL;
    if (n < 1 || n > h->W) return fail(h, PVIO_B200_EINVAL, "bad window count");
    TRY(download_state_async(h, 0, n, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    scatter_states(h, 0, n, frames, frames_stride, inv_depth, inv_depth_stride, summaries);
    return 0;
}

// upload + solve + download with HOST buffers (run_pipelined): one host -> device copy buys up to max_iterations
// Gauss-Newton iterations per window.
int pvio_b200_batch_solve_host(pvio_b200_handle hh, int n, const pvio_b200_options *opt, double *frames, int64_t frames_stride,
                               double *inv_depth, int64_t inv_depth_stride, pvio_b200_summary *summaries) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h) return PVIO_B200_EINVAL;
    const SolveOpts o = solve_opts(opt);
    return run_pipelined(h, n,
        [&](int w0, int m, cudaStream_t st) { return run_solve_loop(h, w0, m, st, o); },
        [&](int w0, int m, cudaStream_t st) { return download_state_async(h, w0, m, st); },
        [&](int w0, int m) {
            scatter_states(h, w0, m, frames, frames_stride, inv_depth, inv_depth_stride, summaries);
            return 0;
        });
}

int pvio_b200_ba_gn_step(pvio_b200_handle hh, const pvio_b200_window *w, const pvio_b200_state *s, double mu,
                         double *dx, double *cost, double *new_cost, double *Hred, double *gred) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || !w || !s) return PVIO_B200_EINVAL;
    TRY(pack_window(h, 0, w, s));
    TRY(upload(h, 1));
    StepCfg c;
    c.mu = mu; c.apply = 0; c.compute_scale = 1; c.dump = (Hred || gred) ? 1 : 0;
    if (c.dump) {
        CK(h, cudaMemsetAsync(h->Hfull.d, 0, sizeof(double) * h->Hfull.n, h->stream));
        CK(h, cudaMemsetAsync(h->gfull.d, 0, sizeof(double) * h->gfull.n, h->stream));
    }
    TRY(run_gn_step(h, 1, c, batch_shape(h, 0, 1, false)));
    double costs[2];
    const int N = w->n_frames, M = w->n_landmarks;
    TRY(download_dx(h, 1, dx, (int64_t)N * 15 + M, costs));
    if (cost) *cost = costs[0];
    if (new_cost) *new_cost = costs[1];
    if (c.dump) {
        const size_t Df = 15 * (size_t)h->Ncap, Dn = 15 * (size_t)N;
        CK(h, cudaMemcpyAsync(h->Hfull.h, h->Hfull.d, sizeof(double) * Df * Df, cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaMemcpyAsync(h->gfull.h, h->gfull.d, sizeof(double) * Df, cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
        if (Hred) for (size_t i = 0; i < Dn; ++i) memcpy(Hred + i * Dn, h->Hfull.h + i * Df, sizeof(double) * Dn);
        if (gred) memcpy(gred, h->gfull.h, sizeof(double) * Dn);
    }
    return 0;
}

// BundleAdjustorSolver::solve (bundle_adjustor.cpp:63-299) behind the shim's gather: pack, one host -> device copy,
// the device-side trust-region loop (ONE graph launch, ba_tr.cuh), the landmark post-pass, one device -> host copy.
int pvio_b200_ba_solve(pvio_b200_handle hh, const pvio_b200_window *w, pvio_b200_state *s,
                       const pvio_b200_options *opt, pvio_b200_summary *summary, uint8_t *valid, double *quality) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || !w || !s) return PVIO_B200_EINVAL;
    TRY(pack_window(h, 0, w, s));
    TRY(upload(h, 1));
    CK(h, cudaEventRecord(h->ev0, h->stream));
    TRY(run_solve_loop(h, 0, 1, h->stream, solve_opts(opt)));
    CK(h, cudaEventRecord(h->ev1, h->stream));
    const int M = w->n_landmarks;
    const bool post = (!opt || opt->run_postpass) && (valid || quality);
    if (post) {
        TRY(run_postpass(h, 1, true, nullptr));
        CK(h, cudaMemcpyAsync(h->valid.h, h->valid.d, (size_t)std::max(M, 1), cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaMemcpyAsync(h->quality.h, h->quality.d, sizeof(double) * std::max(M, 1), cudaMemcpyDeviceToHost, h->stream));
    }
    TRY(download_state_async(h, 0, 1, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    scatter_states(h, 0, 1, s->frames, 0, s->inv_depth, 0, summary);
    if (post) {
        const std::vector<int32_t> &perm = h->perm[0];
        for (int lp = 0; lp < M; ++lp) {
            if (valid) valid[perm[lp]] = h->valid.h[lp];
            if (quality) quality[perm[lp]] = h->quality.h[lp];
        }
    }
    if (summary) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, h->ev0, h->ev1);
        summary->solve_seconds = ms * 1e-3;
    }
    return 0;
}

int pvio_b200_reprojection_error(pvio_b200_handle hh, const pvio_b200_window *w, const pvio_b200_state *s, double *error) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || !w || !s || !error) return PVIO_B200_EINVAL;
    TRY(pack_window(h, 0, w, s));
    TRY(upload(h, 1));
    CK(h, cudaMemsetAsync(h->acc.d, 0, sizeof(double) * 8, h->stream));
    TRY(run_postpass(h, 1, false, h->acc.d));
    CK(h, cudaMemcpyAsync(h->acc.h, h->acc.d, sizeof(double) * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    *error = h->acc.h[0] / std::max(h->acc.h[1], 1.0);
    return 0;
}

int pvio_b200_ba_marginalize(pvio_b200_handle hh, const pvio_b200_window *w, const pvio_b200_state *s, int index,
                             double *S_out, double *e_out, double *H_out, double *b_out) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || !w || !s) return PVIO_B200_EINVAL;
    return marginalize_impl(h, w, s, index, false, S_out, e_out, H_out, b_out);
}

int pvio_b200_pnp_solve(pvio_b200_handle hh, const pvio_b200_pnp_problem *problem, double *frame,
                        const pvio_b200_options *opt, pvio_b200_summary *summary) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || !problem || !frame) return PVIO_B200_EINVAL;
    return pnp_solve_impl(h, problem, frame, opt, summary);
}

int pvio_b200_klt_track(pvio_b200_handle hh, const uint8_t *prev, const uint8_t *next, int width, int height, int stride,
                        const float *prev_pts, float *next_pts, uint8_t *status, float *err, int n_points,
                        int max_level, int max_iter, double eps) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || !prev || !next || !prev_pts || !next_pts || !status) return PVIO_B200_EINVAL;
    return klt_track_impl(h, prev, next, width, height, stride, prev_pts, next_pts, status, err, n_points, max_level,
                          max_iter, eps);
}

int pvio_b200_klt_track_raw(pvio_b200_handle hh, const uint8_t *prev, const uint8_t *next, int width, int height, int stride,
                            const float *prev_pts, float *next_pts, uint8_t *status, float *err, int n_points,
                            int max_level, int max_iter, double eps, double clahe_clip, int tiles_x, int tiles_y,
                            uint8_t *prev_eq, uint8_t *next_eq) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || !prev || !next || !prev_pts || !next_pts || !status) return PVIO_B200_EINVAL;
    if (!(clahe_clip > 0.0)) return fail(h, PVIO_B200_EINVAL, "klt_track_raw: clahe_clip must be positive");
    return klt_track_impl(h, prev, next, width, height, stride, prev_pts, next_pts, status, err, n_points, max_level,
                          max_iter, eps, clahe_clip, tiles_x, tiles_y, prev_eq, next_eq);
}

int pvio_b200_klt_track_cached(pvio_b200_handle hh, uint64_t prev_id, const uint8_t *prev, uint64_t next_id, const uint8_t *next,
                               int width, int height, int stride, const float *prev_pts, float *next_pts, uint8_t *status, float *err,
                               int n_points, int max_level, int max_iter, double eps, double clahe_clip, int tiles_x, int tiles_y,
                               int border) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || !prev_pts || !next_pts || !status) return PVIO_B200_EINVAL;
    if (clahe_clip < 0.0) return fail(h, PVIO_B200_EINVAL, "klt_track_cached: clahe_clip must be >= 0 (0: frames are already equalised)");
    return klt_track_impl(h, prev, next, width, height, stride, prev_pts, next_pts, status, err, n_points, max_level,
                          max_iter, eps, clahe_clip, tiles_x, tiles_y, nullptr, nullptr, prev_id, next_id, border);
}

int pvio_b200_find_fundamental_mask(pvio_b200_handle hh, int n, const float *p, const float *q, double threshold, double confidence,
                                    int max_iters, const int32_t *schedule, int n_schedule, uint8_t *mask, double *F, int32_t *info) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || n < 0 || (n > 0 && (!p || !q || !mask))) return PVIO_B200_EINVAL;
    return fm_ransac_impl(h, n, p, q, threshold, confidence, max_iters, schedule, n_schedule, mask, F, info);
}

int pvio_b200_fm_sample_schedule(int n, const float *p, const float *q, int iters, int32_t *schedule) {
    if (n < 8 || !p || !q || iters < 1 || !schedule) return PVIO_B200_EINVAL;
    return fm_cv_schedule(n, p, q, iters, schedule);
}

int pvio_b200_track_keypoints(pvio_b200_handle hh, uint64_t prev_id, const uint8_t *prev, uint64_t next_id, const uint8_t *next,
                              int width, int height, int stride, const float *prev_pts, float *next_pts, uint8_t *status,
                              int n_points, int max_level, int max_iter, double eps, double clahe_clip, int tiles_x, int tiles_y,
                              int border, double ransac_threshold, double ransac_confidence) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || !prev_pts || !next_pts || !status) return PVIO_B200_EINVAL;
    if (clahe_clip < 0.0) return fail(h, PVIO_B200_EINVAL, "track_keypoints: clahe_clip must be >= 0 (0: frames are already equalised)");
    if (n_points <= 0) return 0;
    TRY(klt_track_impl(h, prev, next, width, height, stride, prev_pts, next_pts, status, nullptr, n_points, max_level,
                       max_iter, eps, clahe_clip, tiles_x, tiles_y, nullptr, nullptr, prev_id, next_id, border));
    // opencv_image.cpp:112-129: the survivors, in order, through findFundamentalMat(FM_RANSAC, 1.0, 0.99) when there are >= 8
    std::vector<int> l;
    std::vector<float> p, q;
    l.reserve(n_points); p.reserve(2 * n_points); q.reserve(2 * n_points);
    for (int i = 0; i < n_points; ++i)
        if (status[i]) {
            l.push_back(i);
            p.push_back(prev_pts[2 * i]); p.push_back(prev_pts[2 * i + 1]);
            q.push_back(next_pts[2 * i]); q.push_back(next_pts[2 * i + 1]);
        }
    if (l.size() >= 8) {
        std::vector<uint8_t> mask(l.size());
        TRY(fm_ransac_impl(h, (int)l.size(), p.data(), q.data(), ransac_threshold, ransac_confidence, 1000, nullptr, 0, mask.data(),
                           nullptr, nullptr));
        for (size_t i = 0; i < l.size(); ++i)
            if (!mask[i]) status[l[i]] = 0;
    }
    return 0;
}

int pvio_b200_clahe(pvio_b200_handle hh, const uint8_t *src, int width, int height, int stride, double clip_limit,
                    int tiles_x, int tiles_y, uint8_t *dst) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || !src || !dst) return PVIO_B200_EINVAL;
    return clahe_impl(h, src, width, height, stride, clip_limit, tiles_x, tiles_y, dst);
}

int pvio_b200_selftest_lie(pvio_b200_handle hh, int n, const double *w, double *out) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || !w || !out || n < 1) return PVIO_B200_EINVAL;
    return selftest_lie_impl(h, n, w, out);
}

#ifdef PVIO_SOLVE_STAMPS
int pvio_b200_debug_solve_stamps(long long *out) {      // tuning builds only (tools/solve_stamps.py); not declared in include/pvio_b200.h
    return cudaMemcpyFromSymbol(out, pvio::g_solve_stamps, sizeof(long long) * 16) == cudaSuccess ? 0 : PVIO_B200_ECUDA;
}
#endif

}  // extern "C"
