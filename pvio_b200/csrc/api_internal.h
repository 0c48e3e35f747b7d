// Internal handle of libpvio_b200 (host side).  Not part of the ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <map>
#include <string>
#include <tuple>
#include <utility>
#include <vector>
#include "../../include/pvio_b200.h"
#include "ba_types.h"

namespace pvio {

// Owns a device array and its optional pinned host staging; both are freed with the buffer.
template <typename T>
struct DevBuf {
    T *d = nullptr;      // device
    T *h = nullptr;      // pinned host staging (optional)
    size_t n = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept { swap(o); }
    DevBuf &operator=(DevBuf &&o) noexcept { DevBuf(std::move(o)).swap(*this); return *this; }
    ~DevBuf() {
        if (d) cudaFree(d);
        if (h) cudaFreeHost(h);
    }
    void swap(DevBuf &o) noexcept { std::swap(d, o.d); std::swap(h, o.h); std::swap(n, o.n); }
};

struct KltState;         // klt.cu
struct MargScratch;      // ba_marg.cu
struct FmState;          // fmat.cu

struct Handle {
    int device = 0;
    int W = 1, Ncap = 0, Mcap = 0, Kcap = 0;
    int Pcap = 4, Tcap = 0, Ocap = 0;            // planes / plane tracks / plane observations per window
    cudaStream_t stream = nullptr;
    cudaStream_t stream_up = nullptr, stream_down = nullptr;   // copy streams of the pipelined host path
    std::vector<cudaStream_t> stream_c;                        // compute streams of the pipelined host path
    cudaEvent_t ev_fork = nullptr;
    cudaStream_t stream_aux = nullptr;                         // second branch of the captured single-window solve (api.cu: iteration_body)
    cudaEvent_t ev_aux_fork = nullptr, ev_aux_join = nullptr;
    std::vector<cudaEvent_t> ev_up, ev_done, ev_down;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    int64_t launches = 0;
    bool prior_resident = false;                  // slot 0's prior (S, e, x0) was written on the device by the marginaliser
    int prior_resident_n = 0;                     // its frame count
    struct ResidentWindow *resident = nullptr;    // resident.cu
    struct DetectState *detect = nullptr;         // detect.cu
    size_t sys_set = 0;                           // elements between the two buffer sets of the reduced-system arrays (LinBufs)
    int sm_count = 148;

    // vision (always allocated)
    DevBuf<WinHdr> hdr;
    DevBuf<WinConst> cst;
    DevBuf<ObsRec> obs;                          // landmark-major table as the shim gathers it (uploaded)
    DevBuf<FObs> fobs;                           // frame-major table, built on the device after every upload
    DevBuf<int32_t> seg;                         // [W][kSegTab]
    DevBuf<LmRec> lms;
    DevBuf<double> rho, frames;
    DevBuf<WinCtrl> ctrl;
    DevBuf<double> rho_cand, frames_cand, lm_scale, dx_lm, lm_v, dx_pose, pose_scale, v_pose;
    DevBuf<LmAux> lm_aux;
    DevBuf<unsigned char> hs;                    // [W][Ncap][Mcap][6] float (visual-only windows) or double (inertial):
    DevBuf<unsigned char> jr;                    //   unscaled h records / [W][Ncap][Mcap][2] (j.j, j.r), linearise -> Schur / update
    DevBuf<unsigned char> lm_w;                  // [W][Mcap][2] real: pivot w_l, w_l g_l
    DevBuf<int32_t> lm_msk;                      // [W][Mcap] frame mask of each landmark
    bool hs_double = false;
    DevBuf<double> frames_out, rho_out;          // pinned landing area of downloaded states (the upload staging stays intact)
    DevBuf<double> Hred, acc, aux_cost;
    double *Hdd = nullptr, *gdir = nullptr, *gred = nullptr, *cost_vis = nullptr;   // views into the Hred allocation
    DevBuf<double> Hfull, gfull;                 // debug dump (single window only)
    DevBuf<uint8_t> valid;                       // post-pass results
    DevBuf<double> quality;
    // inertial / prior / planes (allocated on first use)
    bool have_inertial = false;
    DevBuf<int32_t> imu_idx, prior_frames;
    DevBuf<double> imu_data, prior_S, prior_L, prior_e, prior_x0;
    bool have_planes = false;
    DevBuf<double> plane_param;
    DevBuf<int32_t> pt_plane, pt_begin, pt_frame;
    DevBuf<float> pt_z;
    DevBuf<double> pt_J;                          // [W][Tcap][6 Ncap + 2] scratch of the plane block of solve_kernel
    // host bookkeeping per slot
    std::vector<std::vector<int32_t>> perm;      // packed landmark -> caller landmark
    std::vector<int> slot_M, slot_N, slot_K;
    std::vector<uint8_t> perm_identity;
    int n_uploaded = 0;
    // ring of event triples around the linearise + Schur launches (roofline timing without host syncs)
    std::vector<cudaEvent_t> kev;
    int kev_count = 0;
    // CUDA graphs of the latency path (few windows): the whole trust-region solve / one GN iteration as ONE launch.
    // Key: (kind, n, max_iter, flags) -- no floating-point values; all scalars the kernels need live in WinCtrl.
    // Launch shapes use the handle's capacities, so a graph survives window-shape changes between keyframes.
    // Cleared whenever a device buffer is reallocated (pointers are baked into the nodes).
    typedef std::tuple<int, int, int, int> GraphKey;
    std::map<GraphKey, std::pair<cudaGraphExec_t, int>> graphs;
    bool capturing = false;
    KltState *klt = nullptr;
    MargScratch *marg = nullptr;
    FmState *fm = nullptr;
    double *pnp_dev = nullptr, *pnp_host = nullptr;   // pnp.cu: device buffer + pinned staging, grown on demand
    size_t pnp_words = 0;
};

int fail(Handle *h, int code, const char *what, cudaError_t e = cudaSuccess);

// pvio_b200_options with its defaults filled in (opt may be NULL)
struct SolveOpts {
    int max_iter = 10;
    double radius0 = 1e4;
    int alias_bias = 1;
    double max_time = 0.0;
};
SolveOpts solve_opts(const pvio_b200_options *opt);

#define CK(h, call)                                                        \
    do {                                                                   \
        cudaError_t e__ = (call);                                          \
        if (e__ != cudaSuccess) return fail((h), PVIO_B200_ECUDA, #call, e__); \
    } while (0)

#define TRY(x) do { int rc__ = (x); if (rc__ != 0) return rc__; } while (0)

// api.cu: pack window into slot 0, copy it to the device, build the frame-major table
int pack_and_upload(Handle *h, const pvio_b200_window *w, const pvio_b200_state *s);
// api.cu: linearise + Schur of window 0 with the fp64 pipeline, no loss (the marginaliser's reprojection part)
int run_marg_vision(Handle *h);
void drop_graphs(Handle *h);
// klt.cu
int klt_track_impl(Handle *h, const uint8_t *prev, const uint8_t *next, int width, int height, int stride,
                   const float *prev_pts, float *next_pts, uint8_t *status, float *err, int n_points,
                   int max_level, int max_iter, double eps, double clahe_clip = 0.0, int tiles_x = 0, int tiles_y = 0,
                   uint8_t *prev_eq = nullptr, uint8_t *next_eq = nullptr, uint64_t prev_id = 0, uint64_t next_id = 0, int border = 0);
int clahe_impl(Handle *h, const uint8_t *src, int width, int height, int stride, double clip, int tiles_x, int tiles_y, uint8_t *dst);
void klt_free(Handle *h);
// pnp.cu
int pnp_solve_impl(Handle *h, const pvio_b200_pnp_problem *pb, double *frame, const pvio_b200_options *opt,
                   pvio_b200_summary *summary);
// ba_marg.cu
void resident_free(Handle *h);     // resident.cu
// klt.cu / detect.cu
const uint8_t *klt_cached_level0(Handle *h, uint64_t frame_id, int width, int height, double clahe_clip);
int klt_clahe_device(Handle *h, const uint8_t *d_src, uint8_t *d_dst, uint8_t *d_lut, int width, int height, double clip, int tiles_x, int tiles_y);
void detect_free(Handle *h);
int marginalize_impl(Handle *h, const pvio_b200_window *w, const pvio_b200_state *s, int index, bool keep_on_device,
                     double *S_out, double *e_out, double *H_out, double *b_out);
void marg_free(Handle *h);
// fmat.cu
int fm_ransac_impl(Handle *h, int n, const float *p, const float *q, double threshold, double confidence, int max_iters,
                   const int32_t *schedule, int n_schedule, uint8_t *mask, double *F_out, int32_t *info);
void fm_free(Handle *h);
int fm_cv_schedule(int n, const float *p, const float *q, int iters, int32_t *schedule);
// selftest.cu
int selftest_lie_impl(Handle *h, int n, const double *w_in, double *out);

}  // namespace pvio
