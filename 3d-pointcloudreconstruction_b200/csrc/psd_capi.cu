// psd_capi.cu -- extern "C" surface of libpsd_b200.so (declared in include/psd_b200.h).
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/psd_b200.h"
#include "psd_common.cuh"
#include "psd_device.h"

// launchers implemented in chamfer.cu / emd.cu
cudaError_t psd_launch_chamfer_forward(const float *xyz1, const float *xyz2, int b, int n, int m, int layout,
                                       float *dist1, float *dist2, int *idx1, int *idx2, float *sums, float fs_thr,
                                       int *fs_count, int q_begin, int q_count, cudaStream_t stream, float *zero_buf = nullptr,
                                       long long zero_floats = 0, bool ragged = false, const int *len1 = nullptr,
                                       const int *len2 = nullptr);
cudaError_t psd_launch_chamfer_backward(const float *xyz1, const float *xyz2, float *gradxyz1, float *gradxyz2,
                                        const float *graddist1, const float *graddist2, const int *idx1, const int *idx2,
                                        int b, int n, int m, int layout, int overwrite, cudaStream_t stream,
                                        const float *upstream = nullptr, bool ragged = false, const int *len1 = nullptr,
                                        const int *len2 = nullptr);
cudaError_t psd_launch_chamfer_mean_loss(const float *sums, int b, int n, int m, float *out, cudaStream_t stream);
cudaError_t psd_read_chamfer_stats(unsigned long long *fallback, int reset);
int psd_set_nn_variant(int v);
cudaError_t psd_launch_icp(const void *a, const void *b, int in_f64, int batch, int n, const double *init_pose, int max_iter,
                           double tol, double *T, double *dist, int *iters, cudaStream_t stream);
cudaError_t psd_launch_nn_f64(const void *src, const void *dst, int in_f64, int batch, int n_src, int n_dst, double *distances,
                              int *indices, cudaStream_t stream);
cudaError_t psd_launch_icp_ragged(const void *a, const void *b, int in_f64, int batch, int n, int m, const int *len_a,
                                  const int *len_b, const double *init_pose, int max_iter, double tol, double *T, double *dist,
                                  int *iters, cudaStream_t stream);
int psd_icp_max_points();
int psd_set_emd_solo(int enable);
int psd_set_emd_grid(int enable);
int psd_set_tc_max_ctas(int n);
cudaError_t psd_launch_cont_proj(const float *pcl, int b, int n, int grid_h, int grid_w, float sigma_sq, float *out,
                                 cudaStream_t stream);
cudaError_t psd_launch_cont_proj_backward(const float *pcl, const float *gout, int b, int n, int grid_h, int grid_w,
                                          float sigma_sq, float *gpcl, cudaStream_t stream);
cudaError_t psd_launch_fps(const float *xyz, int b, int n, int npoint, int start, long long *centroids, cudaStream_t stream);
int psd_fps_max_points();
cudaError_t psd_launch_proj_min_dist(const float *pred, const float *gt, const float *table, int b, int h, int w, int mode,
                                     float *out_min, float *out_inv, cudaStream_t stream);
void psd_set_tc_debug(float *dbg, int ld);
void psd_set_tc_prof(long long *prof);
cudaError_t psd_launch_emd_forward(const float *xyz1, const float *xyz2, int b, int n, float *dist, int *assignment,
                                   float *price, int *assignment_inv, int *bid, float *bid_increments,
                                   float *max_increments, float eps, int iters, int force_cluster, int fresh,
                                   float *loss_sums, cudaStream_t stream, int *unsupported);
cudaError_t psd_launch_emd_mean_loss(const float *sums, int b, int n, float *out, cudaStream_t stream);
cudaError_t psd_launch_emd_backward(const float *xyz1, const float *xyz2, float *gradxyz, const float *graddist,
                                    const int *idx, int b, int n, int mode, const float *upstream, cudaStream_t stream);
cudaError_t psd_launch_emd_dual_bound(const float *xyz1, const float *xyz2, int b, int n, const int *assignment, const float *price,
                                      double *bounds, int *status, cudaStream_t stream);
int psd_emd_bound_max_points();
cudaError_t psd_launch_sinkhorn(const float *x, const float *y, int b, int n, int m, bool ragged, const int *x_len,
                                const int *y_len, const float *x_w, const float *y_w, float blur, float scaling, float *loss,
                                float *grad_x, float *grad_y, float *potentials, int *rounds, int force_cluster,
                                cudaStream_t stream);

static thread_local char g_err[512] = "";

namespace psd {
static std::mutex g_state_mutex;
static DeviceState g_devices[kMaxDevices];
std::mutex &state_mutex() { return g_state_mutex; }
DeviceState *device_state(cudaError_t *err) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess && (dev < 0 || dev >= kMaxDevices)) e = cudaErrorInvalidDevice;
    if (e != cudaSuccess) { if (err) *err = e; return nullptr; }
    DeviceState *ds = &g_devices[dev];
    std::lock_guard<std::mutex> lock(g_state_mutex);
    if (!ds->init) {
        e = cudaDeviceGetAttribute(&ds->num_sms, cudaDevAttrMultiProcessorCount, dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&ds->max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        if (e != cudaSuccess) { if (err) *err = e; return nullptr; }
        ds->device = dev;
        ds->init = true;
    }
    return ds;
}
}  // namespace psd
using psd::DeviceState;
using psd::kStepSlots;

void psd_set_error(const char *what, cudaError_t err) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(err));
}
void psd_set_error_msg(const char *what) { snprintf(g_err, sizeof(g_err), "%s", what); }

static int finish(const char *what, cudaError_t e) {
    if (e != cudaSuccess) {
        psd_set_error(what, e);
        (void)cudaGetLastError();  // clear the sticky launch error like the reference's cudaGetLastError() does
        return 0;
    }
    return 1;
}

extern "C" {

int psd_version(void) { return 1000; }

const char *psd_last_error(void) { return g_err; }

int psd_chamfer_forward(const float *xyz1, const float *xyz2, int b, int n, int m, float *dist1, float *dist2,
                        int *idx1, int *idx2, void *stream) {
    return finish("psd_chamfer_forward",
                  psd_launch_chamfer_forward(xyz1, xyz2, b, n, m, 0, dist1, dist2, idx1, idx2, nullptr, 0.f, nullptr, 0,
                                             -1, (cudaStream_t)stream));
}

int psd_chamfer_forward_ex(const float *xyz1, const float *xyz2, int b, int n, int m, int layout, float *dist1,
                           float *dist2, int *idx1, int *idx2, float *sums, float fs_thr, int *fs_count, int q_begin,
                           int q_count, void *stream) {
    if (layout < 0 || layout > 3) {
        psd_set_error_msg("psd_chamfer_forward_ex: layout is a bit mask: 1 = xyz1 is [B,3,N], 2 = xyz2 is [B,3,M]");
        return -1;
    }
    return finish("psd_chamfer_forward_ex",
                  psd_launch_chamfer_forward(xyz1, xyz2, b, n, m, layout, dist1, dist2, idx1, idx2, sums, fs_thr,
                                             fs_count, q_begin, q_count, (cudaStream_t)stream));
}

int psd_chamfer_forward_zero(const float *xyz1, const float *xyz2, int b, int n, int m, int layout, float *dist1,
                             float *dist2, int *idx1, int *idx2, float *sums, float fs_thr, int *fs_count, float *zero_buf,
                             long long zero_floats, void *stream) {
    if (layout < 0 || layout > 3) {
        psd_set_error_msg("psd_chamfer_forward_zero: layout is a bit mask: 1 = xyz1 is [B,3,N], 2 = xyz2 is [B,3,M]");
        return -1;
    }
    return finish("psd_chamfer_forward_zero",
                  psd_launch_chamfer_forward(xyz1, xyz2, b, n, m, layout, dist1, dist2, idx1, idx2, sums, fs_thr,
                                             fs_count, 0, -1, (cudaStream_t)stream, zero_buf, zero_floats));
}

int psd_chamfer_backward(const float *xyz1, const float *xyz2, float *gradxyz1, float *gradxyz2,
                         const float *graddist1, const float *graddist2, const int *idx1, const int *idx2, int b, int n,
                         int m, void *stream) {
    return finish("psd_chamfer_backward",
                  psd_launch_chamfer_backward(xyz1, xyz2, gradxyz1, gradxyz2, graddist1, graddist2, idx1, idx2, b, n, m,
                                              0, 0, (cudaStream_t)stream));
}

int psd_chamfer_backward_ex(const float *xyz1, const float *xyz2, float *gradxyz1, float *gradxyz2,
                            const float *graddist1, const float *graddist2, const int *idx1, const int *idx2, int b, int n,
                            int m, int layout, int overwrite, void *stream) {
    if (layout < 0 || layout > 3) {
        psd_set_error_msg("psd_chamfer_backward_ex: layout is a bit mask: 1 = xyz1 is [B,3,N], 2 = xyz2 is [B,3,M]");
        return -1;
    }
    return finish("psd_chamfer_backward_ex",
                  psd_launch_chamfer_backward(xyz1, xyz2, gradxyz1, gradxyz2, graddist1, graddist2, idx1, idx2, b, n, m,
                                              layout, overwrite != 0, (cudaStream_t)stream));
}

int psd_chamfer_forward_ragged(const float *xyz1, const float *xyz2, int b, int n, int m, int layout, const int *len1,
                               const int *len2, float *dist1, float *dist2, int *idx1, int *idx2, float *sums, float fs_thr,
                               int *fs_count, float *zero_buf, long long zero_floats, void *stream) {
    if (layout < 0 || layout > 3) {
        psd_set_error_msg("psd_chamfer_forward_ragged: layout is a bit mask: 1 = xyz1 is [B,3,N], 2 = xyz2 is [B,3,M]");
        return -1;
    }
    return finish("psd_chamfer_forward_ragged",
                  psd_launch_chamfer_forward(xyz1, xyz2, b, n, m, layout, dist1, dist2, idx1, idx2, sums, fs_thr, fs_count, 0,
                                             -1, (cudaStream_t)stream, zero_buf, zero_floats, true, len1, len2));
}

int psd_chamfer_backward_ragged(const float *xyz1, const float *xyz2, float *gradxyz1, float *gradxyz2,
                                const float *graddist1, const float *graddist2, const int *idx1, const int *idx2,
                                const int *len1, const int *len2, int b, int n, int m, int layout, void *stream) {
    if (layout < 0 || layout > 3) {
        psd_set_error_msg("psd_chamfer_backward_ragged: layout is a bit mask: 1 = xyz1 is [B,3,N], 2 = xyz2 is [B,3,M]");
        return -1;
    }
    return finish("psd_chamfer_backward_ragged",
                  psd_launch_chamfer_backward(xyz1, xyz2, gradxyz1, gradxyz2, graddist1, graddist2, idx1, idx2, b, n, m,
                                              layout, 0, (cudaStream_t)stream, nullptr, true, len1, len2));
}

static const char *kEmdShapeMsg = "the cloud size must be a multiple of the cluster size";

int psd_emd_forward(const float *xyz1, const float *xyz2, int b, int n, int m, float *dist, int *assignment,
                    float *price, int *assignment_inv, int *bid, float *bid_increments, float *max_increments,
                    int *unass_idx, int *unass_cnt, int *unass_cnt_sum, int *cnt_tmp, int *max_idx, float eps,
                    int iters, void *stream) {
    (void)unass_idx; (void)unass_cnt; (void)unass_cnt_sum; (void)cnt_tmp; (void)max_idx;
    // emd_cuda.cu:236-249 (the reference printf()s these and returns -1)
    if (n != m) { psd_set_error_msg("Input Error! The two point clouds should have the same size."); return -1; }
    if (b > 512) { psd_set_error_msg("Input Error! The batch size should be less than 512."); return -1; }
    if (n % 1024 != 0) { psd_set_error_msg("Input Error! The size of the point clouds should be a multiple of 1024."); return -1; }
    int unsupported = 0;
    cudaError_t e = psd_launch_emd_forward(xyz1, xyz2, b, n, dist, assignment, price, assignment_inv, bid, bid_increments,
                                           max_increments, eps, iters, 0, 0, nullptr, (cudaStream_t)stream, &unsupported);
    if (unsupported) { psd_set_error_msg(kEmdShapeMsg); return 0; }
    return finish("psd_emd_forward", e);
}

// test hook: force the cluster size (1,2,4,8; negative = the same size on the global-workspace form of the kernel) so that
// every decomposition can be parity-checked
int psd_emd_forward_cluster(const float *xyz1, const float *xyz2, int b, int n, float *dist, int *assignment,
                            float *price, int *assignment_inv, float eps, int iters, int cluster_size, void *stream) {
    if (b > 512 || n % 1024 != 0) return -1;
    int unsupported = 0;
    cudaError_t e = psd_launch_emd_forward(xyz1, xyz2, b, n, dist, assignment, price, assignment_inv, nullptr, nullptr,
                                           nullptr, eps, iters, cluster_size, 0, nullptr, (cudaStream_t)stream, &unsupported);
    if (unsupported) { psd_set_error_msg(kEmdShapeMsg); return 0; }
    return finish("psd_emd_forward_cluster", e);
}

int psd_emd_forward_fresh(const float *xyz1, const float *xyz2, int b, int n, float *dist, int *assignment, float eps,
                          int iters, void *stream) {
    if (b > 512) { psd_set_error_msg("Input Error! The batch size should be less than 512."); return -1; }
    if (n % 1024 != 0) { psd_set_error_msg("Input Error! The size of the point clouds should be a multiple of 1024."); return -1; }
    int unsupported = 0;
    cudaError_t e = psd_launch_emd_forward(xyz1, xyz2, b, n, dist, assignment, nullptr, nullptr, nullptr, nullptr, nullptr,
                                           eps, iters, 0, 1, nullptr, (cudaStream_t)stream, &unsupported);
    if (unsupported) { psd_set_error_msg(kEmdShapeMsg); return 0; }
    return finish("psd_emd_forward_fresh", e);
}

int psd_emd_backward(const float *xyz1, const float *xyz2, float *gradxyz, const float *graddist, const int *idx,
                     int b, int n, void *stream) {
    return finish("psd_emd_backward", psd_launch_emd_backward(xyz1, xyz2, gradxyz, graddist, idx, b, n, 0, nullptr, (cudaStream_t)stream));
}

int psd_emd_backward_ex(const float *xyz1, const float *xyz2, float *gradxyz, const float *graddist, const int *idx,
                        int b, int n, int overwrite, void *stream) {
    return finish("psd_emd_backward_ex",
                  psd_launch_emd_backward(xyz1, xyz2, gradxyz, graddist, idx, b, n, overwrite ? 1 : 0, nullptr, (cudaStream_t)stream));
}

// Certified EMD: epsilon-scaling phases of the unchanged auction kernel, then the dual-bound certificate.  Every phase starts
// from assignment = -1 and the previous phase's prices (the kernel reads and writes back the caller's price buffer when
// fresh = 0; NULL assignment_inv / max_increments start at -1 / 0 as in the reference's initial state).  Phase i runs
// eps = max(eps_start / scale^i, eps_end) (in double, rounded to float), the last one exactly eps_end.  No host synchronisation.
static const int kEmdMaxPhases = 64;

static int emd_certified_common(const char *what, const float *xyz1, const float *xyz2, int b, int n, float eps_start,
                                float eps_end, float scale, int max_iters_per_phase, float *dist, int *assignment, float *price,
                                double *bounds, int *status, int force_cluster, void *stream_) {
    char msg[256];
    if (b < 0 || b > 512) { snprintf(msg, sizeof(msg), "%s: the batch size must be in [0, 512]", what); psd_set_error_msg(msg); return -1; }
    if (n <= 0 || n % 1024 != 0) { snprintf(msg, sizeof(msg), "%s: the size of the point clouds must be a positive multiple of 1024", what); psd_set_error_msg(msg); return -1; }
    if (!(eps_end >= 1e-5f)) { snprintf(msg, sizeof(msg), "%s: eps_end must be >= 1e-5 (the auction's fp32 prices and +-1e-6 winner window make a smaller eps meaningless)", what); psd_set_error_msg(msg); return -1; }
    if (!(eps_end <= eps_start)) { snprintf(msg, sizeof(msg), "%s: eps_end must not exceed eps_start", what); psd_set_error_msg(msg); return -1; }
    if (!(scale > 1.0f)) { snprintf(msg, sizeof(msg), "%s: scale must be > 1", what); psd_set_error_msg(msg); return -1; }
    if (max_iters_per_phase < 1) { snprintf(msg, sizeof(msg), "%s: max_iters_per_phase must be >= 1", what); psd_set_error_msg(msg); return -1; }
    int phases = 1;
    for (double e = eps_start; e > (double)eps_end && phases <= kEmdMaxPhases; e /= (double)scale) ++phases;
    if (phases > kEmdMaxPhases) { snprintf(msg, sizeof(msg), "%s: more than %d phases (scale too close to 1)", what, kEmdMaxPhases); psd_set_error_msg(msg); return -1; }
    if (b == 0) return 1;
    cudaStream_t stream = (cudaStream_t)stream_;
    const size_t cells = (size_t)b * n;
    cudaError_t e = cudaMemsetAsync(price, 0, sizeof(float) * cells, stream);
    double e_cur = eps_start;
    for (int ph = 0; ph < phases && e == cudaSuccess; ++ph, e_cur /= (double)scale) {
        const float eps = ph == phases - 1 ? eps_end : (float)e_cur;
        e = cudaMemsetAsync(assignment, 0xff, sizeof(int) * cells, stream);   // every point unassigned (-1)
        int unsupported = 0;
        if (e == cudaSuccess)
            e = psd_launch_emd_forward(xyz1, xyz2, b, n, dist, assignment, price, nullptr, nullptr, nullptr, nullptr, eps,
                                       max_iters_per_phase, force_cluster, 0, nullptr, stream, &unsupported);
        if (unsupported) { psd_set_error_msg(kEmdShapeMsg); return 0; }
    }
    if (e == cudaSuccess) e = psd_launch_emd_dual_bound(xyz1, xyz2, b, n, assignment, price, bounds, status, stream);
    return finish(what, e);
}

int psd_emd_certified(const float *xyz1, const float *xyz2, int b, int n, float eps_start, float eps_end, float scale,
                      int max_iters_per_phase, float *dist, int *assignment, float *price, double *bounds, int *status,
                      void *stream) {
    return emd_certified_common("psd_emd_certified", xyz1, xyz2, b, n, eps_start, eps_end, scale, max_iters_per_phase, dist,
                                assignment, price, bounds, status, 0, stream);
}

// test hook: the same with the cluster size of every phase forced as in psd_emd_forward_cluster
int psd_emd_certified_cluster(const float *xyz1, const float *xyz2, int b, int n, float eps_start, float eps_end, float scale,
                              int max_iters_per_phase, float *dist, int *assignment, float *price, double *bounds, int *status,
                              int cluster_size, void *stream) {
    return emd_certified_common("psd_emd_certified_cluster", xyz1, xyz2, b, n, eps_start, eps_end, scale, max_iters_per_phase,
                                dist, assignment, price, bounds, status, cluster_size, stream);
}

int psd_emd_dual_bound(const float *xyz1, const float *xyz2, int b, int n, const int *assignment, const float *price,
                       double *bounds, int *status, void *stream) {
    if (b < 0 || b > 65535 || n < 1 || n > psd_emd_bound_max_points()) {
        psd_set_error_msg("psd_emd_dual_bound: b in [0, 65535] and n in [1, 2^20] required");
        return -1;
    }
    return finish("psd_emd_dual_bound",
                  psd_launch_emd_dual_bound(xyz1, xyz2, b, n, assignment, price, bounds, status, (cudaStream_t)stream));
}

static int sinkhorn_common(const char *what, const float *x, const float *y, int b, int n, int m, bool ragged,
                           const int *x_len, const int *y_len, const float *x_w, const float *y_w, float blur, float scaling,
                           float *loss, float *grad_x, float *grad_y, float *potentials, int *rounds, int force_cluster,
                           void *stream) {
    char msg[256];
    const char *bad = nullptr;
    if (b < 0 || b > 65535) bad = "the batch size must be in [0, 65535]";
    else if (n < 1 || n > (1 << 20) || m < 1 || m > (1 << 20)) bad = "the cloud sizes n and m must be in [1, 2^20]";
    else if (!(blur > 0.f) || !isfinite(blur)) bad = "blur must be finite and > 0";
    else if (!(scaling > 0.f && scaling < 1.f)) bad = "scaling must be in (0, 1)";
    else if (loss == nullptr) bad = "loss must not be NULL";
    else if (force_cluster != 0 && force_cluster != 1 && force_cluster != 2 && force_cluster != 4 && force_cluster != 8)
        bad = "cluster_size must be 1, 2, 4 or 8";
    if (bad) { snprintf(msg, sizeof(msg), "%s: %s", what, bad); psd_set_error_msg(msg); return -1; }
    if (b == 0) return 1;
    return finish(what, psd_launch_sinkhorn(x, y, b, n, m, ragged, x_len, y_len, x_w, y_w, blur, scaling, loss, grad_x, grad_y,
                                            potentials, rounds, force_cluster, (cudaStream_t)stream));
}

int psd_sinkhorn_divergence(const float *x, const float *y, int b, int n, int m, float blur, float scaling, float *loss,
                            float *grad_x, float *grad_y, float *potentials, int *rounds, void *stream) {
    return sinkhorn_common("psd_sinkhorn_divergence", x, y, b, n, m, false, nullptr, nullptr, nullptr, nullptr, blur, scaling, loss,
                           grad_x, grad_y, potentials, rounds, 0, stream);
}

int psd_sinkhorn_divergence_cluster(const float *x, const float *y, int b, int n, int m, float blur, float scaling, float *loss,
                                    float *grad_x, float *grad_y, float *potentials, int *rounds, int cluster_size, void *stream) {
    if (cluster_size == 0) cluster_size = -1;   // 0 selects automatically inside; the hook forces a size
    return sinkhorn_common("psd_sinkhorn_divergence_cluster", x, y, b, n, m, false, nullptr, nullptr, nullptr, nullptr, blur,
                           scaling, loss, grad_x, grad_y, potentials, rounds, cluster_size, stream);
}

int psd_sinkhorn_divergence_weighted(const float *x, const float *y, int b, int n, int m, const int *x_len, const int *y_len,
                                     const float *x_w, const float *y_w, float blur, float scaling, float *loss, float *grad_x,
                                     float *grad_y, float *potentials, int *rounds, void *stream) {
    return sinkhorn_common("psd_sinkhorn_divergence_weighted", x, y, b, n, m, true, x_len, y_len, x_w, y_w, blur, scaling, loss,
                           grad_x, grad_y, potentials, rounds, 0, stream);
}

int psd_sinkhorn_divergence_weighted_cluster(const float *x, const float *y, int b, int n, int m, const int *x_len,
                                             const int *y_len, const float *x_w, const float *y_w, float blur, float scaling,
                                             float *loss, float *grad_x, float *grad_y, float *potentials, int *rounds,
                                             int cluster_size, void *stream) {
    if (cluster_size == 0) cluster_size = -1;
    return sinkhorn_common("psd_sinkhorn_divergence_weighted_cluster", x, y, b, n, m, true, x_len, y_len, x_w, y_w, blur, scaling,
                           loss, grad_x, grad_y, potentials, rounds, cluster_size, stream);
}

int psd_emd_mean_loss_forward(const float *xyz1, const float *xyz2, int b, int n, float *dist, int *assignment, float eps,
                              int iters, float *sums_zeroed, float *loss, void *stream) {
    if (b > 512) { psd_set_error_msg("Input Error! The batch size should be less than 512."); return -1; }
    if (n % 1024 != 0) { psd_set_error_msg("Input Error! The size of the point clouds should be a multiple of 1024."); return -1; }
    int unsupported = 0;
    cudaError_t e = psd_launch_emd_forward(xyz1, xyz2, b, n, dist, assignment, nullptr, nullptr, nullptr, nullptr, nullptr,
                                           eps, iters, 0, 1, sums_zeroed, (cudaStream_t)stream, &unsupported);
    if (unsupported) { psd_set_error_msg(kEmdShapeMsg); return 0; }
    if (e == cudaSuccess) e = psd_launch_emd_mean_loss(sums_zeroed, b, n, loss, (cudaStream_t)stream);
    return finish("psd_emd_mean_loss_forward", e);
}

int psd_emd_mean_loss_backward(const float *xyz1, const float *xyz2, float *gradxyz1, const float *dist, const int *assignment,
                               const float *upstream, int b, int n, void *stream) {
    return finish("psd_emd_mean_loss_backward",
                  psd_launch_emd_backward(xyz1, xyz2, gradxyz1, dist, assignment, b, n, 2, upstream, (cudaStream_t)stream));
}

int psd_chamfer_mean_loss_forward(const float *xyz1, const float *xyz2, int b, int n, int m, int layout, float *dist1,
                                  float *dist2, int *idx1, int *idx2, float *sums_zeroed, float *loss, void *stream) {
    if (layout < 0 || layout > 3) {
        psd_set_error_msg("psd_chamfer_mean_loss_forward: layout is a bit mask: 1 = xyz1 is [B,3,N], 2 = xyz2 is [B,3,M]");
        return -1;
    }
    cudaError_t e = psd_launch_chamfer_forward(xyz1, xyz2, b, n, m, layout, dist1, dist2, idx1, idx2, sums_zeroed, 0.f, nullptr,
                                               0, -1, (cudaStream_t)stream);
    if (e == cudaSuccess) e = psd_launch_chamfer_mean_loss(sums_zeroed, b, n, m, loss, (cudaStream_t)stream);
    return finish("psd_chamfer_mean_loss_forward", e);
}

int psd_chamfer_mean_loss_forward_zero(const float *xyz1, const float *xyz2, int b, int n, int m, int layout, float *dist1,
                                       float *dist2, int *idx1, int *idx2, float *sums_zeroed, float *loss, float *zero_buf,
                                       long long zero_floats, void *stream) {
    if (layout < 0 || layout > 3) {
        psd_set_error_msg("psd_chamfer_mean_loss_forward_zero: layout is a bit mask: 1 = xyz1 is [B,3,N], 2 = xyz2 is [B,3,M]");
        return -1;
    }
    cudaError_t e = psd_launch_chamfer_forward(xyz1, xyz2, b, n, m, layout, dist1, dist2, idx1, idx2, sums_zeroed, 0.f, nullptr,
                                               0, -1, (cudaStream_t)stream, zero_buf, zero_floats);
    if (e == cudaSuccess) e = psd_launch_chamfer_mean_loss(sums_zeroed, b, n, m, loss, (cudaStream_t)stream);
    return finish("psd_chamfer_mean_loss_forward_zero", e);
}

int psd_chamfer_mean_loss_backward(const float *xyz1, const float *xyz2, float *gradxyz1, float *gradxyz2,
                                   const float *upstream, const int *idx1, const int *idx2, int b, int n, int m, void *stream) {
    return finish("psd_chamfer_mean_loss_backward",
                  psd_launch_chamfer_backward(xyz1, xyz2, gradxyz1, gradxyz2, nullptr, nullptr, idx1, idx2, b, n, m, 0, 0,
                                              (cudaStream_t)stream, upstream));
}

int psd_chamfer_mean_loss_backward_ex(const float *xyz1, const float *xyz2, float *gradxyz1, float *gradxyz2,
                                      const float *upstream, const int *idx1, const int *idx2, int b, int n, int m, int layout,
                                      int overwrite, void *stream) {
    if (layout < 0 || layout > 3) {
        psd_set_error_msg("psd_chamfer_mean_loss_backward_ex: layout is a bit mask: 1 = xyz1 is [B,3,N], 2 = xyz2 is [B,3,M]");
        return -1;
    }
    return finish("psd_chamfer_mean_loss_backward_ex",
                  psd_launch_chamfer_backward(xyz1, xyz2, gradxyz1, gradxyz2, nullptr, nullptr, idx1, idx2, b, n, m, layout,
                                              overwrite != 0, (cudaStream_t)stream, upstream));
}

int psd_proj_min_dist(const float *pred, const float *gt, const float *table, int b, int h, int w, int mode, float *min_dist,
                      float *min_dist_inv, void *stream) {
    if (mode != 0 && mode != 1) { psd_set_error_msg("psd_proj_min_dist: mode must be 0 (as written) or 1 (intended)"); return -1; }
    if ((size_t)h * w * 8 > 200 * 1024) { psd_set_error_msg("psd_proj_min_dist: grid too large for the shared-memory table (h*w <= 25600)"); return -1; }
    return finish("psd_proj_min_dist", psd_launch_proj_min_dist(pred, gt, table, b, h, w, mode, min_dist, min_dist_inv, (cudaStream_t)stream));
}

int psd_icp_batch(const void *a, const void *b, int in_f64, int batch, int n, const double *init_pose, int max_iterations,
                  double tolerance, double *T_out, double *distances, int *iterations, void *stream) {
    if (batch < 0 || n < 1 || max_iterations < 0) { psd_set_error_msg("psd_icp_batch: batch >= 0, n >= 1, max_iterations >= 0 required"); return -1; }
    if (n > psd_icp_max_points()) { psd_set_error_msg("psd_icp_batch: n exceeds the shared-memory resident limit (4096 points)"); return -1; }
    return finish("psd_icp_batch", psd_launch_icp(a, b, in_f64, batch, n, init_pose, max_iterations, tolerance, T_out, distances,
                                                  iterations, (cudaStream_t)stream));
}

int psd_icp_batch_ragged(const void *a, const void *b, int in_f64, int batch, int n, int m, const int *len_a, const int *len_b,
                         const double *init_pose, int max_iterations, double tolerance, double *T_out, double *distances,
                         int *iterations, void *stream) {
    if (batch < 0 || n < 1 || m < 1 || max_iterations < 1) {
        psd_set_error_msg("psd_icp_batch_ragged: batch >= 0, n >= 1, m >= 1, max_iterations >= 1 required");
        return -1;
    }
    if (n > psd_icp_max_points() || n + m > 2 * psd_icp_max_points()) {
        psd_set_error_msg("psd_icp_batch_ragged: n <= 4096 and n + m <= 8192 required (shared-memory resident clouds)");
        return -1;
    }
    return finish("psd_icp_batch_ragged", psd_launch_icp_ragged(a, b, in_f64, batch, n, m, len_a, len_b, init_pose, max_iterations,
                                                                tolerance, T_out, distances, iterations, (cudaStream_t)stream));
}

int psd_farthest_point_sample(const float *xyz, int b, int n, int npoint, int start, long long *centroids, void *stream) {
    if (b < 0 || n < 1 || npoint < 0) { psd_set_error_msg("psd_farthest_point_sample: b >= 0, n >= 1, npoint >= 0 required"); return -1; }
    if (start < 0 || start >= n) { psd_set_error_msg("psd_farthest_point_sample: start index outside the cloud"); return -1; }
    if (n > psd_fps_max_points()) { psd_set_error_msg("psd_farthest_point_sample: n exceeds the shared-memory resident limit (16384 points)"); return -1; }
    return finish("psd_farthest_point_sample", psd_launch_fps(xyz, b, n, npoint, start, centroids, (cudaStream_t)stream));
}

int psd_cont_proj(const float *pcl, int b, int n, int grid_h, int grid_w, float sigma_sq, float *out, void *stream) {
    if (b < 0 || n < 0 || grid_h < 1 || grid_w < 1) { psd_set_error_msg("psd_cont_proj: b, n >= 0 and grid_h, grid_w >= 1 required"); return -1; }
    return finish("psd_cont_proj", psd_launch_cont_proj(pcl, b, n, grid_h, grid_w, sigma_sq, out, (cudaStream_t)stream));
}

int psd_cont_proj_backward(const float *pcl, const float *grad_out, int b, int n, int grid_h, int grid_w, float sigma_sq,
                           float *grad_pcl, void *stream) {
    if (b < 0 || n < 0 || grid_h < 1 || grid_w < 1) { psd_set_error_msg("psd_cont_proj_backward: b, n >= 0 and grid_h, grid_w >= 1 required"); return -1; }
    if (sizeof(float) * ((size_t)grid_h * (grid_w + 1) + 8 * (size_t)(grid_h + grid_w)) > 200 * 1024 || b > 65535) {
        psd_set_error_msg("psd_cont_proj_backward: the gradient image must fit in shared memory (about 220 x 220) and b <= 65535");
        return -1;
    }
    return finish("psd_cont_proj_backward",
                  psd_launch_cont_proj_backward(pcl, grad_out, b, n, grid_h, grid_w, sigma_sq, grad_pcl, (cudaStream_t)stream));
}

int psd_nn_f64(const void *src, const void *dst, int in_f64, int batch, int n_src, int n_dst, double *distances, int *indices,
               void *stream) {
    if (batch < 0 || n_src < 0 || n_dst < 1) { psd_set_error_msg("psd_nn_f64: batch >= 0, n_src >= 0, n_dst >= 1 required"); return -1; }
    if ((size_t)n_dst * 24 > 200 * 1024) { psd_set_error_msg("psd_nn_f64: destination cloud too large for shared memory (n_dst <= 8533)"); return -1; }
    return finish("psd_nn_f64", psd_launch_nn_f64(src, dst, in_f64, batch, n_src, n_dst, distances, indices, (cudaStream_t)stream));
}

int psd_chamfer_nn_variant(int variant) { return psd_set_nn_variant(variant); }

int psd_emd_solo_mode(int enable) { return psd_set_emd_solo(enable); }

int psd_emd_grid_mode(int enable) { return psd_set_emd_grid(enable); }

int psd_chamfer_tc_ctas(int max_ctas) { return psd_set_tc_max_ctas(max_ctas); }

int psd_debug_tc_prof(long long *prof_dev) { psd_set_tc_prof(prof_dev); return 1; }

int psd_debug_tc_filter(const float *xyz1, const float *xyz2, int b, int n, int m, float *dist1, float *dist2, int *idx1,
                        int *idx2, float *dump, int dump_ld, void *stream) {
    const int old = psd_set_nn_variant(3);
    psd_set_tc_debug(dump, dump_ld);
    cudaError_t e = psd_launch_chamfer_forward(xyz1, xyz2, b, n, m, 0, dist1, dist2, idx1, idx2, nullptr, 0.f, nullptr, 0,
                                               -1, (cudaStream_t)stream);
    psd_set_tc_debug(nullptr, 0);
    psd_set_nn_variant(old);
    return finish("psd_debug_tc_filter", e);
}

int psd_chamfer_stats(long long *out_host2, int reset) {
    unsigned long long fb = 0;
    cudaError_t e = psd_read_chamfer_stats(&fb, reset);
    if (e != cudaSuccess) return finish("psd_chamfer_stats", e);
    out_host2[0] = -1;  // filtered-path count is (total queries - fallbacks); not tracked on the device
    out_host2[1] = (long long)fb;
    return 1;
}

// ---- host-buffer entry points: stage through grow-only device workspaces owned by the library, one set per device
// (forward-only, and kStepSlots training-step workspaces).  One mutex serialises the bookkeeping of concurrent callers.
static std::mutex g_host_api_mutex;

int psd_chamfer_forward_host(const float *xyz1_host, const float *xyz2_host, int b, int n, int m, float *dist1_host,
                             float *dist2_host, int *idx1_host, int *idx2_host, void *stream_) {
    std::lock_guard<std::mutex> api_lock(g_host_api_mutex);
    cudaStream_t stream = (cudaStream_t)stream_;
    cudaError_t e = cudaSuccess;
    DeviceState *ds = psd::device_state(&e);
    if (ds == nullptr) return finish("psd_chamfer_forward_host(device)", e);
    const size_t s1 = (size_t)b * n, s2 = (size_t)b * m;
    const size_t need = sizeof(float) * (3 * s1 + 3 * s2 + 2 * s1 + 2 * s2);
    if (need > ds->fwd_ws_bytes) {
        if (ds->fwd_ws) { cudaDeviceSynchronize(); cudaFree(ds->fwd_ws); }
        ds->fwd_ws = nullptr; ds->fwd_ws_bytes = 0;
        e = cudaMalloc(&ds->fwd_ws, need);
        if (e != cudaSuccess) return finish("psd_chamfer_forward_host(cudaMalloc)", e);
        ds->fwd_ws_bytes = need;
    }
    float *d_x1 = ds->fwd_ws, *d_x2 = d_x1 + 3 * s1, *d_d1 = d_x2 + 3 * s2, *d_d2 = d_d1 + s1;
    int *d_i1 = reinterpret_cast<int *>(d_d2 + s2), *d_i2 = d_i1 + s1;
    if ((e = cudaMemcpyAsync(d_x1, xyz1_host, sizeof(float) * 3 * s1, cudaMemcpyHostToDevice, stream)) != cudaSuccess ||
        (e = cudaMemcpyAsync(d_x2, xyz2_host, sizeof(float) * 3 * s2, cudaMemcpyHostToDevice, stream)) != cudaSuccess)
        return finish("psd_chamfer_forward_host(H2D)", e);
    e = psd_launch_chamfer_forward(d_x1, d_x2, b, n, m, 0, d_d1, d_d2, d_i1, d_i2, nullptr, 0.f, nullptr, 0, -1, stream);
    if (e != cudaSuccess) return finish("psd_chamfer_forward_host(launch)", e);
    if ((e = cudaMemcpyAsync(dist1_host, d_d1, sizeof(float) * s1, cudaMemcpyDeviceToHost, stream)) != cudaSuccess ||
        (e = cudaMemcpyAsync(dist2_host, d_d2, sizeof(float) * s2, cudaMemcpyDeviceToHost, stream)) != cudaSuccess ||
        (e = cudaMemcpyAsync(idx1_host, d_i1, sizeof(int) * s1, cudaMemcpyDeviceToHost, stream)) != cudaSuccess ||
        (e = cudaMemcpyAsync(idx2_host, d_i2, sizeof(int) * s2, cudaMemcpyDeviceToHost, stream)) != cudaSuccess)
        return finish("psd_chamfer_forward_host(D2H)", e);
    return finish("psd_chamfer_forward_host(sync)", cudaStreamSynchronize(stream));
}


// fwd + fused mean loss + bwd of one training step: the end-to-end form of Loss.get_chamfer_loss (loss/loss.py:30-37)
// followed by loss.backward().  Gradients stay on the device unless host pointers are given.
struct StepArgs {
    const float *x1 = nullptr, *x2 = nullptr;   // xyz1: host, or device when x1_dev; xyz2: host
    bool x1_dev = false;                        // the prediction is already on the device (the generator's output, train.py:160)
    int layout1 = 0;                            // 1: the device prediction is [B,3,N] (the generator's native layout)
    int b = 0, n = 0, m = 0;
    float *loss_host = nullptr, *g1_host = nullptr, *g2_host = nullptr;
    float *g1_user = nullptr;                   // x1_dev: device buffer that receives d loss / d xyz1 (same layout as xyz1)
};

// One training step's stream work (H2D, forward, mean loss, backward, D2H) for a given workspace.
static cudaError_t enqueue_loss_step(const StepArgs &a, float *ws, cudaStream_t stream) {
    const int b = a.b, n = a.n, m = a.m;
    const size_t s1 = (size_t)b * n, s2 = (size_t)b * m;
    // layout: xyz1 | xyz2 | grad1 | grad2 | dist1 | dist2 | idx1 | idx2 | sums[2b] | loss
    float *d_x1 = ws, *d_x2 = d_x1 + 3 * s1, *d_g1 = d_x2 + 3 * s2, *d_g2 = d_g1 + 3 * s1;
    float *d_d1 = d_g2 + 3 * s2, *d_d2 = d_d1 + s1;
    int *d_i1 = reinterpret_cast<int *>(d_d2 + s2), *d_i2 = d_i1 + s1;
    float *d_sums = reinterpret_cast<float *>(d_i2 + s2), *d_loss = d_sums + 2 * (size_t)b;
    cudaError_t e;
    const float *x1 = d_x1;
    float *g1 = d_g1;
    int layout = 0;
    if (a.x1_dev) {
        // only the ground truth travels: the prediction (and its gradient) are the caller's device tensors
        x1 = a.x1; g1 = a.g1_user ? a.g1_user : d_g1; layout = a.layout1 ? 1 : 0;
        e = cudaMemcpyAsync(d_x2, a.x2, sizeof(float) * 3 * s2, cudaMemcpyHostToDevice, stream);
    } else if (a.x2 == a.x1 + 3 * s1) {
        // the two clouds are adjacent in the workspace: one copy when they are adjacent on the host too
        e = cudaMemcpyAsync(d_x1, a.x1, sizeof(float) * 3 * (s1 + s2), cudaMemcpyHostToDevice, stream);
    } else {
        e = cudaMemcpyAsync(d_x1, a.x1, sizeof(float) * 3 * s1, cudaMemcpyHostToDevice, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_x2, a.x2, sizeof(float) * 3 * s2, cudaMemcpyHostToDevice, stream);
    }
    if (e != cudaSuccess) return e;
    // per-cloud sums start from zero (one small memset); the gradients are zero-filled by the forward launch itself when they
    // sit in the workspace (grad1 | grad2 adjacent), so the backward is the single accumulate launch
    if ((e = cudaMemsetAsync(d_sums, 0, sizeof(float) * (2 * (size_t)b + 1), stream)) != cudaSuccess) return e;
    const bool own_g1 = (g1 == d_g1);
    if (!own_g1 && (e = cudaMemsetAsync(g1, 0, sizeof(float) * 3 * s1, stream)) != cudaSuccess) return e;
    e = psd_launch_chamfer_forward(x1, d_x2, b, n, m, layout, d_d1, d_d2, d_i1, d_i2, d_sums, 0.f, nullptr, 0, -1, stream,
                                   own_g1 ? d_g1 : d_g2, (long long)(own_g1 ? 3 * (s1 + s2) : 3 * s2));
    if (e == cudaSuccess) e = psd_launch_chamfer_mean_loss(d_sums, b, n, m, d_loss, stream);
    if (e == cudaSuccess) e = psd_launch_chamfer_backward(x1, d_x2, g1, d_g2, nullptr, nullptr, d_i1, d_i2, b, n, m, layout, 0, stream, nullptr);
    if (e != cudaSuccess) return e;
    e = cudaMemcpyAsync(a.loss_host, d_loss, sizeof(float), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess && a.g1_host) e = cudaMemcpyAsync(a.g1_host, g1, sizeof(float) * 3 * s1, cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess && a.g2_host) e = cudaMemcpyAsync(a.g2_host, d_g2, sizeof(float) * 3 * s2, cudaMemcpyDeviceToHost, stream);
    return e;
}

// A training loop calls the step with the same few pinned staging buffers over and over: the second time a
// (buffers, shape, workspace) combination is seen its stream work is captured into a CUDA graph, and from then on one
// cudaGraphLaunch replaces the API calls of a step (the host side, not the GPU, bounds a 40 us step otherwise).
struct StepGraph {
    const void *x1 = nullptr, *x2 = nullptr, *loss = nullptr, *g1 = nullptr, *g2 = nullptr, *g1u = nullptr, *ws = nullptr;
    int b = 0, n = 0, m = 0, variant = 0, device = -1, tc_ctas = 0, flags = 0;
    cudaGraphExec_t exec = nullptr;
    bool plain = false;   // capture was not possible (pageable buffers, stream already capturing): keep the plain path
    unsigned long long last_use = 0;
    bool same(const StepGraph &o) const {
        return x1 == o.x1 && x2 == o.x2 && loss == o.loss && g1 == o.g1 && g2 == o.g2 && g1u == o.g1u && ws == o.ws && b == o.b &&
               n == o.n && m == o.m && variant == o.variant && device == o.device && tc_ctas == o.tc_ctas && flags == o.flags;
    }
};
static const int kStepGraphs = 64;
static StepGraph g_step_graph[kStepGraphs];
static unsigned long long g_step_clock = 0;
static int g_step_graph_enabled = -1;   // -1: read PSD_HOST_STEP_GRAPH on first use

static void drop_step_graphs(const void *ws) {
    for (StepGraph &g : g_step_graph)
        if (g.ws == ws) {
            if (g.exec) cudaGraphExecDestroy(g.exec);
            g = StepGraph();
        }
}

static bool pinned_host(const void *p) {
    if (!p) return true;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

int psd_host_step_graphs(int enable) {
    std::lock_guard<std::mutex> api_lock(g_host_api_mutex);
    const int old = g_step_graph_enabled;
    if (enable == 0 || enable == 1) g_step_graph_enabled = enable;
    return old;
}

static int loss_step_common(const StepArgs &a, float **gradxyz1_dev, float **gradxyz2_dev, int slot, int sync, void *stream_) {
    if (slot < 0 || slot >= kStepSlots) { psd_set_error_msg("psd_chamfer_loss_step: slot must be 0..7"); return -1; }
    std::unique_lock<std::mutex> api_lock(g_host_api_mutex);
    cudaStream_t stream = (cudaStream_t)stream_;
    cudaError_t e0 = cudaSuccess;
    DeviceState *ds = psd::device_state(&e0);
    if (ds == nullptr) return finish("psd_chamfer_loss_step(device)", e0);
    const int b = a.b, n = a.n, m = a.m;
    const size_t s1 = (size_t)b * n, s2 = (size_t)b * m;
    const size_t nfloat = 6 * (s1 + s2) + 2 * (s1 + s2) + 2 * (size_t)b + 4;
    const size_t need = sizeof(float) * nfloat;
    if (need > ds->step_ws_bytes[slot]) {
        if (ds->step_ws[slot]) { cudaDeviceSynchronize(); drop_step_graphs(ds->step_ws[slot]); cudaFree(ds->step_ws[slot]); }
        ds->step_ws[slot] = nullptr; ds->step_ws_bytes[slot] = 0;
        cudaError_t e = cudaMalloc(&ds->step_ws[slot], need);
        if (e != cudaSuccess) return finish("psd_chamfer_loss_step(cudaMalloc)", e);
        ds->step_ws_bytes[slot] = need;
    }
    float *const ws = ds->step_ws[slot];
    if (gradxyz1_dev) *gradxyz1_dev = (a.x1_dev && a.g1_user) ? a.g1_user : ws + 3 * (s1 + s2);
    if (gradxyz2_dev) *gradxyz2_dev = ws + 3 * (s1 + s2) + 3 * s1;

    if (g_step_graph_enabled < 0) {
        const char *env = getenv("PSD_HOST_STEP_GRAPH");
        g_step_graph_enabled = (env && env[0] == '0') ? 0 : 1;
    }
    bool launched = false;
    if (g_step_graph_enabled && stream != nullptr && stream != cudaStreamLegacy) {
        StepGraph key;
        key.x1 = a.x1; key.x2 = a.x2; key.loss = a.loss_host; key.g1 = a.g1_host; key.g2 = a.g2_host; key.g1u = a.g1_user;
        key.ws = ws; key.b = b; key.n = n; key.m = m; key.variant = psd_set_nn_variant(-1); key.tc_ctas = psd_set_tc_max_ctas(-1);
        key.flags = (a.x1_dev ? 1 : 0) | (a.layout1 ? 2 : 0);
        key.device = ds->device;
        StepGraph *hit = nullptr, *victim = &g_step_graph[0];
        for (StepGraph &g : g_step_graph) {
            if (g.ws && g.same(key)) { hit = &g; break; }
            if (g.last_use < victim->last_use) victim = &g;
        }
        if (hit == nullptr) {   // first sighting: remember the combination, run the plain path below
            if (victim->exec) cudaGraphExecDestroy(victim->exec);
            *victim = key;
            victim->last_use = ++g_step_clock;
        } else {
            hit->last_use = ++g_step_clock;
            if (hit->exec == nullptr && !hit->plain &&
                !((a.x1_dev || pinned_host(a.x1)) && pinned_host(a.x2) && pinned_host(a.loss_host) && pinned_host(a.g1_host) &&
                  pinned_host(a.g2_host)))
                hit->plain = true;
            if (hit->exec == nullptr && !hit->plain) {
                cudaGraph_t graph = nullptr;
                cudaError_t e = cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal);
                if (e == cudaSuccess) {
                    e = enqueue_loss_step(a, ws, stream);
                    cudaError_t e2 = cudaStreamEndCapture(stream, &graph);
                    if (e == cudaSuccess) e = e2;
                }
                if (e == cudaSuccess) e = cudaGraphInstantiate(&hit->exec, graph, 0);
                if (graph) cudaGraphDestroy(graph);
                if (e != cudaSuccess) {
                    cudaGetLastError();
                    hit->exec = nullptr;
                    hit->plain = true;
                }
            }
            if (hit->exec) {
                cudaError_t e = cudaGraphLaunch(hit->exec, stream);
                if (e != cudaSuccess) return finish("psd_chamfer_loss_step(graph launch)", e);
                launched = true;
            }
        }
    }
    if (!launched) {
        cudaError_t e = enqueue_loss_step(a, ws, stream);
        if (e != cudaSuccess) return finish("psd_chamfer_loss_step(enqueue)", e);
    }
    api_lock.unlock();
    if (!sync) return 1;   // asynchronous: the caller synchronises `stream` before it reads loss_host / the gradients
    return finish("psd_chamfer_loss_step(sync)", cudaStreamSynchronize(stream));
}

int psd_chamfer_loss_step_host_ex(const float *xyz1_host, const float *xyz2_host, int b, int n, int m, float *loss_host,
                                  float *gradxyz1_host, float *gradxyz2_host, float **gradxyz1_dev, float **gradxyz2_dev,
                                  int slot, int sync, void *stream_) {
    StepArgs a;
    a.x1 = xyz1_host; a.x2 = xyz2_host; a.b = b; a.n = n; a.m = m; a.loss_host = loss_host;
    a.g1_host = gradxyz1_host; a.g2_host = gradxyz2_host;
    return loss_step_common(a, gradxyz1_dev, gradxyz2_dev, slot, sync, stream_);
}

int psd_chamfer_loss_step_host(const float *xyz1_host, const float *xyz2_host, int b, int n, int m, float *loss_host,
                               float *gradxyz1_host, float *gradxyz2_host, float **gradxyz1_dev, float **gradxyz2_dev,
                               void *stream_) {
    return psd_chamfer_loss_step_host_ex(xyz1_host, xyz2_host, b, n, m, loss_host, gradxyz1_host, gradxyz2_host, gradxyz1_dev,
                                         gradxyz2_dev, 0, 1, stream_);
}

int psd_chamfer_loss_step_pred_dev(const float *xyz1_dev, int layout1, const float *xyz2_host, int b, int n, int m,
                                   float *loss_host, float *gradxyz1_dev, int slot, int sync, void *stream_) {
    if (layout1 != 0 && layout1 != 1) { psd_set_error_msg("psd_chamfer_loss_step_pred_dev: layout1 must be 0 ([B,N,3]) or 1 ([B,3,N])"); return -1; }
    StepArgs a;
    a.x1 = xyz1_dev; a.x1_dev = true; a.layout1 = layout1; a.x2 = xyz2_host; a.b = b; a.n = n; a.m = m; a.loss_host = loss_host;
    a.g1_user = gradxyz1_dev;
    return loss_step_common(a, nullptr, nullptr, slot, sync, stream_);
}

}  // extern "C"

// ---- FP32 FMA peak microbenchmark (roofline denominator, measured live by bench.py)
namespace {
__global__ void __launch_bounds__(256) ffma_peak_kernel(float *out, int iters, float seed) {
    float a[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = seed * (float)(i + 1) + (float)threadIdx.x;
    const float b = seed * 0.5f, c = seed * 0.25f;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) a[i] = __fmaf_rn(a[i], b, c);
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += a[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
}  // namespace

extern "C" int psd_fp32_fma_peak(float ms_target, float *tflops, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    int dev = 0, num_sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    const int grid = num_sms * 8, block = 256;
    float *out = nullptr;
    cudaError_t e = cudaMalloc(&out, sizeof(float) * grid * block);
    if (e != cudaSuccess) return finish("psd_fp32_fma_peak(cudaMalloc)", e);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    // per launch: grid*block*iters*16 FMAs; at ~74 TFLOP/s, iters=4096 takes about 0.55 ms
    int iters = 4096;
    if (ms_target > 0.f) iters = (int)(4096.f * ms_target / 0.55f);
    if (iters < 256) iters = 256;
    ffma_peak_kernel<<<grid, block, 0, stream>>>(out, iters, 1.0001f);  // warm-up
    float best_ms = 1e30f;
    for (int r = 0; r < 5; ++r) {
        cudaEventRecord(e0, stream);
        ffma_peak_kernel<<<grid, block, 0, stream>>>(out, iters, 1.0001f);
        cudaEventRecord(e1, stream);
        cudaEventSynchronize(e1);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best_ms) best_ms = ms;
    }
    e = cudaGetLastError();
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    if (e != cudaSuccess) return finish("psd_fp32_fma_peak", e);
    *tflops = (float)(2.0 * 16.0 * (double)iters * (double)grid * (double)block / ((double)best_ms * 1e-3) / 1e12);
    return 1;
}
