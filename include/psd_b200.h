/*
 * psd_b200.h -- C ABI of the B200-native point-set-distance library (libpsd_b200.so).
 *
 * Drop-in boundary for the hot path of sunhui-3D/3D-PointCloudReconstruction (3D-FENet): the two
 * native modules `chamfer_3D` and `emd` that the reference binds with pybind11.  Every entry point
 * below names the reference interface it replaces (paths relative to the reference repo root).
 * Plain pointers and sizes only: no torch types cross this boundary.  All pointers are DEVICE
 * pointers on the current CUDA device unless a name ends in `_host`; `stream` is a cudaStream_t
 * passed as void* (NULL = the legacy default stream, which is what the reference launches on).
 *
 * Layout contract (same as the reference, metric/chamfer3D/chamfer3D.cu:12-25, emd_cuda.cu:95-123):
 * row-major contiguous fp32 clouds [B, N, 3], fp32 distances [B, N], int32 indices [B, N].
 *
 * Return convention (same as the reference): 1 = ok, 0 = CUDA error (message via psd_last_error(),
 * the reference printf()s it), -1 = shape violation (EMD only, emd_cuda.cu:236-249).
 * The kernels are asynchronous on `stream`; nothing here synchronises the host.
 */
#ifndef PSD_B200_H_
#define PSD_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

/* Library / ABI version: major * 1000 + minor. */
int psd_version(void);

/* Last error message of the calling thread ("" if none). */
const char *psd_last_error(void);

/* ---------------------------------------------------------------------------------------------
 * Chamfer distance.
 * ------------------------------------------------------------------------------------------- */

/* Replaces chamfer_3D.forward(xyz1, xyz2, dist1, dist2, idx1, idx2)
 *   = chamfer_forward, metric/chamfer3D/chamfer_cuda.cpp:17-19
 *   -> chamfer_cuda_forward, metric/chamfer3D/chamfer3D.cu:136-154 (two NmDistanceKernel launches).
 * dist1[b, j] = min_k |xyz1[b, j] - xyz2[b, k]|^2 evaluated as fma(dz,dz, fma(dx,dx, rn(dy*dy))) with
 * d* = xyz2 - xyz1, idx1[b, j] = the lowest k attaining it; dist2/idx2 the same with the roles swapped.
 * Bit-exact with the reference for finite inputs; NaN inputs follow the reference's 512-target-tile
 * semantics (chamfer3D.cu:36,126).  One kernel launch for both directions. */
int psd_chamfer_forward(const float *xyz1, const float *xyz2, int b, int n, int m, float *dist1, float *dist2,
                        int *idx1, int *idx2, void *stream);

/* Extended forward: the same NN search with fused epilogues and the generator's native layout.
 *   layout   : bit mask.  bit 0 (1): xyz1 is [B, 3, N]; bit 1 (2): xyz2 is [B, 3, M]; a clear bit means the reference layout
 *              [B, N, 3].  1 is the training step's call (train.py:163: the generator output fake[B,3,N] against the
 *              ground truth points[B,N,3]) -- it removes dist_chamfer_3D.py:79-80's .contiguous() transpose copy.
 *   sums     : optional [B, 2] fp32, sums[b] += (sum_j dist1[b, j], sum_k dist2[b, k])   (loss/loss.py:36)
 *   fs_thr   : F-score threshold on the squared distances (loss/loss_.py:122, default 1e-4)
 *   fs_count : optional [B, 2] int32, fs_count[b] += (#{dist1[b,:] < thr}, #{dist2[b,:] < thr})  (loss_.py:132-133)
 * sums / fs_count are accumulated with atomics and must be zeroed by the caller.
 * q_begin/q_count select a slice of the QUERY points of both directions (query sharding across GPUs:
 * rank r passes its slice, targets stay whole); pass 0 and -1 for everything.  Outputs are still
 * indexed by the global query index.  Returns -1 for an invalid layout. */
int psd_chamfer_forward_ex(const float *xyz1, const float *xyz2, int b, int n, int m, int layout, float *dist1,
                           float *dist2, int *idx1, int *idx2, float *sums, float fs_thr, int *fs_count, int q_begin,
                           int q_count, void *stream);

/* psd_chamfer_forward_ex over all queries that ALSO zero-fills zero_buf[0 .. zero_floats) inside the same launch (a few
 * stores per thread before the search starts): pass the gradient buffers that the backward following on the stream will
 * accumulate into and the step needs no memset (the reference's wrapper zero-fills them on the CPU and copies,
 * dist_chamfer_3D.py:62-66).  zero_buf may be NULL. */
int psd_chamfer_forward_zero(const float *xyz1, const float *xyz2, int b, int n, int m, int layout, float *dist1,
                             float *dist2, int *idx1, int *idx2, float *sums, float fs_thr, int *fs_count, float *zero_buf,
                             long long zero_floats, void *stream);

/* Replaces chamfer_3D.backward(xyz1, xyz2, gradxyz1, gradxyz2, graddist1, graddist2, idx1, idx2)
 *   = chamfer_backward, metric/chamfer3D/chamfer_cuda.cpp:22-26
 *   -> chamfer_cuda_backward, metric/chamfer3D/chamfer3D.cu:176-195 (two NmDistanceGradKernel launches).
 * ACCUMULATES into gradxyz1/gradxyz2 (the reference relies on caller-zeroed buffers, chamfer3D.cu:177-178):
 *   g = 2*graddist1[b,j]; v = g*(xyz1[b,j]-xyz2[b,idx1[b,j]]); gradxyz1[b,j] += v; gradxyz2[b,idx1[b,j]] -= v
 * and the mirror image for direction 2.  One launch; scatter uses warp-aggregated atomics. */
int psd_chamfer_backward(const float *xyz1, const float *xyz2, float *gradxyz1, float *gradxyz2,
                         const float *graddist1, const float *graddist2, const int *idx1, const int *idx2, int b, int n,
                         int m, void *stream);

/* The same gradient with the layouts of psd_chamfer_forward_ex (a gradient has the layout of its cloud) and, with
 * overwrite != 0, WITHOUT the caller-zeroed contract: a first launch stores every point's own term (each element of both
 * gradients exactly once), a second one adds the scatter terms.  overwrite == 0 accumulates like psd_chamfer_backward;
 * the cheapest step is overwrite == 0 on buffers that the FORWARD launch zero-filled (psd_chamfer_forward_zero). */
int psd_chamfer_backward_ex(const float *xyz1, const float *xyz2, float *gradxyz1, float *gradxyz2,
                            const float *graddist1, const float *graddist2, const int *idx1, const int *idx2, int b, int n,
                            int m, int layout, int overwrite, void *stream);

/* Ragged batches in one launch.  xyz1 [b, n, 3] and xyz2 [b, m, 3] are padded (layout as psd_chamfer_forward_ex); pair c
 * takes part with its first len1[c] points of xyz1 and len2[c] points of xyz2 (device int [b]; NULL = n / m for every pair).
 * Points beyond the lengths are never read (they may hold NaN, inf or garbage).  dist / idx of pair c are the bits of
 * psd_chamfer_forward on its participating points alone (lowest index on ties, the reference's 512-target NaN rule);
 * rows beyond the lengths get dist 0 and idx -1 and add nothing to sums / fs_count (optional [b, 2], caller-zeroed, as in
 * psd_chamfer_forward_ex).  A pair with a length outside [1, n] / [1, m] gets dist NaN and idx -1 in every row, NaN sums
 * and zero counts, without affecting the others.  zero_buf / zero_floats: as in psd_chamfer_forward_zero.  The launch
 * grid is that of the padded sizes and the lengths are read on the device only: no host synchronisation, graph-capturable.
 * psd_chamfer_nn_variant applies.  Returns -1 for a bad layout, else the convention above. */
int psd_chamfer_forward_ragged(const float *xyz1, const float *xyz2, int b, int n, int m, int layout, const int *len1,
                               const int *len2, float *dist1, float *dist2, int *idx1, int *idx2, float *sums, float fs_thr,
                               int *fs_count, float *zero_buf, long long zero_floats, void *stream);
/* The gradient of psd_chamfer_forward_ragged, accumulated into caller-zeroed buffers (psd_chamfer_backward's form, e.g. the
 * buffers the ragged forward zero-filled).  Rows beyond the lengths get no term (their gradient stays 0) and their graddist
 * entries are never read; every gradient row of a pair with an invalid length becomes NaN. */
int psd_chamfer_backward_ragged(const float *xyz1, const float *xyz2, float *gradxyz1, float *gradxyz2,
                                const float *graddist1, const float *graddist2, const int *idx1, const int *idx2,
                                const int *len1, const int *len2, int b, int n, int m, int layout, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Earth mover's distance, auction approximation.
 * ------------------------------------------------------------------------------------------- */

/* Replaces emd.forward(xyz1, xyz2, dist, assignment, price, assignment_inv, bid, bid_increments,
 *                      max_increments, unass_idx, unass_cnt, unass_cnt_sum, cnt_tmp, max_idx, eps, iters)
 *   = emd_forward, metric/emd/emd.cpp:12-17 -> emd_cuda_forward, metric/emd/emd_cuda.cu:228-282
 *   (7 launches per iteration + CalcDist; here one persistent launch).
 * Caller-initialised state exactly as metric/emd/emd_module.py:43-54: assignment = assignment_inv = -1,
 * everything else 0.  dist and assignment are the results; price and assignment_inv are left in their final
 * state; the remaining scratch tensors may be NULL (they are not needed by this implementation).
 * Winner rule among bidders within +-1e-6 of an object's maximum increment: lowest bidder index
 * (the reference's GetMax, emd_cuda.cu:188-191, is a last-writer-wins race).
 * Returns -1 if m != n, b > 512 or n % 1024 != 0 (emd_cuda.cu:236-249). */
int psd_emd_forward(const float *xyz1, const float *xyz2, int b, int n, int m, float *dist, int *assignment,
                    float *price, int *assignment_inv, int *bid, float *bid_increments, float *max_increments,
                    int *unass_idx, int *unass_cnt, int *unass_cnt_sum, int *cnt_tmp, int *max_idx, float eps,
                    int iters, void *stream);

/* Same auction when the caller has no state to hand over: starts from assignment = -1, price = 0 inside the
 * kernel (what emd_module.py:43-54 builds with 12 allocator calls and fills) and writes only dist and
 * assignment.  One launch, no host-side fills. */
int psd_emd_forward_fresh(const float *xyz1, const float *xyz2, int b, int n, float *dist, int *assignment, float eps,
                          int iters, void *stream);

/* Test hook (not part of the reference surface): the same auction with the cluster size forced to
 * 1, 2, 4 or 8 CTAs per cloud, so that every decomposition can be parity-checked against the oracle.  A NEGATIVE
 * cluster_size runs the global-workspace form of the kernel (the one clouds of more than 8192 points take, whose state
 * does not fit the shared memory of a cluster) with |cluster_size| CTAs per cloud. */
int psd_emd_forward_cluster(const float *xyz1, const float *xyz2, int b, int n, float *dist, int *assignment,
                            float *price, int *assignment_inv, float eps, int iters, int cluster_size, void *stream);

/* Replaces emd.backward(xyz1, xyz2, gradxyz, graddist, idx)
 *   = emd_backward, metric/emd/emd.cpp:19-23 -> emd_cuda_backward, metric/emd/emd_cuda.cu:302-316.
 * gradxyz[b,j] += 2*graddist[b,j]*(xyz1[b,j] - xyz2[b,idx[b,j]]) (xyz1 only; emd_module.py:84-87). */
int psd_emd_backward(const float *xyz1, const float *xyz2, float *gradxyz, const float *graddist, const int *idx,
                     int b, int n, void *stream);
/* overwrite != 0: gradxyz is stored, not accumulated (one term per address: no zero fill needed before the call). */
int psd_emd_backward_ex(const float *xyz1, const float *xyz2, float *gradxyz, const float *graddist, const int *idx,
                        int b, int n, int overwrite, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Certified earth mover's distance (not part of the reference surface).
 * ------------------------------------------------------------------------------------------- */

/* Weak-duality certificate of an (assignment, prices) pair.  With d_jk = |xyz1[b,j] - xyz2[b,k]| (Euclidean, not squared):
 *   L = sum_j min_k (d_jk + price[b,k]) - sum_k price[b,k]  <=  optimal matching cost  <=  U = sum_j d(j, assignment[b,j])
 * where L holds for ANY prices and U whenever the assignment is a permutation.  Outputs per cloud: bounds[b] = (L / n, U / n)
 * fp64, the unit of sqrt(dist).mean(1); status[b] = 1 (a permutation, both bounds valid) or 0 (not a permutation: the lower
 * bound is still valid, the upper one is NaN).  Every term is rounded towards its bound (fp64 directed rounding) and the sums
 * run in a fixed order, so the bounds are rigorous for the fp32 inputs and reproducible bit for bit.  price may be NULL (all
 * zero).  A cloud with a NaN or infinite coordinate in xyz1 or xyz2 has no certificate: both bounds NaN, status 0.  A NaN
 * price makes the lower bound NaN (the upper bound and status do not depend on prices).  Any n in [1, 2^20], b <= 65535;
 * about one fp64 evaluation of every pair.  Returns 1 / 0 CUDA error / -1 argument. */
int psd_emd_dual_bound(const float *xyz1, const float *xyz2, int b, int n, const int *assignment, const float *price,
                       double *bounds, int *status, void *stream);

/* The auction run to a true matching by epsilon-scaling, with its certificate.  Phases with eps = eps_start, eps_start / scale,
 * ... (computed in double, rounded to float) down to exactly eps_end, each one the auction of psd_emd_forward started from
 * assignment = -1 and the PREVIOUS phase's prices, run until every point is assigned or max_iters_per_phase iterations (a phase
 * that runs out of iterations ends with the auction's forced assignment, which the certificate reports as status 0; several
 * winners of one object then add to its price in the same iteration, as in the reference, so such a result is not
 * reproducible bit for bit, while its certificate stays valid).  Then
 * psd_emd_dual_bound on the final (assignment, price).  Outputs: dist [B, n] (squared, as psd_emd_forward), assignment [B, n],
 * price [B, n] (final prices), bounds [B, 2], status [B].  U - L <= eps_end per point is what epsilon-complementary slackness
 * gives; the certificate measures it instead of assuming it.  Everything is enqueued on `stream` with no host
 * synchronisation (a call can be captured in a CUDA graph); one launch per phase plus two for the certificate.
 * Limits of psd_emd_forward (b <= 512, n % 1024 == 0, coordinates in [0, 1]); -1 also for eps_end < 1e-5 (the kernel's fp32
 * prices and +-1e-6 winner window make a smaller eps meaningless), eps_end > eps_start, scale <= 1, max_iters_per_phase < 1 and
 * more than 64 phases. */
int psd_emd_certified(const float *xyz1, const float *xyz2, int b, int n, float eps_start, float eps_end, float scale,
                      int max_iters_per_phase, float *dist, int *assignment, float *price, double *bounds, int *status,
                      void *stream);
/* Test hook: psd_emd_certified with the cluster size of every phase forced as in psd_emd_forward_cluster (negative = the
 * global-workspace form). */
int psd_emd_certified_cluster(const float *xyz1, const float *xyz2, int b, int n, float eps_start, float eps_end, float scale,
                              int max_iters_per_phase, float *dist, int *assignment, float *price, double *bounds, int *status,
                              int cluster_size, void *stream);

/* Fused training loss of the EMD term: Loss.get_emd_loss (loss/loss.py:18-28) = sqrt(dist).mean(1).mean() over emdModule's
 * distances.  Forward: the auction kernel adds sum_j sqrt(dist[b, j]) to sums_zeroed[b] (zero-filled by the caller) in its
 * CalcDist tail and a one-warp kernel reduces them to the scalar *loss (device); dist / assignment are still written.
 * Backward: gradxyz1[b,j] = 2 g (xyz1[b,j] - xyz2[b,assignment[b,j]]) with g = ((*upstream / B) / n) / (2 sqrt(dist[b,j]))
 * formed in the kernel (autograd's sequence, including the infinite factor at dist == 0; upstream NULL = 1.0); gradxyz1 is
 * stored, not accumulated.  Same return convention as psd_emd_forward_fresh. */
int psd_emd_mean_loss_forward(const float *xyz1, const float *xyz2, int b, int n, float *dist, int *assignment, float eps,
                              int iters, float *sums_zeroed, float *loss, void *stream);
int psd_emd_mean_loss_backward(const float *xyz1, const float *xyz2, float *gradxyz1, const float *dist, const int *assignment,
                               const float *upstream, int b, int n, void *stream);

/* Debiased Sinkhorn divergence per cloud pair (geomloss SamplesLoss("sinkhorn", p=2, blur, scaling, debias=True), uniform
 * weights, cost |u - v|^2 / 2), for clouds x [b, n, 3] and y [b, m, 3] of any sizes, anywhere in space.  The epsilon schedule
 * runs from the squared diameter of both clouds down to blur^2 by factors scaling^2, each value rounded to fp32 and raised to
 * at least 2^-128 so that 1/eps stays finite (this changes only a diameter or blur below 5.4e-20); rounds[b] (optional)
 * receives its length, len(eps_list).  Outputs: loss[b] = S; grad_x [b, n, 3] and grad_y [b, m, 3] (each optional) dS/dx and dS/dy of geomloss's
 * last extrapolation step; potentials [b, 2n + 2m] (optional) the final f_ba, f_aa (n each), g_ab, g_bb (m each).  A pair
 * whose points all coincide gives S = 0, zero gradients and potentials, 0 rounds; a pair with a NaN or infinite coordinate
 * gives NaN everywhere and 0 rounds, without affecting the other pairs.  Deterministic: no float atomics, and the result does
 * not depend on the launch decomposition.  One launch plus a stream-ordered workspace of 2 (2n + 2m) floats per pair; no host
 * synchronisation (capturable in a CUDA graph).  Returns 1 / 0 CUDA error / -1 argument: b outside [0, 65535], n or m
 * outside [1, 2^20], blur not finite and > 0, scaling outside (0, 1), loss NULL.  b = 0 does nothing and returns 1. */
int psd_sinkhorn_divergence(const float *x, const float *y, int b, int n, int m, float blur, float scaling, float *loss,
                            float *grad_x, float *grad_y, float *potentials, int *rounds, void *stream);
/* Test hook: the same with the cluster size (CTAs per cloud pair) forced to 1, 2, 4 or 8 (-1 for another value). */
int psd_sinkhorn_divergence_cluster(const float *x, const float *y, int b, int n, int m, float blur, float scaling, float *loss,
                                    float *grad_x, float *grad_y, float *potentials, int *rounds, int cluster_size, void *stream);
/* The same for ragged and weighted batches.  x [b, n, 3] and y [b, m, 3] are padded; pair c takes part with its first
 * x_len[c] points of x and y_len[c] points of y (device int [b]; NULL = n / m for every pair), with the point weights
 * x_w [b, n] and y_w [b, m] (device fp32; NULL = uniform 1 / length).  Points beyond the lengths are never read.  The
 * diameter, the schedule and every softmin use the participating points only; a weight w enters as log w in the softmins
 * (a weight of 0 removes the point as a target), as w in the gradient row and in S = sum_i a_i (f_ba - f_aa) +
 * sum_j b_j (g_ab - g_bb), summed in fp64.  Weights are not normalised: that they sum to 1 per side is the caller's contract,
 * as in geomloss.  Outputs keep the padded shapes; gradient rows and potential entries beyond the lengths are 0.  A pair gets
 * NaN loss, NaN in every gradient and potential row and 0 rounds, without affecting the others, when a coordinate is not
 * finite, a length is outside [1, n] / [1, m], a participating weight is negative, NaN or infinite, or all participating
 * weights of one side are 0.  Each pair gives the bits of a psd_sinkhorn_divergence call on its participating points alone
 * when the weights are NULL.  Same argument checks and return convention as psd_sinkhorn_divergence; lengths and weights are
 * device data and are not checked on the host. */
int psd_sinkhorn_divergence_weighted(const float *x, const float *y, int b, int n, int m, const int *x_len, const int *y_len,
                                     const float *x_w, const float *y_w, float blur, float scaling, float *loss, float *grad_x,
                                     float *grad_y, float *potentials, int *rounds, void *stream);
/* Test hook: the same with the cluster size forced as in psd_sinkhorn_divergence_cluster. */
int psd_sinkhorn_divergence_weighted_cluster(const float *x, const float *y, int b, int n, int m, const int *x_len,
                                             const int *y_len, const float *x_w, const float *y_w, float blur, float scaling,
                                             float *loss, float *grad_x, float *grad_y, float *potentials, int *rounds,
                                             int cluster_size, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Fused training loss of the hot path's caller: Loss.get_chamfer_loss (loss/loss.py:30-37) =
 * mean(dist1) + mean(dist2) over chamfer_3DDist's outputs.  Forward: the NN kernel accumulates per-cloud sums in its
 * epilogue (sums_zeroed[B,2], zero-filled by the caller) and a one-warp kernel reduces them to the scalar *loss (device);
 * dist/idx are still written.  Backward: what autograd would hand to psd_chamfer_backward for this loss, graddist1 =
 * *upstream/(B*N), graddist2 = *upstream/(B*M), is formed inside the kernel from the device scalar `upstream`
 * (NULL = 1.0), so no gradient tensors are materialised; gradxyz1/gradxyz2 must be zero-filled by the caller.
 * The _ex form takes the layout mask of psd_chamfer_forward_ex and, with overwrite != 0, needs no zero fill
 * (see psd_chamfer_backward_ex).  Same return convention as above. */
int psd_chamfer_mean_loss_forward(const float *xyz1, const float *xyz2, int b, int n, int m, int layout, float *dist1,
                                  float *dist2, int *idx1, int *idx2, float *sums_zeroed, float *loss, void *stream);
int psd_chamfer_mean_loss_forward_zero(const float *xyz1, const float *xyz2, int b, int n, int m, int layout, float *dist1,
                                       float *dist2, int *idx1, int *idx2, float *sums_zeroed, float *loss, float *zero_buf,
                                       long long zero_floats, void *stream);   /* + the zero fill of psd_chamfer_forward_zero */
int psd_chamfer_mean_loss_backward(const float *xyz1, const float *xyz2, float *gradxyz1, float *gradxyz2,
                                   const float *upstream, const int *idx1, const int *idx2, int b, int n, int m, void *stream);
int psd_chamfer_mean_loss_backward_ex(const float *xyz1, const float *xyz2, float *gradxyz1, float *gradxyz2,
                                      const float *upstream, const int *idx1, const int *idx2, int b, int n, int m, int layout,
                                      int overwrite, void *stream);

/* ---------------------------------------------------------------------------------------------
 * psd_proj_min_dist  =  the min-distance branch of get_loss_proj, loss/proj_loss.py:21-40 (with grid_dist, :46-54).
 * pred, gt: [B,H,W] fp32 projection images (device); table: [H,W] fp32 with table[dh*W+dw] = float32(sqrt(dh^2+dw^2)) + k,
 * k = how often the caller's `dist_mat += 1` has run (1 in finetune.py:154-158).  Outputs min_dist, min_dist_inv [B,H,W].
 * mode 0 = as written (weights broadcast along the first pixel pair: the minimum over (h',w') collapses to an end point of
 * the distance range; bit-exact with the reference's dense evaluation), mode 1 = intended CAPNet-style masked nearest
 * pixel search (weights on the target pixel).  Returns 1 ok / 0 CUDA error / -1 argument error.
 * ------------------------------------------------------------------------------------------- */
int psd_proj_min_dist(const float *pred, const float *gt, const float *table, int b, int h, int w, int mode, float *min_dist,
                      float *min_dist_inv, void *stream);

/* ---------------------------------------------------------------------------------------------
 * psd_icp_batch  =  icp(A, B, init_pose, max_iterations, tolerance) of utils/icp.py:68-118 for a whole batch in ONE launch
 * (the reference runs it per sample on the CPU: testnet.py:62-64, test_pix3d.py:62-64, tolerance 1e-10, 1024 iterations).
 * a, b: [batch, n, 3] source / destination clouds on the device, fp32 (in_f64 = 0) or fp64 (in_f64 = 1); n <= 4096.
 * init_pose: optional device 4x4 fp64 row-major rigid transform (last row 0 0 0 1) applied to every source, or NULL.
 * Each sample iterates NN (nearest_neighbor, :49-65) -> best_fit_transform (:4-46) -> src = T src until
 * |prev_error - mean_error| < tolerance or max_iterations, on its own.  Outputs (device): T_out [batch,4,4] fp64 row-major =
 * best_fit_transform(A, final src); distances [batch,n] fp64 (last NN pass; may be NULL); iterations [batch] = the
 * reference's returned `i` (may be NULL).  max_iterations = 0 returns best_fit_transform(A, B) of the given correspondences.
 * All arithmetic is fp64.  Returns 1 ok / 0 CUDA error / -1 argument error.
 *
 * psd_nn_f64  =  nearest_neighbor(src, dst) (utils/icp.py:49-65) for a batch: distances [batch,n_src] fp64 (Euclidean, not
 * squared) and indices [batch,n_src] int32 into dst; n_dst <= 8533.
 * ------------------------------------------------------------------------------------------- */
int psd_icp_batch(const void *a, const void *b, int in_f64, int batch, int n, const double *init_pose, int max_iterations,
                  double tolerance, double *T_out, double *distances, int *iterations, void *stream);
int psd_nn_f64(const void *src, const void *dst, int in_f64, int batch, int n_src, int n_dst, double *distances, int *indices,
               void *stream);
/* The same for ragged batches: a [batch, n, 3] and b [batch, m, 3] are padded (fp32 or fp64 as in psd_icp_batch), and sample
 * s aligns its first len_a[s] source points to its first len_b[s] destination points (device int [batch]; NULL = n / m),
 * which need not be equal.  Points beyond the lengths are never read.  Outputs keep the padded shapes: distances
 * [batch, n] is 0 beyond len_a[s].  A sample with a length outside [1, n] / [1, m] gets T all NaN, a NaN distance row and
 * iterations -1, without affecting the others.  Each sample with len_a[s] == len_b[s] gives the bits of psd_icp_batch on
 * its participating points alone.  The lengths are device data and are not read on the host (no synchronisation; capturable
 * in a CUDA graph).  Returns -1 for batch < 0, n < 1, m < 1, n > 4096, n + m > 8192 or max_iterations < 1 (the
 * max_iterations = 0 mode of psd_icp_batch needs equal sizes); otherwise as psd_icp_batch. */
int psd_icp_batch_ragged(const void *a, const void *b, int in_f64, int batch, int n, int m, const int *len_a, const int *len_b,
                         const double *init_pose, int max_iterations, double tolerance, double *T_out, double *distances,
                         int *iterations, void *stream);

/* ---------------------------------------------------------------------------------------------
 * psd_farthest_point_sample  =  farthest_point_sample(xyz, npoint, RAN) of utils/utils.py:335-360 (called by the dataset
 * for the 128- and 256-point ground-truth clouds, utils/datasets_sample_pcl.py:87-91).
 * xyz: [B, N, 3] fp32 device; centroids: [B, npoint] int64 device (the reference returns torch.long).  start = the first
 * centroid: the reference draws torch.randint(0, 1) = 0 when RAN is true and torch.randint(1, 2) = 1 otherwise.
 * Distances are fp32 ((dx*dx + dy*dy) + dz*dz, no contraction), ties go to the lowest index: the indices are bit-identical
 * to the reference's on the CPU.  N <= 16384.  Returns 1 ok / 0 CUDA error / -1 argument error.
 * ------------------------------------------------------------------------------------------- */
int psd_farthest_point_sample(const float *xyz, int b, int n, int npoint, int start, long long *centroids, void *stream);

/* ---------------------------------------------------------------------------------------------
 * psd_cont_proj  =  cont_proj(pcl, grid_h, grid_w, device, sigma_sq) of utils/projection.py:4-67 (Gaussian splat of a cloud
 * to a silhouette image; feeds get_loss_proj, utils/utils.py:232,241).
 * pcl: [B, N, 3] fp32 device, coordinates in (-1, 1); out: [B, grid_h, grid_w] fp32 device,
 *   out[b,h,w] = sum_p exp(-(x_p - h)^2 / (2 sigma_sq)) * exp(-(y_p - w)^2 / (2 sigma_sq)),
 *   x_p = ((p.x + 1) * grid_h) / 2, y_p = ((p.y + 1) * grid_w) / 2,
 * with the reference's fp32 rounding sequence and summation order (points in order); the only difference to the CPU reference
 * is the last ulp of expf.  Returns 1 ok / 0 CUDA error / -1 argument error.
 * ------------------------------------------------------------------------------------------- */
int psd_cont_proj(const float *pcl, int b, int n, int grid_h, int grid_w, float sigma_sq, float *out, void *stream);
/* Its backward (the reference's cont_proj is differentiable torch code): grad_pcl [B, N, 3] = d loss / d pcl for
 * grad_out [B, grid_h, grid_w] = d loss / d out; the z component is zero.  grad_pcl is stored, not accumulated.  The gradient
 * image of a sample is staged in shared memory: grid_h * (grid_w + 1) + 8 (grid_h + grid_w) floats <= 200 KB (about 220 x 220),
 * else -1. */
int psd_cont_proj_backward(const float *pcl, const float *grad_out, int b, int n, int grid_h, int grid_w, float sigma_sq,
                           float *grad_pcl, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Host-buffer convenience entry points (end-to-end path: pinned or pageable HOST pointers, the library
 * stages them through its own device workspace on `stream` and copies the results back).
 * ------------------------------------------------------------------------------------------- */
int psd_chamfer_forward_host(const float *xyz1_host, const float *xyz2_host, int b, int n, int m, float *dist1_host,
                             float *dist2_host, int *idx1_host, int *idx2_host, void *stream);

/* One training step of the chamfer loss with HOST inputs (pinned or pageable): H2D of both clouds (one copy when
 * xyz2_host == xyz1_host + 3*b*n), forward, fused mean loss (loss/loss.py:36), backward of that loss (upstream 1.0), the
 * scalar loss copied to *loss_host, then a stream synchronise.  Gradients are copied to gradxyz1_host / gradxyz2_host
 * when those are non-NULL; *gradxyz1_dev / *gradxyz2_dev (when non-NULL) receive the device pointers of the gradients,
 * valid until the next call (they feed the caller's own backward on the device).  Same return convention. */
int psd_chamfer_loss_step_host(const float *xyz1_host, const float *xyz2_host, int b, int n, int m, float *loss_host,
                               float *gradxyz1_host, float *gradxyz2_host, float **gradxyz1_dev, float **gradxyz2_dev,
                               void *stream);
/* The same step on workspace `slot` (0..7); with sync == 0 the call only enqueues the work on `stream` and returns, so a
 * training loop can keep several steps in flight, each on its own slot and stream: the H2D copy of step s+2 and the host's
 * own latency (wake-up after step s-1, the next call) then hide behind the kernels of steps s and s+1.  The caller
 * synchronises the stream before reading loss_host (which must then be pinned) or the gradients. */
int psd_chamfer_loss_step_host_ex(const float *xyz1_host, const float *xyz2_host, int b, int n, int m, float *loss_host,
                                  float *gradxyz1_host, float *gradxyz2_host, float **gradxyz1_dev, float **gradxyz2_dev,
                                  int slot, int sync, void *stream);
/* The training step as the reference's loop has it (train.py:160-163): the PREDICTION is already on the device (the
 * generator's output, layout1 = 1 for its native [B,3,N], 0 for [B,N,3]) and only the ground truth comes from the host.
 * H2D of xyz2, forward, fused mean loss, backward; d loss / d xyz1 is stored to gradxyz1_dev (device, the layout of xyz1; NULL =
 * kept in the workspace), the loss is copied to *loss_host.  slot / sync / stream as above. */
int psd_chamfer_loss_step_pred_dev(const float *xyz1_dev, int layout1, const float *xyz2_host, int b, int n, int m,
                                   float *loss_host, float *gradxyz1_dev, int slot, int sync, void *stream);
/* Repeated calls of the host step with the same pinned buffers, shape, slot and a non-default stream are replayed from a
 * cached CUDA graph (one cudaGraphLaunch instead of nine API calls per step) from the second sighting on; pageable
 * buffers and the default stream always take the plain path.  enable: 0 / 1 sets it, anything else only queries;
 * returns the previous setting (-1 = not decided yet: env PSD_HOST_STEP_GRAPH=0 disables).  The result is identical. */
int psd_host_step_graphs(int enable);

/* ---------------------------------------------------------------------------------------------
 * Measurement helpers (used by bench.py; not part of the reference surface).
 * ------------------------------------------------------------------------------------------- */

/* FP32-FMA roofline denominator measured live: runs an FFMA-only kernel on every SM for roughly
 * `ms_target` milliseconds and returns the achieved TFLOP/s (2 flop per FMA per lane) in *tflops. */
int psd_fp32_fma_peak(float ms_target, float *tflops, void *stream);

/* Counters of the chamfer forward's exact-fallback path since the last reset (diagnostics):
 * out[0] = queries resolved by the filtered path, out[1] = queries that took the exact full scan. */
int psd_chamfer_stats(long long *out_host2, int reset);

/* Test/measurement hook: choose the chamfer NN forward kernel.  0 = automatic (default: the tensor-core kernel when
 * the launch has at least two 128-query units per SM, else the FFMA kernel), 1 = FFMA kernel, 3 = tensor-core (tcgen05)
 * kernel; any other value only queries.  Both produce identical results.  Returns the previous setting. */
int psd_chamfer_nn_variant(int variant);

/* Test / profiling switch of the auction kernel's solo mode (once a cloud is down to <= 32 unassigned points, one CTA of its
 * cluster finishes the auction alone, one warp per bidder, without cluster barriers; results are identical).  enable: 0 / 1
 * sets it, anything else only queries; returns the previous setting.  Default 1. */
int psd_emd_solo_mode(int enable);
/* The same kind of switch for the auction kernel's object grid (bidders visit the grid cells around them shell by shell and
 * stop at their exact pruning radius instead of testing all n objects; results are identical).  Default 1. */
int psd_emd_grid_mode(int enable);
/* Upper bound on the CTAs of one launch of the tensor-core NN kernel (0 = one per SM, the default; a negative value only
 * queries).  A caller that keeps several launches in flight on different streams (a pipelined training loop) can set it to
 * half the SM count: every CTA then owns twice as many units, so its serial prologue and tail amortise, and the launch on
 * the other stream fills the remaining SMs.  Returns the previous value.  Results are identical. */
int psd_chamfer_tc_ctas(int max_ctas);

/* Bring-up / calibration hook of the tensor-core kernel: runs psd_chamfer_forward on that kernel and additionally
 * dumps every raw filter value a_k (before the exact rescan) to dump[(unit*128 + row) * dump_ld + target], where a
 * unit is a block of 128 queries in launch order (direction 1 blocks first).  dump_ld >= n and m rounded up to 128. */
int psd_debug_tc_filter(const float *xyz1, const float *xyz2, int b, int n, int m, float *dist1, float *dist2, int *idx1,
                        int *idx2, float *dump, int dump_ld, void *stream);

/* Phase clocks of the tensor-core kernel (tools/tc_phase_clocks.py): while prof_dev is non-NULL every launch of that
 * kernel runs its instrumented build and writes 64 clock64 slots per CTA to prof_dev[148*64], and CTA 0 its per-tile
 * timeline (tools/tc_timeline.py) to the 512 entries behind them: prof_dev holds 148*64 + 512 values.  NULL switches it off. */
int psd_debug_tc_prof(long long *prof_dev);

#ifdef __cplusplus
}
#endif
#endif /* PSD_B200_H_ */
