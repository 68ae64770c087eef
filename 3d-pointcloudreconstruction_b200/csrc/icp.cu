// icp.cu -- batched point-to-point ICP alignment (utils/icp.py:4-118), the eval-time caller of the 1-NN query
// (testnet.py:57-64, test_pix3d.py:60-64: one icp() per sample, tolerance 1e-10, up to 1024 iterations).
//
// The reference runs, per sample and per iteration, an sklearn KD-tree build + query on the CPU, numpy means / a 3x3 SVD,
// and a 4xN matrix product.  Here ONE launch aligns the whole batch: one CTA per sample keeps the destination cloud and the
// moving source cloud in shared memory (fp64 SoA) and iterates on-chip until its own convergence test fires:
//     NN (utils/icp.py:49-65)            fp64 brute force, d2 = (dx*dx + dy*dy) + dz*dz without contraction (what the KD-tree's
//                                         reduced distance evaluates), strict '<' in target order, distances = sqrt(d2)
//     best_fit_transform (:4-46)         centroids and H = AA^T BB by deterministic block reductions, R = V U^T by a one-sided
//                                         Jacobi SVD in one thread; the reflection rule (:33-35, last row of Vt negated when
//                                         det R < 0) is the proper-rotation completion u3 = u1 x u2, v3 = v1 x v2
//     src = T src, mean error, |prev - mean| < tolerance -> break (:103-110), final T = best_fit_transform(A, src) (:113)
// All arithmetic is fp64 like numpy's; inputs are fp32 (what the callers pass; the conversion is exact) or fp64.
// Ragged batches (psd_icp_batch_ragged): sample s aligns its first len_a[s] source points to its first len_b[s] destination
// points (any two sizes, as the reference's icp() allows without its shape assert); the uniform instantiations are unchanged.
#include <type_traits>

#include "psd_common.cuh"

namespace psd {

constexpr int kIcpThreads = 512;
constexpr int kIcpMaxN = 4096;     // 6 fp64 arrays of n in shared memory

struct IcpParams {
    const void *a, *b;        // [batch, n, 3] fp32 or fp64
    int in_f64;
    const double *init_pose;  // optional 4x4 (row-major, last row 0 0 0 1), applied to every sample's source
    int batch, n, max_iter;
    double tol;
    double *T;                // [batch, 4, 4]
    double *dist;             // [batch, n] distances of the last NN pass (may be null)
    int *iters;               // [batch] the reference's `i` (may be null)
};

// a, dist: [batch, n, *] and b: [batch, m, 3] padded; a sample takes part with its first len_a / len_b points
struct IcpRaggedParams : IcpParams {
    int m;                    // padded destination size
    const int *len_a, *len_b; // [batch] device (NULL = n / m)
};

__device__ __forceinline__ double ld_coord(const void *p, int f64, long long i) {
    return f64 ? reinterpret_cast<const double *>(p)[i] : (double)reinterpret_cast<const float *>(p)[i];
}

// sum of K per-thread doubles over the CTA, fixed order (lanes by shuffle tree, then warps 0..31 serially): every thread
// gets the totals in out[0..K)
template <int K>
__device__ __forceinline__ void block_sum(double (&v)[K], double *red, double *out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double x = v[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) red[warp * K + k] = x;
    }
    __syncthreads();
    if (threadIdx.x < K) {
        double s = 0.0;
        for (int w = 0; w < kIcpThreads / 32; ++w) s += red[w * K + threadIdx.x];
        out[threadIdx.x] = s;
    }
    __syncthreads();
}

__device__ __forceinline__ void cross3(const double *a, const double *b, double *c) {
    c[0] = a[1] * b[2] - a[2] * b[1];
    c[1] = a[2] * b[0] - a[0] * b[2];
    c[2] = a[0] * b[1] - a[1] * b[0];
}

// unit vector orthogonal to the unit vector u (for rank-deficient H, where numpy's answer is arbitrary as well)
__device__ void any_orthogonal(const double *u, double *o) {
    int ax = 0;
    if (fabs(u[1]) < fabs(u[ax])) ax = 1;
    if (fabs(u[2]) < fabs(u[ax])) ax = 2;
    double e[3] = {0.0, 0.0, 0.0};
    e[ax] = 1.0;
    const double d = u[ax];
    double nrm = 0.0;
    for (int i = 0; i < 3; ++i) { o[i] = e[i] - d * u[i]; nrm += o[i] * o[i]; }
    nrm = rsqrt(nrm);
    for (int i = 0; i < 3; ++i) o[i] *= nrm;
}

// R = V U^T for H = U S V^T (row-major 3x3), as a proper rotation (utils/icp.py:29-35).
__device__ void kabsch3(const double *H, double *R) {
    double g[3][3], v[3][3];   // g[c] = column c of H V, v[c] = column c of V
    for (int c = 0; c < 3; ++c)
        for (int r = 0; r < 3; ++r) { g[c][r] = H[r * 3 + c]; v[c][r] = (r == c) ? 1.0 : 0.0; }
    for (int sweep = 0; sweep < 40; ++sweep) {
        bool rotated = false;
        for (int p = 0; p < 2; ++p)
            for (int q = p + 1; q < 3; ++q) {
                double al = 0.0, be = 0.0, ga = 0.0;
                for (int r = 0; r < 3; ++r) { al += g[p][r] * g[p][r]; be += g[q][r] * g[q][r]; ga += g[p][r] * g[q][r]; }
                if (ga == 0.0 || fabs(ga) <= 1e-17 * sqrt(al * be)) continue;
                rotated = true;
                const double zeta = (be - al) / (2.0 * ga);
                const double t = copysign(1.0, zeta) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
                for (int r = 0; r < 3; ++r) {
                    const double gp = g[p][r], gq = g[q][r];
                    g[p][r] = c * gp - s * gq; g[q][r] = s * gp + c * gq;
                    const double vp = v[p][r], vq = v[q][r];
                    v[p][r] = c * vp - s * vq; v[q][r] = s * vp + c * vq;
                }
            }
        if (!rotated) break;
    }
    double sg[3];
    for (int c = 0; c < 3; ++c) sg[c] = g[c][0] * g[c][0] + g[c][1] * g[c][1] + g[c][2] * g[c][2];
    int i0 = 0;
    if (sg[1] > sg[i0]) i0 = 1;
    if (sg[2] > sg[i0]) i0 = 2;
    int i1 = (i0 + 1) % 3, i2 = (i0 + 2) % 3;
    if (sg[i2] > sg[i1]) { const int t = i1; i1 = i2; i2 = t; }
    for (int i = 0; i < 9; ++i) R[i] = (i % 4 == 0) ? 1.0 : 0.0;
    if (!(sg[i0] > 0.0)) return;                        // H = 0: identity
    double u1[3], u2[3], u3[3], v1[3], v2[3], v3[3];
    const double n1 = rsqrt(sg[i0]);
    for (int r = 0; r < 3; ++r) { u1[r] = g[i0][r] * n1; v1[r] = v[i0][r]; }
    if (sg[i1] > 1e-30 * sg[i0]) {
        double d = 0.0, nn = 0.0;
        for (int r = 0; r < 3; ++r) d += g[i1][r] * u1[r];
        for (int r = 0; r < 3; ++r) { u2[r] = g[i1][r] - d * u1[r]; nn += u2[r] * u2[r]; }
        nn = rsqrt(nn);
        for (int r = 0; r < 3; ++r) { u2[r] *= nn; v2[r] = v[i1][r]; }
    } else {                                            // rank 1: the rotation about u1 is not determined
        any_orthogonal(u1, u2);
        any_orthogonal(v1, v2);
    }
    cross3(u1, u2, u3);
    cross3(v1, v2, v3);
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) R[r * 3 + c] = v1[r] * u1[c] + v2[r] * u2[c] + v3[r] * u3[c];
}

// T (4x4 row-major) from the sums of one correspondence set: sa = sum A, sb = sum B, hs = sum (A - cA)(B - cB)^T
__device__ void transform_from_sums(const double *cA, const double *cB, const double *H, double *T) {
    double R[9];
    kabsch3(H, R);
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) T[r * 4 + c] = R[r * 3 + c];
        T[r * 4 + 3] = cB[r] - (R[r * 3 + 0] * cA[0] + R[r * 3 + 1] * cA[1] + R[r * 3 + 2] * cA[2]);
    }
    T[12] = 0.0; T[13] = 0.0; T[14] = 0.0; T[15] = 1.0;
}

// the sample's source / destination point counts and the padded destination size
__device__ __forceinline__ int src_count(const IcpParams &p, int) { return p.n; }
__device__ __forceinline__ int dst_count(const IcpParams &p, int) { return p.n; }
__device__ __forceinline__ int dst_stride(const IcpParams &p) { return p.n; }
__device__ __forceinline__ int src_count(const IcpRaggedParams &p, int s) { return p.len_a ? p.len_a[s] : p.n; }
__device__ __forceinline__ int dst_count(const IcpRaggedParams &p, int s) { return p.len_b ? p.len_b[s] : p.m; }
__device__ __forceinline__ int dst_stride(const IcpRaggedParams &p) { return p.m; }

// Q = source points per thread (n <= Q * 512).  RAGGED (IcpRaggedParams): n below is the sample's own source count and nb its
// destination count; Q still comes from the padded n, so thread tid owns the points tid + r*512 in the same order as in a
// uniform launch on the sample alone, and the slots beyond the count are skipped as there: the results are its bits.
template <int Q, bool RAGGED>
__global__ void __launch_bounds__(kIcpThreads, 1) icp_kernel(const std::conditional_t<RAGGED, IcpRaggedParams, IcpParams> p) {
    extern __shared__ double smd[];
    const int sample = blockIdx.x;
    const int n = src_count(p, sample), nb = dst_count(p, sample), tid = threadIdx.x;
    if constexpr (RAGGED) {
        if (!(n >= 1 && n <= p.n && nb >= 1 && nb <= p.m)) {   // invalid lengths: NaN, -1, none of the points read
            const double qnan = __longlong_as_double(0x7ff8000000000000LL);
            if (tid < 16) p.T[(long long)sample * 16 + tid] = qnan;
            if (p.dist)
                for (int j = tid; j < p.n; j += kIcpThreads) p.dist[(long long)sample * p.n + j] = qnan;
            if (p.iters && tid == 0) p.iters[sample] = -1;
            return;
        }
    }
    double *sx = smd, *sy = sx + n, *sz = sy + n, *tx = sz + n, *ty = tx + nb, *tz = ty + nb;
    double *red = tz + nb;           // 16 warps * 9 (sized for 32)
    double *tot = red + 32 * 9;      // 9 totals
    double *sT = tot + 9;            // 12 + flag
    const long long base = (long long)sample * p.n * 3, bbase = (long long)sample * dst_stride(p) * 3;

    for (int j = tid; j < (RAGGED ? max(n, nb) : n); j += kIcpThreads) {
        if (!RAGGED || j < n) {
            double x = ld_coord(p.a, p.in_f64, base + 3 * j), y = ld_coord(p.a, p.in_f64, base + 3 * j + 1),
                   z = ld_coord(p.a, p.in_f64, base + 3 * j + 2);
            if (p.init_pose && p.max_iter > 0) {
                const double *P = p.init_pose;
                const double nx = P[0] * x + P[1] * y + P[2] * z + P[3], ny = P[4] * x + P[5] * y + P[6] * z + P[7],
                             nz = P[8] * x + P[9] * y + P[10] * z + P[11];
                x = nx; y = ny; z = nz;
            }
            sx[j] = x; sy[j] = y; sz[j] = z;
        }
        if (!RAGGED || j < nb) {
            tx[j] = ld_coord(p.b, p.in_f64, bbase + 3 * j);
            ty[j] = ld_coord(p.b, p.in_f64, bbase + 3 * j + 1);
            tz[j] = ld_coord(p.b, p.in_f64, bbase + 3 * j + 2);
        }
    }
    __syncthreads();

    double best[Q];
    int bidx[Q];
#pragma unroll
    for (int r = 0; r < Q; ++r) { best[r] = 0.0; bidx[r] = 0; }
    double prev_error = 0.0;
    int it_out = 0;
    const double inv_n = 1.0 / (double)n;

    for (int it = 0; it < p.max_iter; ++it) {
        it_out = it;
        // ---- nearest neighbour of every source point in the destination cloud: each destination point is read from shared
        // memory once per thread and tested against the thread's Q source points
        {
            double qx[Q], qy[Q], qz[Q], bd[Q];
#pragma unroll
            for (int r = 0; r < Q; ++r) {
                const int j = min(tid + r * kIcpThreads, n - 1);
                qx[r] = sx[j]; qy[r] = sy[j]; qz[r] = sz[j];
                bd[r] = __longlong_as_double(0x7ff0000000000000LL);
                bidx[r] = 0;
            }
#pragma unroll 2
            for (int k = 0; k < nb; ++k) {
                const double kx = tx[k], ky = ty[k], kz = tz[k];
#pragma unroll
                for (int r = 0; r < Q; ++r) {
                    const double dx = kx - qx[r], dy = ky - qy[r], dz = kz - qz[r];
                    const double d = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
                    if (d < bd[r]) { bd[r] = d; bidx[r] = k; }
                }
            }
#pragma unroll
            for (int r = 0; r < Q; ++r) best[r] = sqrt(bd[r]);
        }
        // ---- centroids and mean error
        double s7[7] = {0, 0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int r = 0; r < Q; ++r) {
            const int j = tid + r * kIcpThreads;
            if (j >= n) continue;
            const int k = bidx[r];
            s7[0] += sx[j]; s7[1] += sy[j]; s7[2] += sz[j];
            s7[3] += tx[k]; s7[4] += ty[k]; s7[5] += tz[k];
            s7[6] += best[r];
        }
        block_sum<7>(s7, red, tot);
        const double cA[3] = {tot[0] * inv_n, tot[1] * inv_n, tot[2] * inv_n};
        const double cB[3] = {tot[3] * inv_n, tot[4] * inv_n, tot[5] * inv_n};
        const double mean_error = tot[6] * inv_n;
        // ---- H = AA^T BB
        double h9[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int r = 0; r < Q; ++r) {
            const int j = tid + r * kIcpThreads;
            if (j >= n) continue;
            const int k = bidx[r];
            const double ax = sx[j] - cA[0], ay = sy[j] - cA[1], az = sz[j] - cA[2];
            const double bx = tx[k] - cB[0], by = ty[k] - cB[1], bz = tz[k] - cB[2];
            h9[0] += ax * bx; h9[1] += ax * by; h9[2] += ax * bz;
            h9[3] += ay * bx; h9[4] += ay * by; h9[5] += ay * bz;
            h9[6] += az * bx; h9[7] += az * by; h9[8] += az * bz;
        }
        block_sum<9>(h9, red, tot);
        if (tid == 0) {
            double T[16];
            transform_from_sums(cA, cB, tot, T);
            for (int i = 0; i < 12; ++i) sT[i] = T[i];
        }
        __syncthreads();
        // ---- src = T src
        for (int j = tid; j < n; j += kIcpThreads) {
            const double x = sx[j], y = sy[j], z = sz[j];
            sx[j] = sT[0] * x + sT[1] * y + sT[2] * z + sT[3];
            sy[j] = sT[4] * x + sT[5] * y + sT[6] * z + sT[7];
            sz[j] = sT[8] * x + sT[9] * y + sT[10] * z + sT[11];
        }
        __syncthreads();
        if (fabs(prev_error - mean_error) < p.tol) break;   // uniform: every thread holds the same totals
        prev_error = mean_error;
    }

    if (p.dist && p.max_iter > 0) {
#pragma unroll
        for (int r = 0; r < Q; ++r) {
            const int j = tid + r * kIcpThreads;
            if constexpr (RAGGED) {
                if (j < p.n) p.dist[(long long)sample * p.n + j] = j < n ? best[r] : 0.0;
            } else {
                if (j < n) p.dist[(long long)sample * n + j] = best[r];
            }
        }
    }
    if (p.iters && tid == 0) p.iters[sample] = it_out;

    // ---- final transform: best_fit_transform(A, src) (utils/icp.py:113); with max_iter == 0 this is the plain
    // best_fit_transform(A, B) of the two given clouds
    const double *fx = p.max_iter > 0 ? sx : tx, *fy = p.max_iter > 0 ? sy : ty, *fz = p.max_iter > 0 ? sz : tz;
    // icp() hands the caller's own array A to this last call: when that is float32 (testnet.py:57-63), numpy forms
    // centroid_A and AA = A - centroid_A in float32 (np.mean over axis 0 adds row after row), and only the product with the
    // float64 BB is double.  Reproduced here so that T agrees to rounding, not to 1e-7.
    const bool a_f32 = !p.in_f64 && p.max_iter > 0;
    float *cA32 = reinterpret_cast<float *>(sT + 12);
    if (a_f32 && tid < 3) {
        const float *af = reinterpret_cast<const float *>(p.a) + base + tid;
        float s = 0.f;
#pragma unroll 8
        for (int j = 0; j < n; ++j) s = __fadd_rn(s, af[3 * j]);
        cA32[tid] = __fdiv_rn(s, (float)n);
    }
    double s6[6] = {0, 0, 0, 0, 0, 0};
    for (int j = tid; j < n; j += kIcpThreads) {
        s6[0] += ld_coord(p.a, p.in_f64, base + 3 * j); s6[1] += ld_coord(p.a, p.in_f64, base + 3 * j + 1);
        s6[2] += ld_coord(p.a, p.in_f64, base + 3 * j + 2);
        s6[3] += fx[j]; s6[4] += fy[j]; s6[5] += fz[j];
    }
    block_sum<6>(s6, red, tot);
    double cA[3] = {tot[0] * inv_n, tot[1] * inv_n, tot[2] * inv_n};
    if (a_f32) { cA[0] = (double)cA32[0]; cA[1] = (double)cA32[1]; cA[2] = (double)cA32[2]; }
    const double cB[3] = {tot[3] * inv_n, tot[4] * inv_n, tot[5] * inv_n};
    double h9[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int j = tid; j < n; j += kIcpThreads) {
        double ax, ay, az;
        if (a_f32) {
            const float *af = reinterpret_cast<const float *>(p.a) + base + 3 * j;
            ax = (double)__fsub_rn(af[0], cA32[0]); ay = (double)__fsub_rn(af[1], cA32[1]); az = (double)__fsub_rn(af[2], cA32[2]);
        } else {
            ax = ld_coord(p.a, p.in_f64, base + 3 * j) - cA[0]; ay = ld_coord(p.a, p.in_f64, base + 3 * j + 1) - cA[1];
            az = ld_coord(p.a, p.in_f64, base + 3 * j + 2) - cA[2];
        }
        const double bx = fx[j] - cB[0], by = fy[j] - cB[1], bz = fz[j] - cB[2];
        h9[0] += ax * bx; h9[1] += ax * by; h9[2] += ax * bz;
        h9[3] += ay * bx; h9[4] += ay * by; h9[5] += ay * bz;
        h9[6] += az * bx; h9[7] += az * by; h9[8] += az * bz;
    }
    block_sum<9>(h9, red, tot);
    if (tid == 0) {
        double T[16];
        transform_from_sums(cA, cB, tot, T);
        for (int i = 0; i < 16; ++i) p.T[(long long)sample * 16 + i] = T[i];
    }
}

// nearest_neighbor(src, dst) on its own (utils/icp.py:49-65): one CTA = (sample, 256 source points), destination in smem
__global__ void __launch_bounds__(256) nn_f64_kernel(const void *src, const void *dst, int in_f64, int n_src, int n_dst,
                                                     double *distances, int *indices) {
    extern __shared__ double smd[];
    double *tx = smd, *ty = tx + n_dst, *tz = ty + n_dst;
    const int qblocks = (n_src + 255) / 256;
    const int sample = blockIdx.x / qblocks;
    const int j = (blockIdx.x - sample * qblocks) * 256 + threadIdx.x;
    const long long tb = (long long)sample * n_dst * 3, sb = (long long)sample * n_src * 3;
    for (int k = threadIdx.x; k < n_dst; k += 256) {
        tx[k] = ld_coord(dst, in_f64, tb + 3 * k); ty[k] = ld_coord(dst, in_f64, tb + 3 * k + 1);
        tz[k] = ld_coord(dst, in_f64, tb + 3 * k + 2);
    }
    __syncthreads();
    if (j >= n_src) return;
    const double qx = ld_coord(src, in_f64, sb + 3 * j), qy = ld_coord(src, in_f64, sb + 3 * j + 1),
                 qz = ld_coord(src, in_f64, sb + 3 * j + 2);
    double bd = __longlong_as_double(0x7ff0000000000000LL);
    int bi = 0;
#pragma unroll 4
    for (int k = 0; k < n_dst; ++k) {
        const double dx = tx[k] - qx, dy = ty[k] - qy, dz = tz[k] - qz;
        const double d = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
        if (d < bd) { bd = d; bi = k; }
    }
    distances[(long long)sample * n_src + j] = sqrt(bd);
    indices[(long long)sample * n_src + j] = bi;
}

}  // namespace psd

cudaError_t psd_launch_icp(const void *a, const void *b, int in_f64, int batch, int n, const double *init_pose, int max_iter,
                           double tol, double *T, double *dist, int *iters, cudaStream_t stream) {
    using namespace psd;
    if (batch <= 0) return cudaSuccess;
    IcpParams p{a, b, in_f64, init_pose, batch, n, max_iter, tol, T, dist, iters};
    const size_t smem = sizeof(double) * ((size_t)6 * n + 32 * 9 + 9 + 16);
    const int q = (n + kIcpThreads - 1) / kIcpThreads;
    void (*kern)(IcpParams) = q <= 1 ? icp_kernel<1, false> : q <= 2 ? icp_kernel<2, false>
                            : q <= 4 ? icp_kernel<4, false> : icp_kernel<8, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<batch, kIcpThreads, smem, stream>>>(p);
    return cudaGetLastError();
}

// n <= 4096 (Q <= 8), n + m <= 8192 (the fp64 SoA clouds take the shared memory of the uniform n = 4096), max_iter >= 1
cudaError_t psd_launch_icp_ragged(const void *a, const void *b, int in_f64, int batch, int n, int m, const int *len_a,
                                  const int *len_b, const double *init_pose, int max_iter, double tol, double *T, double *dist,
                                  int *iters, cudaStream_t stream) {
    using namespace psd;
    if (batch <= 0) return cudaSuccess;
    IcpRaggedParams p;
    static_cast<IcpParams &>(p) = IcpParams{a, b, in_f64, init_pose, batch, n, max_iter, tol, T, dist, iters};
    p.m = m; p.len_a = len_a; p.len_b = len_b;
    const size_t smem = sizeof(double) * ((size_t)3 * (n + m) + 32 * 9 + 9 + 16);
    const int q = (n + kIcpThreads - 1) / kIcpThreads;
    void (*kern)(IcpRaggedParams) = q <= 1 ? icp_kernel<1, true> : q <= 2 ? icp_kernel<2, true>
                                  : q <= 4 ? icp_kernel<4, true> : icp_kernel<8, true>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<batch, kIcpThreads, smem, stream>>>(p);
    return cudaGetLastError();
}

int psd_icp_max_points() { return psd::kIcpMaxN; }

cudaError_t psd_launch_nn_f64(const void *src, const void *dst, int in_f64, int batch, int n_src, int n_dst, double *distances,
                              int *indices, cudaStream_t stream) {
    using namespace psd;
    if (batch <= 0 || n_src <= 0) return cudaSuccess;
    const size_t smem = sizeof(double) * (size_t)3 * n_dst;
    cudaError_t e = cudaFuncSetAttribute(nn_f64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int qblocks = (n_src + 255) / 256;
    nn_f64_kernel<<<batch * qblocks, 256, smem, stream>>>(src, dst, in_f64, n_src, n_dst, distances, indices);
    return cudaGetLastError();
}
