// sinkhorn.cu -- debiased Sinkhorn divergence between point clouds of any sizes (DESIGN.md §4.10).
//
// Contract: geomloss 0.2.x SamplesLoss("sinkhorn", p=2, blur, scaling, debias=True), tensorized backend, uniform weights,
// evaluated per cloud pair: cost C(u, v) = |u - v|^2 / 2 from direct differences, an epsilon schedule from the diameter of both
// clouds down to blur^2, symmetric (averaged) updates of the four potentials f_ba, f_aa, g_ab, g_bb, one extrapolation step at
// blur^2, and S = <a, f_ba - f_aa> + <b, g_ab - g_bb>.  The gradient is that of the extrapolation step with its inputs held
// constant (geomloss .detach()s them), fused into that step.
//
// One launch per call.  Cloud pair c belongs to a cluster of S CTAs (S in {1, 2, 4, 8}).  Every CTA derives the bounding box,
// the diameter and the whole epsilon schedule itself (a min / max reduction is exact, so the CTAs agree bit for bit), then
// takes a fixed slice of the x-queries and of the y-queries.  A round stages the target clouds through shared memory in index
// order and every query thread reduces its two softmins over all targets in that order, so a query's arithmetic does not depend
// on S.  The four potentials of a cloud live in a stream-ordered global workspace, two buffers of 2n + 2m floats (L2
// resident): a round reads the old buffer through L2 and writes the new one, so the averaging fuses into the softmin, and one
// cluster barrier (release / acquire) separates rounds.  No float atomics: rank 0 sums S in fp64 in a fixed order.
//
// Ragged and weighted batches (sinkhorn_kernel<GRAD, true>, psd_sinkhorn_divergence_weighted): pair c takes part with its first
// x_len[c] / y_len[c] points and point weights x_w / y_w (geomloss's SamplesLoss(...)(a, x, b, y)).  The lengths replace n and m
// everywhere a pair's arithmetic uses them; the arrays keep their padded strides.  A weight enters as logf(w) in the staged h
// and as w in the gradient and S; a group of 8 targets of weight 0 is skipped.  With NULL weights a pair gives the bits of the
// uniform kernel on its points alone, and sinkhorn_kernel<GRAD, false> compiles to the code it had before the variant existed.
#include <cooperative_groups.h>
#include <math.h>

#include <type_traits>

#include "psd_common.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int kSkThreads = 256;
constexpr int kSkTile = 512;        // targets staged per tile
constexpr int kSkGroup = 8;         // targets per running-max update
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kHalfLog2e = 0.7213475204444817f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr long long kSkMaxLoopEps = 1 << 30;
constexpr float kSkMinEps = 0x1p-128f;  // the least eps for which kHalfLog2e / eps is finite, to a power of 2

struct SkParams {
    const float *x, *y;
    int b, n, m;
    float blur, scaling;
    float *loss, *grad_x, *grad_y, *pot;
    int *rounds;
    float *ws;                      // [b][2][2n + 2m]
};

// The ragged variant's parameters: participating points and point weights (NULL: n / m, uniform).
struct SkRaggedParams : SkParams {
    const int *x_len, *y_len;       // [b]
    const float *x_w, *y_w;         // [b][n] / [b][m]
};

__device__ __forceinline__ float ex2(float v) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}

// Running log-sum-exp in base 2 of one query over one target cloud: sum_j 2^(z_j - M) with M the running maximum (w: the
// same weights times (q - t_j), the gradient's transport term).
struct Lse {
    float M, s, wx, wy, wz;
};

// epsilon of round t (0 = init at eps_list[0], 1..K = eps_list[t-1], K + 1 = extrapolation at blur^2), K = L + 2: computed in
// double, rounded to fp32, and raised to at least kSkMinEps.  Below it kk = kHalfLog2e / eps overflows and a query's own
// target gives fma(-0, inf, h) = NaN; only D < 5.4e-20 (eps_list[0] = D^2) or blur < 5.4e-20 reach it.  For a tiny D the
// raised rounds are those at D^2, whose potentials (of order D^2) vanish against blur^2 in the later rounds' h.
__device__ __forceinline__ float eps_of_round(int t, long long L, double D, double lnD2, double lnS2, float blur) {
    const long long i = t == 0 ? 0 : t - 1;             // index into eps_list
    double e;
    if (i == 0) e = D * D;
    else if (i <= L) e = exp(lnD2 + (double)(i - 1) * lnS2);
    else e = (double)blur * (double)blur;
    return fmaxf((float)e, kSkMinEps);
}

// SKIP: leave out a group whose z are all -inf (targets of weight 0).  It adds nothing to s or w, and while M is still -inf
// its rescale would be ex2(-inf - (-inf)) = NaN.
template <bool GRAD, bool SKIP>
__device__ __forceinline__ void lse_tile(Lse &a, const float4 *tt, int cnt8, float qx, float qy, float qz, float kk) {
    for (int k = 0; k < cnt8; k += kSkGroup) {
        float z[kSkGroup], dx[kSkGroup], dy[kSkGroup], dz[kSkGroup];
#pragma unroll
        for (int u = 0; u < kSkGroup; ++u) {
            const float4 t = tt[k + u];
            dx[u] = __fsub_rn(qx, t.x);
            dy[u] = __fsub_rn(qy, t.y);
            dz[u] = __fsub_rn(qz, t.z);
            z[u] = __fmaf_rn(-psd::sqdist_exact(dx[u], dy[u], dz[u]), kk, t.w);
        }
        const float zm = fmaxf(fmaxf(fmaxf(z[0], z[1]), fmaxf(z[2], z[3])), fmaxf(fmaxf(z[4], z[5]), fmaxf(z[6], z[7])));
        if (SKIP && zm == -INFINITY) continue;
        if (zm > a.M) {
            const float f = ex2(__fsub_rn(a.M, zm));     // 0 when M is still -inf
            a.s = __fmul_rn(a.s, f);
            if (GRAD) { a.wx = __fmul_rn(a.wx, f); a.wy = __fmul_rn(a.wy, f); a.wz = __fmul_rn(a.wz, f); }
            a.M = zm;
        }
#pragma unroll
        for (int u = 0; u < kSkGroup; ++u) {
            const float e = ex2(__fsub_rn(z[u], a.M));
            a.s = __fadd_rn(a.s, e);
            if (GRAD) {
                a.wx = __fmaf_rn(e, dx[u], a.wx);
                a.wy = __fmaf_rn(e, dy[u], a.wy);
                a.wz = __fmaf_rn(e, dz[u], a.wz);
            }
        }
    }
}

// Ragged variant: writes v to the gradient rows and potential entries [lo, hi) of one side of a pair (padded strides), spread
// over the threads of the cluster.
__device__ __forceinline__ void fill_rows(const SkParams &p, int cloud, bool is_x, int lo, int hi, int rank, int S, float v) {
    const int n = p.n, m = p.m, N = is_x ? n : m;
    float *g = is_x ? p.grad_x : p.grad_y;
    float *pp = p.pot ? p.pot + (size_t)cloud * (2 * (size_t)n + 2 * (size_t)m) + (is_x ? 0 : 2 * (size_t)n) : nullptr;
    for (int i = lo + rank * kSkThreads + (int)threadIdx.x; i < hi; i += S * kSkThreads) {
        if (g) {
            float *gp = g + ((size_t)cloud * N + i) * 3;
            gp[0] = v; gp[1] = v; gp[2] = v;
        }
        if (pp) { pp[i] = v; pp[N + i] = v; }
    }
}

// One cloud pair.  RAGGED: pair c takes part with its first nc = x_len[c] points of x and mc = y_len[c] points of y, with
// weights x_w / y_w (log w per target in h, a_i in the gradient and in S); rows beyond the lengths are written as 0.  A length
// outside [1, n] / [1, m], a participating weight that is negative or not finite, or a side whose participating weights are all
// 0 makes the pair NaN, as a non-finite coordinate does.  Every array keeps its padded stride n / m.
template <bool GRAD, bool RAGGED>
__global__ void __launch_bounds__(kSkThreads) sinkhorn_kernel(std::conditional_t<RAGGED, SkRaggedParams, SkParams> p) {
    cg::cluster_group cluster = cg::this_cluster();
    const int S = (int)cluster.num_blocks();
    const int rank = (int)cluster.block_rank();
    const int cloud = blockIdx.x / S;
    const int tid = threadIdx.x;
    const int n = p.n, m = p.m;
    const float *X = p.x + (size_t)cloud * n * 3;
    const float *Y = p.y + (size_t)cloud * m * 3;
    const size_t stride = 2 * (size_t)n + 2 * (size_t)m;
    int nc = n, mc = m;
    bool len_ok = true;
    const float *XW = nullptr, *YW = nullptr;
    if constexpr (RAGGED) {
        if (p.x_len) nc = p.x_len[cloud];
        if (p.y_len) mc = p.y_len[cloud];
        len_ok = nc >= 1 && nc <= n && mc >= 1 && mc <= m;
        if (!len_ok) nc = mc = 0;      // read no point
        if (p.x_w) XW = p.x_w + (size_t)cloud * n;
        if (p.y_w) YW = p.y_w + (size_t)cloud * m;
    }

    __shared__ float4 tA[kSkTile];    // targets with the h of the x-queries
    __shared__ float4 tB[kSkTile];    // targets with the h of the y-queries
    __shared__ float red[6][kSkThreads / 32];
    __shared__ int bad_any;
    __shared__ double dred[kSkThreads];

    // ---- bounding box of both clouds, and whether any coordinate is not finite
    if (tid == 0) bad_any = 0;
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    int bad = 0;
    for (int k = tid; k < nc + mc; k += kSkThreads) {
        const float *pt = k < nc ? X + 3 * (size_t)k : Y + 3 * (size_t)(k - nc);
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float v = pt[a];
            bad |= !isfinite(v);
            lo[a] = fminf(lo[a], v);
            hi[a] = fmaxf(hi[a], v);
        }
        if constexpr (RAGGED) {      // bit 0: invalid; bits 1 / 2: a positive weight in x / y
            const float *W = k < nc ? XW : YW;
            const float w = W ? W[k < nc ? k : k - nc] : 1.f;
            if (!(w >= 0.f && w <= 3.402823466e38f)) bad |= 1;
            if (w > 0.f) bad |= k < nc ? 2 : 4;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
    }
    __syncthreads();
    if constexpr (RAGGED) {
        if (bad) atomicOr(&bad_any, bad);
    } else {
        if (bad) bad_any = 1;
    }
    if ((tid & 31) == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) { red[a][tid >> 5] = lo[a]; red[3 + a][tid >> 5] = hi[a]; }
    }
    __syncthreads();
    double D2 = 0.0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        float l = red[a][0], h = red[3 + a][0];
        for (int w = 1; w < kSkThreads / 32; ++w) { l = fminf(l, red[a][w]); h = fmaxf(h, red[3 + a][w]); }
        const double e = (double)h - (double)l;
        D2 += e * e;
    }
    const double D = sqrt(D2);
    const bool nonfinite = RAGGED ? !len_ok || bad_any != 6 : bad_any != 0;

    // ---- this CTA's query slices
    const int xs0 = (int)(((long long)rank * nc) / S), xs1 = (int)(((long long)(rank + 1) * nc) / S);
    const int ys0 = (int)(((long long)rank * mc) / S), ys1 = (int)(((long long)(rank + 1) * mc) / S);
    const int Rx = xs1 - xs0, R = Rx + (ys1 - ys0);

    if (nonfinite || D == 0.0) {
        // no schedule: NaN for a cloud pair with a NaN / infinite coordinate, 0 when every point coincides
        const float v = nonfinite ? __int_as_float(0x7fffffff) : 0.f;
        if constexpr (RAGGED) {      // every row, beyond the lengths too
            fill_rows(p, cloud, true, 0, n, rank, S, v);
            fill_rows(p, cloud, false, 0, m, rank, S, v);
        } else {
            for (int r = tid; r < R; r += kSkThreads) {
                const bool is_x = r < Rx;
                const int i = is_x ? xs0 + r : ys0 + (r - Rx);
                float *g = is_x ? p.grad_x : p.grad_y;
                if (g) {
                    float *gp = g + ((size_t)cloud * (is_x ? n : m) + i) * 3;
                    gp[0] = v; gp[1] = v; gp[2] = v;
                }
                if (p.pot) {
                    float *pp = p.pot + (size_t)cloud * stride;
                    if (is_x) { pp[i] = v; pp[n + i] = v; } else { pp[2 * n + i] = v; pp[2 * n + m + i] = v; }
                }
            }
        }
        if (rank == 0 && tid == 0) {
            p.loss[cloud] = v;
            if (p.rounds) p.rounds[cloud] = 0;
        }
        return;
    }

    // ---- schedule: eps_list = [D^2] + exp(arange(2 ln D, 2 ln blur, 2 ln scaling)) + [blur^2], numpy arange length
    const double lnD2 = 2.0 * log(D), lnB2 = 2.0 * log((double)p.blur), lnS2 = 2.0 * log((double)p.scaling);
    const double v = ceil((lnB2 - lnD2) / lnS2);
    const long long L = v > 0.0 ? (v < (double)kSkMaxLoopEps ? (long long)v : kSkMaxLoopEps) : 0;
    const int K = (int)(L + 2);

    const float loga = logf(__fdiv_rn(1.f, (float)nc)), logb = logf(__fdiv_rn(1.f, (float)mc));
    float *ws = p.ws + (size_t)cloud * 2 * stride;
    if constexpr (RAGGED) {
        fill_rows(p, cloud, true, nc, n, rank, S, 0.f);
        fill_rows(p, cloud, false, mc, m, rank, S, 0.f);
    }

    for (int t = 0; t < K + 2; ++t) {
        const float eps = eps_of_round(t, L, D, lnD2, lnS2, p.blur);
        const bool init = t == 0, extrap = t == K + 1;
        const float *old = ws + (size_t)((t + 1) & 1) * stride;
        float *nw = ws + (size_t)(t & 1) * stride;
        const float kk = __fdiv_rn(kHalfLog2e, eps);
        const float neg_eps_ln2 = __fmul_rn(-eps, kLn2);

        for (int c0 = 0; c0 < R; c0 += kSkThreads) {
            const int r = c0 + tid;
            const bool active = r < R;
            const bool is_x = r < Rx;
            const int qi = is_x ? xs0 + r : ys0 + (r - Rx);
            float qx = 0.f, qy = 0.f, qz = 0.f;
            if (active) {
                const float *qp = (is_x ? X : Y) + 3 * (size_t)qi;
                qx = qp[0]; qy = qp[1]; qz = qp[2];
            }
            Lse cross{-INFINITY, 0.f, 0.f, 0.f, 0.f}, self{-INFINITY, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int tc = 0; tc < 2; ++tc) {
                const int Tn = tc == 0 ? mc : nc;
                const float *TP = tc == 0 ? Y : X;     // target cloud of this pass
                const float *TW = tc == 0 ? YW : XW;
                const float logw = tc == 0 ? logb : loga;
                // potential in h of the x-queries / the y-queries: (g_ab, g_bb) against Y, (f_aa, f_ba) against X
                const float *potA = old + (tc == 0 ? 2 * (size_t)n : (size_t)n);
                const float *potB = old + (tc == 0 ? 2 * (size_t)n + m : (size_t)0);
                Lse acc{-INFINITY, 0.f, 0.f, 0.f, 0.f};
                for (int j0 = 0; j0 < Tn; j0 += kSkTile) {
                    const int cnt = min(kSkTile, Tn - j0);
                    const int cnt8 = (cnt + kSkGroup - 1) & ~(kSkGroup - 1);
                    __syncthreads();
                    for (int k = tid; k < cnt8; k += kSkThreads) {
                        const int j = j0 + k;
                        if (k < cnt) {
                            const float *tp = TP + 3 * (size_t)j;
                            const float x0 = tp[0], x1 = tp[1], x2 = tp[2];
                            const float pa = init ? 0.f : __ldcg(potA + j), pb = init ? 0.f : __ldcg(potB + j);
                            const float lw = RAGGED && TW ? logf(TW[j]) : logw;     // -inf for a weight of 0
                            tA[k] = make_float4(x0, x1, x2, __fmul_rn(__fadd_rn(lw, __fdiv_rn(pa, eps)), kLog2e));
                            tB[k] = make_float4(x0, x1, x2, __fmul_rn(__fadd_rn(lw, __fdiv_rn(pb, eps)), kLog2e));
                        } else {
                            tA[k] = make_float4(0.f, 0.f, 0.f, -INFINITY);
                            tB[k] = tA[k];
                        }
                    }
                    __syncthreads();
                    if (active) {
                        // only the extrapolation round carries the gradient sums; M and s take the same steps either way
                        if (GRAD && extrap) lse_tile<true, RAGGED>(acc, is_x ? tA : tB, cnt8, qx, qy, qz, kk);
                        else lse_tile<false, RAGGED>(acc, is_x ? tA : tB, cnt8, qx, qy, qz, kk);
                    }
                }
                // the x-queries' cross softmin is against Y, the y-queries' against X
                if (is_x == (tc == 0)) cross = acc; else self = acc;
            }
            if (active) {
                float fc = __fmul_rn(neg_eps_ln2, __fadd_rn(cross.M, log2f(cross.s)));
                float fs = __fmul_rn(neg_eps_ln2, __fadd_rn(self.M, log2f(self.s)));
                const size_t ic = is_x ? (size_t)qi : 2 * (size_t)n + qi;      // f_ba / g_ab
                const size_t is = is_x ? (size_t)n + qi : 2 * (size_t)n + m + qi; // f_aa / g_bb
                if (!init && !extrap) {
                    fc = __fmul_rn(0.5f, __fadd_rn(__ldcg(old + ic), fc));
                    fs = __fmul_rn(0.5f, __fadd_rn(__ldcg(old + is), fs));
                }
                __stcg(nw + ic, fc);
                __stcg(nw + is, fs);
                if (extrap) {
                    if (p.pot) {
                        float *pp = p.pot + (size_t)cloud * stride;
                        pp[ic] = fc;
                        pp[is] = fs;
                    }
                    if (GRAD) {
                        float *g = is_x ? p.grad_x : p.grad_y;
                        if (g) {
                            const float *QW = is_x ? XW : YW;
                            const float a = RAGGED && QW ? QW[qi] : __fdiv_rn(1.f, (float)(is_x ? nc : mc));
                            float *gp = g + ((size_t)cloud * (is_x ? n : m) + qi) * 3;
                            gp[0] = __fmul_rn(a, __fsub_rn(__fdiv_rn(cross.wx, cross.s), __fdiv_rn(self.wx, self.s)));
                            gp[1] = __fmul_rn(a, __fsub_rn(__fdiv_rn(cross.wy, cross.s), __fdiv_rn(self.wy, self.s)));
                            gp[2] = __fmul_rn(a, __fsub_rn(__fdiv_rn(cross.wz, cross.s), __fdiv_rn(self.wz, self.s)));
                        }
                    }
                }
            }
        }
        cluster.sync();   // this round's potentials visible cluster-wide; every read of the old buffer done
    }

    // ---- S = <a, f_ba - f_aa> + <b, g_ab - g_bb>, fp64 in a fixed order (rank 0)
    if (rank != 0) return;
    const float *fin = ws + (size_t)((K + 1) & 1) * stride;
    double part[2];
#pragma unroll
    for (int side = 0; side < 2; ++side) {
        const int N = side == 0 ? nc : mc;
        const float *pc = fin + (side == 0 ? 0 : 2 * (size_t)n);
        const float *ps = pc + (side == 0 ? n : m);
        const float *W = side == 0 ? XW : YW;
        double acc = 0.0;
        if (RAGGED && W) {
            for (int i = tid; i < N; i += kSkThreads)
                acc = fma((double)W[i], (double)__ldcg(pc + i) - (double)__ldcg(ps + i), acc);
        } else {
            for (int i = tid; i < N; i += kSkThreads) acc += (double)__ldcg(pc + i) - (double)__ldcg(ps + i);
        }
        __syncthreads();
        dred[tid] = acc;
        __syncthreads();
        for (int h = kSkThreads / 2; h > 0; h >>= 1) {
            if (tid < h) dred[tid] += dred[tid + h];
            __syncthreads();
        }
        part[side] = RAGGED && W ? dred[0] : dred[0] / (double)N;
    }
    if (tid == 0) {
        p.loss[cloud] = (float)(part[0] + part[1]);
        if (p.rounds) p.rounds[cloud] = K;
    }
}

}  // namespace

// Grid: b clusters of S CTAs.  force_cluster: 0 = automatic (as psd_launch_emd_forward: the largest S <= 8 with b * S CTAs
// within the SM count), 1 / 2 / 4 / 8 = that size (test hook).  Returns cudaErrorInvalidValue for another size.  ragged: the
// variant that reads x_len / y_len / x_w / y_w (each may be NULL); otherwise they are ignored.
cudaError_t psd_launch_sinkhorn(const float *x, const float *y, int b, int n, int m, bool ragged, const int *x_len,
                                const int *y_len, const float *x_w, const float *y_w, float blur, float scaling, float *loss,
                                float *grad_x, float *grad_y, float *potentials, int *rounds, int force_cluster,
                                cudaStream_t stream) {
    if (b <= 0) return cudaSuccess;
    int S = 1;
    if (force_cluster != 0) {
        S = force_cluster;
        if (S != 1 && S != 2 && S != 4 && S != 8) return cudaErrorInvalidValue;
    } else {
        int dev = 0, num_sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
        while (S < 8 && b * (S * 2) <= num_sms) S *= 2;
    }
    SkRaggedParams p;
    p.x = x; p.y = y; p.b = b; p.n = n; p.m = m; p.blur = blur; p.scaling = scaling;
    p.loss = loss; p.grad_x = grad_x; p.grad_y = grad_y; p.pot = potentials; p.rounds = rounds;
    p.x_len = x_len; p.y_len = y_len; p.x_w = x_w; p.y_w = y_w;
    const size_t ws_floats = (size_t)b * 2 * (2 * (size_t)n + 2 * (size_t)m);
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(&p.ws), sizeof(float) * ws_floats, stream);
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned int)(b * S));
    cfg.blockDim = dim3(kSkThreads);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned int)S;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const bool grad = grad_x || grad_y;
    if (ragged) e = cudaLaunchKernelEx(&cfg, grad ? sinkhorn_kernel<true, true> : sinkhorn_kernel<false, true>, p);
    else e = cudaLaunchKernelEx(&cfg, grad ? sinkhorn_kernel<true, false> : sinkhorn_kernel<false, false>, SkParams(p));
    const cudaError_t e2 = cudaFreeAsync(p.ws, stream);
    return e != cudaSuccess ? e : e2;
}
