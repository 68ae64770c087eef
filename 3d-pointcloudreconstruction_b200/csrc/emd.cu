// emd.cu -- B200-native auction EMD (forward) and its gradient.
//
// Replaces metric/emd/emd_cuda.cu of the reference: the host loop of 7 launches per iteration
// (clear, calc_unass_cnt, calc_unass_cnt_sum, calc_unass_idx, Bid, GetMax, Assign :23-215,256-268),
// CalcDist (:217-226) and NmDistanceGradKernel (:284-300) become ONE persistent launch (+1 for the
// gradient).  Clouds are independent, so the synchronisation scope is one cloud, not the grid: a cloud is
// owned by a thread-block CLUSTER of S CTAs (S = 1,2,4,8 chosen so that B*S fills the 148 SMs) whose
// per-cloud auction state lives in (distributed) shared memory for the whole run:
//   replicated in every CTA : object coordinates xyz2 (SoA) and prices          (read in the O(u*n) scan)
//   sliced by object owner  : max_increments, winner (the reference's max_idx), assignment_inv
//   sliced by bidder home   : assignment, bid, bid_increments, the compacted bidder list
// Per iteration: compact own unassigned points -> scan ALL objects for the own bidders (best / second-best
// value, exact reference arithmetic) -> float atomicMax into the object owner's max_increments over DSMEM
// -> cluster.sync -> winner = atomicMin(bidder index) among bidders within +-1e-6 of the maximum
// -> cluster.sync -> winners commit: evict previous owner, broadcast the new price to every replica
// -> cluster.sync.  The run stops early once no cloud point is unassigned (remaining iterations are no-ops).
//
// Arithmetic follows the reference bit for bit (SURVEY.md 8a E6-E9):
//   s = fma(dz,dz, fma(dx,dx, rn(dy*dy))), d* = xyz2 - xyz1;  v = (float)(3.0 - (double)sqrtf(s) - (double)price)
//   best: strict '>' in index order (lowest index wins ties), better: second best with multiplicity,
//   both from -1e9;  increment = (best - better) + eps  (two fp32 roundings).
// The only filter is a distance cut-off that is provably result-neutral: an object can change
// (best, better) only if v > better, which requires sqrt(s) < 3 - better + 2e-6 (prices are >= 0).
#include <cooperative_groups.h>
#include <limits.h>
#include <stdlib.h>

#include <atomic>

#include "psd_common.cuh"

namespace cg = cooperative_groups;

#ifndef PSD_EMD_RHS_FMA
#define PSD_EMD_RHS_FMA 1     // pass 2 of the two-pass bound scan: the per-object threshold as one fma (0: the round-2 form, A/B builds)
#endif

#ifdef PSD_EMD_PROF
// Instrumented A/B build (tools/emd_phase_clocks.py): thread 0 of block 0 stamps clock64 at the phase boundaries of every
// iteration of the cluster-wide loop: [it][0..5] = start, compacted + counts exchanged, bids done, barrier A passed,
// GetMax + barrier B passed, Assign + barrier C passed; [it][6] = bidders of the cluster, [it][7] = 1 for a grid iteration.
__device__ long long g_emd_prof[256 * 8];
extern "C" int psd_debug_emd_prof(long long *host_out) {
    return cudaMemcpyFromSymbol(host_out, g_emd_prof, sizeof(g_emd_prof)) == cudaSuccess ? 1 : 0;
}
#define EMD_STAMP(it_, slot_) do { if (blockIdx.x == 0 && threadIdx.x == 0 && (it_) < 256) g_emd_prof[(it_) * 8 + (slot_)] = clock64(); } while (0)
#define EMD_NOTE(it_, slot_, v_) do { if (blockIdx.x == 0 && threadIdx.x == 0 && (it_) < 256) g_emd_prof[(it_) * 8 + (slot_)] = (v_); } while (0)
#else
#define EMD_STAMP(it_, slot_) do { } while (0)
#define EMD_NOTE(it_, slot_, v_) do { } while (0)
#endif

namespace psd {

constexpr int kEmdThreads = 1024;
constexpr float kNegInit = -1e9f;
constexpr int kGridG = 8;                      // cells per axis of the object grid
constexpr int kGridCells = kGridG * kGridG * kGridG;
constexpr int kSoloMax = 32;   // bidders per cloud at or below which one CTA finishes the auction alone (one warp per bidder)

struct EmdParams {
    const float *xyz1, *xyz2;
    float *dist;
    int *assignment;
    float *price;          // may be NULL
    int *assignment_inv;   // may be NULL
    float *max_increments; // may be NULL
    int *bid;              // may be NULL (written if given)
    float *bid_increments; // may be NULL (written if given)
    int b, n;
    float eps;
    int iters;
    int fresh;  // 1: ignore the caller's state tensors and start from assignment = -1, price = 0
    int solo;   // 1: shared memory holds the solo-mode arrays (see emd_auction_kernel)
    int grid;   // 1: shared memory holds the object grid (cell-sorted copy of the objects)
    int grid_min_u;   // iterations with fewer bidders in the cluster use the full scan (a bidder per warp is latency bound)
    float *gws;       // GLOBAL mode (n too large for shared memory): per-cloud state in global memory, 11 n floats per cloud
    float *loss_sums; // optional [B]: loss_sums[cloud] += sum_j sqrt(dist[cloud, j])  (Loss.get_emd_loss, loss/loss.py:25)
};

// vector loads of four consecutive objects: shared memory (resident mode) or global memory through L2 (GLOBAL mode, where
// the arrays are written by other CTAs of the cluster: ld.global.cg never looks at this SM's L1)
template <bool GLOBAL>
__device__ __forceinline__ float4 ld4(const float *base, unsigned int sbase, int k) {
    float4 v;
    if (GLOBAL) {
        v = __ldcg(reinterpret_cast<const float4 *>(base + k));
    } else {
        asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(sbase + 4u * k));
    }
    return v;
}
template <bool GLOBAL>
__device__ __forceinline__ float ld1(const float *ptr) { return GLOBAL ? __ldcg(ptr) : *ptr; }

// float atomicMax with the reference's semantics (emd_cuda.cu:10-20): CAS loop, `val > old` in float.
__device__ __forceinline__ void atomic_max_float(float *address, float val) {
    if (val >= 0.f) {
        // a non-negative float is larger than another float exactly when its bit pattern is larger as a signed int (negative
        // floats have the sign bit set): one fire-and-forget integer max, same final value as the CAS loop
        atomicMax(reinterpret_cast<int *>(address), __float_as_int(val));
        return;
    }
    int ret = __float_as_int(*reinterpret_cast<volatile float *>(address));
    while (val > __int_as_float(ret)) {
        const int old = ret;
        if ((ret = atomicCAS(reinterpret_cast<int *>(address), old, __float_as_int(val))) == old) break;
    }
}

struct Top2 {
    float best, better;
    int idx;
};

// merge two partial (best, second best with multiplicity, lowest index of best) results
__device__ __forceinline__ void merge_top2(Top2 &a, float ob, float o2, int oi) {
    if (ob > a.best) {
        a.better = fmaxf(a.best, o2);
        a.best = ob;
        a.idx = oi;
    } else if (ob == a.best) {
        a.better = a.best;                      // two copies of the maximum -> second best equals it
        a.idx = (oi >= 0 && (a.idx < 0 || oi < a.idx)) ? oi : a.idx;
    } else {
        a.better = fmaxf(a.better, ob);
    }
}

// monotone map float -> uint32 (no NaN, no -0 among the values it is used for)
__device__ __forceinline__ unsigned int ford(float v) {
    const unsigned int u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float funord(unsigned int o) {
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

// Full-warp merge of 32 partial (best, second best with multiplicity, lowest index of best) results with redux.sync:
// best = max; index = lowest among the lanes holding the max; second best = the max again if two lanes hold it, else the
// largest of (holder's own second best, everybody else's best).  Same function of the multiset as a chain of merge_top2.
__device__ __forceinline__ void warp_top2_redux(Top2 &r) {
    const unsigned int ob = ford(r.best);
    const unsigned int m1 = __reduce_max_sync(0xffffffffu, ob);
    const bool holder = ob == m1;
    const int nh = __popc(__ballot_sync(0xffffffffu, holder));
    const unsigned int idx = __reduce_min_sync(0xffffffffu, holder ? (unsigned int)r.idx : 0xffffffffu);
    const unsigned int second = __reduce_max_sync(0xffffffffu, ford(holder ? r.better : r.best));
    r.best = funord(m1);
    r.idx = (int)idx;
    r.better = nh >= 2 ? r.best : funord(second);
}

// One bidder group's scan of all n objects: thread t of tpb (a power of two) looks at objects t, t + tpb, ... and returns its
// partial (best, second best, index of best); the caller merges the group.
// Scan with deferred value evaluation.  A pair can change the top two only if v > better, i.e.
// sqrt(s) < 3 - better - price <= 3 - better (prices are >= 0): pairs with s above R2 = (3 - better + 2e-6)^2, or
// above (3 - better - price[k] + slack)^2 once the object's price is looked at, are skipped exactly.  The survivors' values
// (IEEE sqrt + fp64 arithmetic, ~30 instructions) used to be evaluated inside the scan, where one surviving lane sends the
// whole warp down the long path (27-60 % of the iterations).  Now a lane queues its survivors (in index order, so the strict
// '>' tie rule is unchanged) and the warp evaluates them together when some lane has two; `better` for the radius is then
// the second best of the whole bidder group inside the warp (a valid lower bound of the final second best), not only the
// lane's own.
template <bool GLOBAL>
__device__ __forceinline__ Top2 scan_bidder(const float *ox, const float *oy, const float *oz, const float *price, int n,
                                            float x1, float y1, float z1, int tpb, int t, bool valid) {
    Top2 r;
    r.best = kNegInit; r.better = kNegInit; r.idx = -1;
    const int wl = tpb < 32 ? tpb : 32;
    float R2 = 3.0e38f, Rg = 3.0e38f;   // squared / plain pruning radius from the group's second best so far
    int qn = 0, qk0 = 0, qk1 = 0;
    float qs0 = 0.f, qs1 = 0.f;
    auto apply = [&](int k, float v) {
        if (v > r.best) {
            r.better = r.best; r.best = v; r.idx = k;
        } else if (v > r.better) {
            r.better = v;
        }
    };
    auto evaluate_queue = [&]() {
        // both values first (two independent sqrt / fp64 chains in flight), then the updates in index order
        const float v0 = (float)(3.0 - (double)__fsqrt_rn(qs0) - (double)ld1<GLOBAL>(price + qk0));
        const float v1 = (float)(3.0 - (double)__fsqrt_rn(qs1) - (double)ld1<GLOBAL>(price + qk1));
        if (qn > 0) apply(qk0, v0);
        if (qn > 1) apply(qk1, v1);
        qn = 0;
    };
    auto flush = [&]() {   // warp-uniform
        evaluate_queue();
        float gb = r.best, g2 = r.better;   // group-wide (best, second best with multiplicity) so far
        for (int o = wl >> 1; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, gb, o);
            const float o2 = __shfl_xor_sync(0xffffffffu, g2, o);
            g2 = fmaxf(fminf(gb, ob), fmaxf(g2, o2));
            gb = fmaxf(gb, ob);
        }
        Rg = 3.0f - g2;
        const float R = Rg + 2e-6f;
        R2 = R * R * 1.000001f;
    };
    // n is a multiple of 1024 and tpb a power of two <= 1024: every lane of the warp runs n / tpb iterations
    auto consider = [&](int k, float s, bool pass) {   // warp-uniform call; `pass` = survived the price-free test
        if (pass) {
            // per-object test with the object's own price: v > better needs sqrt(s) < 3 - better - price[k].  The
            // slack covers the fp32 rounding of this test and of the reference's value (|terms| are O(1): 3 ulp(4)).
            const float pk = ld1<GLOBAL>(price + k);
            const float Rk = (Rg - pk) + (4e-6f + 1e-6f * (fabsf(Rg) + fabsf(pk)));
            if (Rk > 0.f && s <= Rk * Rk * 1.000002f) {
                if (qn == 0) { qk0 = k; qs0 = s; } else { qk1 = k; qs1 = s; }
                ++qn;
            }
        }
        if (__any_sync(0xffffffffu, qn == 2)) flush();
    };
    if (n <= 4 * tpb) {
        // A handful of objects per thread (few bidders, many threads each; a warp belongs to one bidder).  The queue / vote
        // / radius machinery is a long dependent chain here and prunes nothing, and evaluating every value exactly is bound
        // by the fp32<->fp64 conversions (16 lanes per clock).  So: an fp32 estimate a = (3 - sqrt(s)) - price of every
        // value with an error bound delta, the warp's second best LOWER bound g2 (at least two objects have an exact value
        // >= g2, so the group's final second best is >= g2), and the exact evaluation only of objects whose UPPER bound
        // reaches g2 -- nothing else can enter the top two.  Candidates are applied in index order.
        {
            const int k0 = t;   // n / tpb is 1, 2 or 4
            float au[4], sv[4];            // upper bounds of the values, squared distances
            float a1 = kNegInit, a2 = kNegInit;   // this thread's two largest LOWER bounds
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int k = k0 + i * tpb;
                au[i] = kNegInit; sv[i] = 0.f;
                if (k < n && valid) {
                    sv[i] = sqdist_exact(ld1<GLOBAL>(ox + k) - x1, ld1<GLOBAL>(oy + k) - y1, ld1<GLOBAL>(oz + k) - z1);
                    const float pk = ld1<GLOBAL>(price + k);
                    float d;
                    asm("sqrt.approx.f32 %0, %1;" : "=f"(d) : "f"(sv[i]));   // relative error <= 2^-23
                    const float a = (3.0f - d) - pk;
                    // |a - v| <= 2^-23 d + ulp(3 - d)/2 + ulp(a) <= 3.6e-7 (3 + d + |pk|)
                    const float delta = 1e-6f * (3.0f + d + fabsf(pk));
                    const float al = a - delta;
                    au[i] = a + delta;
                    a2 = fmaxf(a2, fminf(a1, al));
                    a1 = fmaxf(a1, al);
                }
            }
            // warp-wide second best (with multiplicity) of the lower bounds: the group's final second best is at least this
            const unsigned int o1 = ford(a1);
            const unsigned int m1 = __reduce_max_sync(0xffffffffu, o1);
            const bool holder = o1 == m1;
            const int nh = __popc(__ballot_sync(0xffffffffu, holder));
            const float g2 = nh >= 2 ? funord(m1) : funord(__reduce_max_sync(0xffffffffu, ford(holder ? a2 : a1)));
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int k = k0 + i * tpb;
                const bool cand = k < n && valid && au[i] >= g2;
                if (__any_sync(0xffffffffu, cand)) {
                    const float v = (float)(3.0 - (double)__fsqrt_rn(sv[i]) - (double)ld1<GLOBAL>(price + (cand ? k : 0)));
                    if (cand) apply(k, v);
                }
            }
        }
        return r;
    }
    if (tpb >= 32 && ((n / tpb) & 3) == 0) {
        // A warp (or several) per bidder, many objects per lane: two passes without any per-step dependency on earlier
        // evaluations.  Pass 1: fp32 bounds of every value (as above) and the warp's second best lower bound g2.  Pass 2: the
        // same sweep again, exact evaluation only of the objects whose upper bound reaches g2 (a handful per warp).  The
        // adaptive-radius scan below is a chain of ~2 k cycles per step for such a warp: the radius of the bidders that are
        // still unassigned late in the auction is large, so most steps took its slow path.
        const unsigned int sx = GLOBAL ? 0u : (unsigned int)__cvta_generic_to_shared(ox), sy = GLOBAL ? 0u : (unsigned int)__cvta_generic_to_shared(oy),
                           sz = GLOBAL ? 0u : (unsigned int)__cvta_generic_to_shared(oz);
        float a1 = kNegInit, a2 = kNegInit;
        auto bounds4 = [&](int k, float (&sv)[4], float (&au)[4], float (&al)[4]) {
            const float4 xa = ld4<GLOBAL>(ox, sx, k), ya = ld4<GLOBAL>(oy, sy, k), za = ld4<GLOBAL>(oz, sz, k);
            const float4 pk = GLOBAL ? __ldcg(reinterpret_cast<const float4 *>(price + k)) : *reinterpret_cast<const float4 *>(price + k);
            const float xs[4] = {xa.x, xa.y, xa.z, xa.w}, ys[4] = {ya.x, ya.y, ya.z, ya.w}, zs[4] = {za.x, za.y, za.z, za.w};
            const float ps[4] = {pk.x, pk.y, pk.z, pk.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                sv[i] = sqdist_exact(xs[i] - x1, ys[i] - y1, zs[i] - z1);
                float d;
                asm("sqrt.approx.f32 %0, %1;" : "=f"(d) : "f"(sv[i]));   // relative error <= 2^-23
                const float a = (3.0f - d) - ps[i];
                const float delta = 1e-6f * (3.0f + d + fabsf(ps[i]));   // |a - v| <= 3.6e-7 (3 + d + |p|)
                al[i] = a - delta;
                au[i] = a + delta;
            }
        };
        // pass 1 on every fourth chunk only: ANY two objects give a valid lower bound of the final second best; a quarter of
        // them gives one that still leaves only a handful of candidates
        for (int k = 4 * t; k < n; k += 16 * tpb) {
            float sv[4], au[4], al[4];
            bounds4(k, sv, au, al);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                a2 = fmaxf(a2, fminf(a1, al[i]));
                a1 = fmaxf(a1, al[i]);
            }
        }
        const unsigned int o1 = ford(a1);
        const unsigned int m1 = __reduce_max_sync(0xffffffffu, o1);
        const bool holder = o1 == m1;
        const int nh = __popc(__ballot_sync(0xffffffffu, holder));
        const float g2 = nh >= 2 ? funord(m1) : funord(__reduce_max_sync(0xffffffffu, ford(holder ? a2 : a1)));
        // pass 2 in the squared domain (no sqrt): v >= g2 needs sqrt(s) <= (3 - g2) - price + delta; delta2 bounds the delta
        // of pass 1 for every object that can pass (d <= |c| + |p| + 1)
        const float c = 3.0f - g2;
        // rhs_k = (c - p_k) + 2e-6 (4 + |c| + 2 |p_k|) as ONE fma per object: prices are >= 0 (they start at 0 and only rise), so
        // rhs_k = cA - (1 - 4e-6) p_k with cA = c + 2e-6 (4 + |c|).  The different rounding (a few ulp of O(1) values, < 3e-7)
        // is far inside the slack, which is twice the bound delta of pass 1 (>= 4e-6 to spare).
        const float cA = c + 2e-6f * (4.0f + fabsf(c));
        const float cB = cA * 1.0000005f, kB = -0.999996f * 1.0000005f;
        for (int k = 4 * t; k < n; k += 4 * tpb) {
            const float4 xa = ld4<GLOBAL>(ox, sx, k), ya = ld4<GLOBAL>(oy, sy, k), za = ld4<GLOBAL>(oz, sz, k);
            const float4 pk = GLOBAL ? __ldcg(reinterpret_cast<const float4 *>(price + k)) : *reinterpret_cast<const float4 *>(price + k);
            const float xs[4] = {xa.x, xa.y, xa.z, xa.w}, ys[4] = {ya.x, ya.y, ya.z, ya.w}, zs[4] = {za.x, za.y, za.z, za.w};
            const float ps[4] = {pk.x, pk.y, pk.z, pk.w};
            float sv[4];
            bool cs[4];
            bool any = false;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                sv[i] = sqdist_exact(xs[i] - x1, ys[i] - y1, zs[i] - z1);
                // (PSD_EMD_RHS_FMA: the factor 1.000001 of the squared threshold is folded into cB / kB: (1.0000005 rhs)^2 >= 1.000001 rhs^2)
                const float rhs = PSD_EMD_RHS_FMA ? __fmaf_rn(kB, ps[i], cB) : (c - ps[i]) + 2e-6f * (4.0f + fabsf(c) + 2.0f * fabsf(ps[i]));
                cs[i] = valid && rhs > 0.f && sv[i] <= (PSD_EMD_RHS_FMA ? rhs * rhs : rhs * rhs * 1.000001f);
                any |= cs[i];
            }
            if (__any_sync(0xffffffffu, any)) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    if (__any_sync(0xffffffffu, cs[i])) {
                        const float v = (float)(3.0 - (double)__fsqrt_rn(sv[i]) - (double)ps[i]);
                        if (cs[i]) apply(k + i, v);
                    }
                }
            }
        }
        return r;
    }
    if (((n / tpb) & 3) == 0) {
        // four CONSECUTIVE objects per lane and step (3 x LDS.128), one vote for the common all-skipped case; a lane still
        // meets its objects in index order, and the group merge breaks ties by the lowest index.  The coordinates never
        // change after the prologue, so they are read through explicit shared-space addresses (no generic -> shared window
        // arithmetic in the loop).
        const unsigned int sx = GLOBAL ? 0u : (unsigned int)__cvta_generic_to_shared(ox), sy = GLOBAL ? 0u : (unsigned int)__cvta_generic_to_shared(oy),
                           sz = GLOBAL ? 0u : (unsigned int)__cvta_generic_to_shared(oz);
        for (int k = 4 * t; k < n; k += 4 * tpb) {
            const float4 xa = ld4<GLOBAL>(ox, sx, k), ya = ld4<GLOBAL>(oy, sy, k), za = ld4<GLOBAL>(oz, sz, k);
            const float s0 = sqdist_exact(xa.x - x1, ya.x - y1, za.x - z1);
            const float s1 = sqdist_exact(xa.y - x1, ya.y - y1, za.y - z1);
            const float s2 = sqdist_exact(xa.z - x1, ya.z - y1, za.z - z1);
            const float s3 = sqdist_exact(xa.w - x1, ya.w - y1, za.w - z1);
            const bool p0 = valid && s0 <= R2, p1 = valid && s1 <= R2, p2 = valid && s2 <= R2, p3 = valid && s3 <= R2;
            if (__any_sync(0xffffffffu, p0 || p1 || p2 || p3)) {
                consider(k, s0, p0);
                consider(k + 1, s1, p1);
                consider(k + 2, s2, p2);
                consider(k + 3, s3, p3);
            }
        }
    } else {
        for (int k = t; k < n; k += tpb) {
            const float s = sqdist_exact(ld1<GLOBAL>(ox + k) - x1, ld1<GLOBAL>(oy + k) - y1, ld1<GLOBAL>(oz + k) - z1);
            consider(k, s, valid && s <= R2);
        }
    }
    if (__any_sync(0xffffffffu, qn > 0)) evaluate_queue();   // what is still queued; no radius is needed any more
    return r;
}

// merge of a bidder group's partial results inside a warp (over min(tpb, 32) lanes)
__device__ __forceinline__ void warp_merge_top2(Top2 &r, int wl) {
    for (int o = wl >> 1; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, r.best, o);
        const float o2 = __shfl_xor_sync(0xffffffffu, r.better, o);
        const int oi = __shfl_xor_sync(0xffffffffu, r.idx, o);
        merge_top2(r, ob, o2, oi);
    }
}

// GLOBAL = false: the cloud's whole state lives in (distributed) shared memory (n <= 8192).
// GLOBAL = true : clouds too large for that (the reference accepts any n % 1024 == 0, emd_cuda.cu:125-133,236-249): the same
//                 auction with the object coordinates, prices and the sliced state in a per-cloud global workspace (L2
//                 resident); a CTA's slice pointer is array + rank * ns, so a remote slice is plain pointer arithmetic.
//                 The cluster barriers order the global accesses (release / acquire at cluster scope); mutable state that
//                 other CTAs write is read through L2 (ld.global.cg / atomics).  No object grid, no solo phase.
template <bool GLOBAL>
__global__ void __launch_bounds__(kEmdThreads, 1) emd_auction_kernel(const EmdParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cg::cluster_group cluster = cg::this_cluster();
    const int S = (int)cluster.num_blocks();
    const int rank = (int)cluster.block_rank();
    const int cloud = blockIdx.x / S;
    const int n = p.n;
    const int ns = n / S;           // slice length (objects owned / bidders homed by this CTA)
    const int base = rank * ns;     // first global index of the slice
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // ---- carve-up (identical offsets in every CTA of the cluster): shared memory, or the cloud's global workspace
    float *gbase = GLOBAL ? p.gws + (size_t)cloud * 11 * n : reinterpret_cast<float *>(smem_raw);
    float *ox = gbase;
    float *oy = ox + n;
    float *oz = oy + n;
    float *price = oz + n;
    float *sl = price + n;                                      // sliced arrays: [ns] each in shared memory, [n] each (this CTA's part at + base) in GLOBAL mode
    const int sstride = GLOBAL ? n : ns, soff = GLOBAL ? base : 0;
    float *max_inc = sl + soff;                                 // [ns] owner slice
    int *winner = reinterpret_cast<int *>(sl + sstride) + soff;         // [ns] owner slice
    int *ass_inv = reinterpret_cast<int *>(sl + 2 * sstride) + soff;    // [ns] owner slice
    int *assign = reinterpret_cast<int *>(sl + 3 * sstride) + soff;     // [ns] home slice
    int *bid = reinterpret_cast<int *>(sl + 4 * sstride) + soff;        // [ns] home slice
    float *bid_inc = sl + 5 * sstride + soff;                           // [ns] home slice
    int *list = reinterpret_cast<int *>(sl + 6 * sstride) + soff;       // [ns] compacted local bidder ids
    float *w_best = GLOBAL ? reinterpret_cast<float *>(smem_raw) : sl + 7 * ns;   // [32] cross-warp merge scratch
    float *w_better = w_best + 32;
    int *w_idx = reinterpret_cast<int *>(w_better + 32);
    int *ucount = w_idx + 32;                                   // [8] bidder count of every rank
    int *cnt = ucount + 8;                                      // [1]
    // slice of cluster rank r2 of a sliced array (given this CTA's slice pointer)
    auto rmt = [&](auto *ptr, int r2) { return GLOBAL ? ptr + (r2 - rank) * ns : cluster.map_shared_rank(ptr, r2); };
    // object grid: the objects sorted by cell of a kGridG^3 grid over their bounding box
    float *gx = reinterpret_cast<float *>(cnt + 4);             // [n] cell-sorted coordinates
    float *gy = gx + n;
    float *gz = gy + n;
    int *gperm = reinterpret_cast<int *>(gz + n);               // [n] original object index
    int *cell_start = gperm + n;                                // [kGridCells + 4]
    int *cell_fill = cell_start + kGridCells + 4;               // [kGridCells]
    float *gbox = reinterpret_cast<float *>(cell_fill + kGridCells);   // [8] min xyz, inverse cell size xyz, hmin, abs slack
    unsigned int *gred = reinterpret_cast<unsigned int *>(gbox + 8);    // [8] min / max reduction (ordered uints), ok flag
    float *after_grid = p.grid ? reinterpret_cast<float *>(gred + 8) : reinterpret_cast<float *>(cnt + 4);
    // solo mode (only rank 0's copies are used): the whole cloud's sliced state gathered into full-length arrays
    float *F_maxinc = after_grid;                               // [n]
    int *F_winner = reinterpret_cast<int *>(F_maxinc + n);      // [n]
    int *F_inv = F_winner + n;                                  // [n]
    int *F_assign = F_inv + n;                                  // [n]
    int *F_bid = F_assign + n;                                  // [n]
    float *F_binc = reinterpret_cast<float *>(F_bid + n);       // [n]
    int *s_list = reinterpret_cast<int *>(F_binc + n);          // [2][kSoloMax] bidder lists (global point indices)
    int *s_cnt = s_list + 2 * kSoloMax;                         // [2]
    int *s_sbid = s_cnt + 2;                                    // [kSoloMax]
    float *s_sinc = reinterpret_cast<float *>(s_sbid + kSoloMax);   // [kSoloMax]
    float *F_x1 = s_sinc + kSoloMax;                            // [3n] the cloud's points (bidder coordinates)

    const float *x1g = p.xyz1 + (size_t)cloud * n * 3;
    const float *x2g = p.xyz2 + (size_t)cloud * n * 3;
    const size_t cb = (size_t)cloud * n;

    // ---- load state (the caller pre-initialises it as emd_module.py:43-54; honour what is there)
    // resident mode: every CTA keeps its own replica of all n objects and prices; GLOBAL mode: one copy, filled slice by slice
    for (int k = (GLOBAL ? base : 0) + tid; k < (GLOBAL ? base + ns : n); k += kEmdThreads) {
        ox[k] = x2g[k * 3 + 0];
        oy[k] = x2g[k * 3 + 1];
        oz[k] = x2g[k * 3 + 2];
        price[k] = (p.price && !p.fresh) ? p.price[cb + k] : 0.f;
    }
    for (int k = tid; k < ns; k += kEmdThreads) {
        max_inc[k] = (p.max_increments && !p.fresh) ? p.max_increments[cb + base + k] : 0.f;
        winner[k] = INT_MAX;
        ass_inv[k] = (p.assignment_inv && !p.fresh) ? p.assignment_inv[cb + base + k] : -1;
        assign[k] = p.fresh ? -1 : p.assignment[cb + base + k];
    }
    if (p.solo && tid < 2) s_cnt[tid] = 0;
    // ---- object grid (every CTA builds its own copy).  A bidder then visits the cells around it ring by ring and stops
    // as soon as everything closer than its pruning radius has been seen, instead of testing all n objects.
    bool use_grid = false;
    if (!GLOBAL && p.grid) {
        if (tid < 8) gred[tid] = (tid < 3) ? 0xffffffffu : 0u;
        for (int c = tid; c < kGridCells; c += kEmdThreads) cell_fill[c] = 0;
        __syncthreads();
        {
            unsigned int mn[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, mx[3] = {0u, 0u, 0u};
            unsigned int bad = 0;
            for (int k = tid; k < n; k += kEmdThreads) {
                const float c3[3] = {ox[k], oy[k], oz[k]};
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    bad |= !(fabsf(c3[a]) < 1e18f);
                    const unsigned int o = ford(c3[a]);
                    mn[a] = min(mn[a], o); mx[a] = max(mx[a], o);
                }
            }
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                mn[a] = __reduce_min_sync(0xffffffffu, mn[a]);
                mx[a] = __reduce_max_sync(0xffffffffu, mx[a]);
            }
            bad = __reduce_max_sync(0xffffffffu, bad);
            if (lane == 0) {
#pragma unroll
                for (int a = 0; a < 3; ++a) { atomicMin(gred + a, mn[a]); atomicMax(gred + 3 + a, mx[a]); }
                if (bad) atomicMax(gred + 6, 1u);
            }
        }
        __syncthreads();
        if (tid == 0) {
            float hmin = 3.0e38f, slack = 0.f;
            for (int a = 0; a < 3; ++a) {
                const float lo3 = funord(gred[a]), hi3 = funord(gred[3 + a]);
                const float h = (hi3 - lo3) / (float)kGridG;
                gbox[a] = lo3;
                gbox[3 + a] = h > 0.f ? 1.0f / h : 0.f;
                hmin = fminf(hmin, h);
                slack += fabsf(lo3) + fabsf(hi3);
            }
            gbox[6] = hmin;
            gbox[7] = 2e-6f * slack + 1e-30f;   // cell assignment of objects and bidders is exact up to a few ulps of the coordinates
        }
        __syncthreads();
        use_grid = gred[6] == 0u && gbox[6] > 0.f;
        if (use_grid) {
            auto cell_of = [&](float x, float y, float z) {
                const int cx = min(kGridG - 1, max(0, (int)((x - gbox[0]) * gbox[3])));
                const int cy = min(kGridG - 1, max(0, (int)((y - gbox[1]) * gbox[4])));
                const int cz = min(kGridG - 1, max(0, (int)((z - gbox[2]) * gbox[5])));
                return (cz * kGridG + cy) * kGridG + cx;
            };
            for (int k = tid; k < n; k += kEmdThreads) atomicAdd(cell_fill + cell_of(ox[k], oy[k], oz[k]), 1);
            __syncthreads();
            if (warp == 0) {   // exclusive scan of the 512 counts: 16 per lane
                int loc[kGridCells / 32], sum = 0;
#pragma unroll
                for (int i = 0; i < kGridCells / 32; ++i) { loc[i] = cell_fill[lane * (kGridCells / 32) + i]; sum += loc[i]; }
                int incl = sum;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += v;
                }
                int run = incl - sum;
#pragma unroll
                for (int i = 0; i < kGridCells / 32; ++i) {
                    cell_start[lane * (kGridCells / 32) + i] = run;
                    cell_fill[lane * (kGridCells / 32) + i] = run;
                    run += loc[i];
                }
                if (lane == 31) cell_start[kGridCells] = run;
                int mx = 0;
#pragma unroll
                for (int i = 0; i < kGridCells / 32; ++i) mx = max(mx, loc[i]);
                mx = __reduce_max_sync(0xffffffffu, mx);
                if (lane == 0) gred[7] = (unsigned int)mx;   // (slot 7 is the bidder counter of the iterations later on)
            }
            __syncthreads();
            // a cloud that piles a quarter of its objects into one cell (tight clusters plus outliers) gains nothing from
            // the grid: every block would hold most of the objects
            if ((int)gred[7] * 4 > n) use_grid = false;
            for (int k = tid; k < n; k += kEmdThreads) {
                const int pos = atomicAdd(cell_fill + cell_of(ox[k], oy[k], oz[k]), 1);
                gx[pos] = ox[k]; gy[pos] = oy[k]; gz[pos] = oz[k]; gperm[pos] = k;
            }
        }
    }
    cluster.sync();

    int solo_from = -1;
    for (int it = 0; it < p.iters; ++it) {
        const bool last = (it == p.iters - 1);
        EMD_STAMP(it, 0);
        // ---- 1. compact the unassigned points homed here (order is result-neutral, emd_cuda.cu:85-93)
        if (tid == 0) *cnt = 0;
        __syncthreads();
        for (int k = tid; k < ns; k += kEmdThreads) {
            const bool un = assign[k] == -1;
            const unsigned int m = __ballot_sync(0xffffffffu, un);
            int wbase = 0;
            if (lane == 0 && m) wbase = atomicAdd(cnt, __popc(m));
            wbase = __shfl_sync(0xffffffffu, wbase, 0);
            if (un) list[wbase + __popc(m & ((1u << lane) - 1u))] = k;
        }
        __syncthreads();
        const int u = *cnt;
        if (tid < S) *cluster.map_shared_rank(ucount + rank, tid) = u;
        // The bidders are homed by point index, so the CTAs of a cluster hold different numbers of them and the slowest one
        // sets the pace of every iteration (cluster-barrier stalls were 26 % of the samples).  One more barrier makes the
        // counts known before the scan, and every CTA takes an equal share of the cluster's bidder list: bidder ids are read
        // from their home CTA's list over DSMEM, the results go back to the home CTA's bid / bid_increments.
        if (S > 1) cluster.sync();  // [R] counts visible
        int total_u = 0, lo = 0, hi = u;
        if (S > 1) {
            for (int r2 = 0; r2 < S; ++r2) total_u += ucount[r2];
            lo = (int)(((long long)rank * total_u) / S);
            hi = (int)(((long long)(rank + 1) * total_u) / S);
        } else {
            total_u = u;
        }
        if (total_u == 0) break;  // uniform across the cluster; later iterations cannot change anything
        const int mine = hi - lo;
        EMD_STAMP(it, 1);
        EMD_NOTE(it, 6, total_u);

        // ---- 2./3. Bid with the object grid: one warp per bidder.  The warp visits the 3x3x3 block of cells around the
        // bidder, then the next shell, ... every object it meets is evaluated exactly.  After a shell of Chebyshev radius
        // rr, every unvisited object is at least rr cells away along some axis, i.e. farther than `covered`; once that is
        // at least the pruning radius R = 3 - better + 2e-6 (an object can change the top two only if sqrt(s) < R, prices
        // being >= 0) nothing unvisited can matter and the scan stops -- the same exact cut-off as the full scan below.
        const bool grid_now = !GLOBAL && use_grid && total_u >= p.grid_min_u;
        if (grid_now) {
            int *next_bidder = reinterpret_cast<int *>(gred + 7);
            if (tid == 0) *next_bidder = 0;
            __syncthreads();
            for (;;) {   // bidders need different numbers of shells: warps take them from a counter
                int a0 = 0;
                if (lane == 0) a0 = atomicAdd(next_bidder, 1);
                a0 = __shfl_sync(0xffffffffu, a0, 0);
                if (a0 >= mine) break;
                int a = lo + a0, hr = 0;
                if (S > 1) {
                    while (hr < S - 1 && a >= ucount[hr]) { a -= ucount[hr]; ++hr; }
                }
                const int jl = *(rmt(list, hr) + a);
                const int j = hr * ns + jl;
                const float x1 = x1g[j * 3 + 0], y1 = x1g[j * 3 + 1], z1 = x1g[j * 3 + 2];
                const int bcx = min(kGridG - 1, max(0, (int)((x1 - gbox[0]) * gbox[3])));
                const int bcy = min(kGridG - 1, max(0, (int)((y1 - gbox[1]) * gbox[4])));
                const int bcz = min(kGridG - 1, max(0, (int)((z1 - gbox[2]) * gbox[5])));
                Top2 r, m;
                int run_incl = 0, run_beg = 0, run_n = 0;   // this lane's run: inclusive prefix of lengths, first object
                // The objects of x-adjacent cells are contiguous in the sorted arrays: the (2rr+1)^3 block around the bidder
                // is (2rr+1)^2 runs.  Their objects are spread evenly over the lanes, four independent evaluations in
                // flight per lane.  rr = 1, then 2 (the whole block again, from scratch); beyond that every object.
                float Rprev2 = 3.0e38f, Rgprev = 3.0e38f;   // pruning radius known from the previous shell: R^2 and 3 - better
                for (int rr = 1;; ++rr) {
                    r.best = kNegInit; r.better = kNegInit; r.idx = -1;
                    int total;
                    if (rr <= 2) {
                        const int side = 2 * rr + 1, nruns = side * side;
                        int len = 0, beg = 0;
                        if (lane < nruns) {
                            const int dz = lane / side - rr, dy = lane - (lane / side) * side - rr;
                            const int cy = bcy + dy, cz = bcz + dz;
                            if ((unsigned)cy < (unsigned)kGridG && (unsigned)cz < (unsigned)kGridG) {
                                const int rowc = (cz * kGridG + cy) * kGridG;
                                beg = cell_start[rowc + max(0, bcx - rr)];
                                len = cell_start[rowc + min(kGridG - 1, bcx + rr) + 1] - beg;
                            }
                        }
                        int incl = len;
#pragma unroll
                        for (int o = 1; o < 32; o <<= 1) {
                            const int v = __shfl_up_sync(0xffffffffu, incl, o);
                            if (lane >= o) incl += v;
                        }
                        run_incl = incl; run_beg = beg; run_n = nruns;
                        total = __shfl_sync(0xffffffffu, incl, 31);
                    } else {
                        total = n;                     // everything (rare: the radius exceeds two cells)
                    }
                    for (int base0 = 0; base0 < total; base0 += 128) {   // warp-uniform trip count (shuffles inside)
                        const int pos0 = base0 + lane;
                        int ks[4], os[4];
                        float ss[4], vs[4];
                        if (rr <= 2) {
                            // run of each of the lane's four positions: the number of runs whose inclusive prefix is <= pos
                            int q[4] = {0, 0, 0, 0};
                            for (int t2 = 0; t2 < run_n; ++t2) {
                                const int pre = __shfl_sync(0xffffffffu, run_incl, t2);
#pragma unroll
                                for (int i = 0; i < 4; ++i) q[i] += (pre <= pos0 + 32 * i);
                            }
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int qq = min(q[i], 31);
                                const int b0 = __shfl_sync(0xffffffffu, run_beg, qq);
                                const int pinc = __shfl_sync(0xffffffffu, run_incl, max(qq - 1, 0));
                                os[i] = b0 + (pos0 + 32 * i - (qq ? pinc : 0));
                            }
                        } else {
#pragma unroll
                            for (int i = 0; i < 4; ++i) os[i] = pos0 + 32 * i;
                        }
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            ks[i] = -1; ss[i] = 0.f;
                            if (pos0 + 32 * i < total) {
                                const int o = os[i];
                                ss[i] = sqdist_exact(gx[o] - x1, gy[o] - y1, gz[o] - z1);
                                if (ss[i] <= Rprev2) {
                                    // inside the radius known from the previous shell; as in the full scan, the object's own
                                    // price tightens it: v > better needs sqrt(s) < 3 - better - price[k]
                                    const int k = gperm[o];
                                    const float pk = price[k];
                                    const float Rk = (Rgprev - pk) + (4e-6f + 1e-6f * (fabsf(Rgprev) + fabsf(pk)));
                                    if (Rk > 0.f && ss[i] <= Rk * Rk * 1.000002f) ks[i] = k;
                                }
                            }
                        }
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            vs[i] = (float)(3.0 - (double)__fsqrt_rn(ss[i]) - (double)price[ks[i] < 0 ? 0 : ks[i]]);
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const int k = ks[i];
                            const float v = vs[i];
                            if (k >= 0) {   // objects arrive in no particular order: equal values keep the lowest index
                                if (v > r.best) { r.better = r.best; r.best = v; r.idx = k; }
                                else if (v == r.best) { r.better = r.best; r.idx = min(r.idx, k); }
                                else if (v > r.better) r.better = v;
                            }
                        }
                    }
                    __syncwarp();
                    m = r;
                    warp_top2_redux(m);
                    if (rr > 2) break;
                    const float R = (3.0f - m.better) + 2e-6f;
                    const float covered = (float)rr * gbox[6] - gbox[7];
                    if (covered >= R * 1.000001f) break;
                    Rprev2 = R * R * 1.000001f;   // as in the full scan: sqrt(s) > R cannot change the top two
                    Rgprev = 3.0f - m.better;
                    // a radius beyond two cells cannot be covered by the 5x5x5 block either (it only shrinks if far, cheap
                    // objects beat the near ones): go straight to the every-object pass
                    if (rr == 1 && 2.0f * gbox[6] - gbox[7] < R * 1.000001f) rr = 2;
                }
                if (lane == 0) {
                    const float inc = __fadd_rn(__fsub_rn(m.best, m.better), p.eps);
                    *(rmt(bid, hr) + jl) = m.idx;
                    *(rmt(bid_inc, hr) + jl) = inc;
                    if (m.idx >= 0) {
                        const int orank = m.idx / ns;
                        atomic_max_float(rmt(max_inc, orank) + (m.idx - orank * ns), inc);
                    }
                }
            }
        }
        // ---- 2./3. Bid (emd_cuda.cu:95-179): G bidders at a time, tpb threads per bidder
        // The bidders are processed in passes of G = a power of two bidders (tpb = 1024 / G threads each).  One pass of
        // the next power of two >= mine wastes up to half of the lanes: take that pass only if at least 3/4 of its groups
        // are real, else a full pass of half the size and continue with the remainder.
        for (int a0 = 0, G = 1; a0 < mine && !grid_now; a0 += G) {
            const int rem = mine - a0;
            G = 1;
            while (G < rem && G < kEmdThreads) G <<= 1;
            if (G > 1 && rem * 4 < G * 3) G >>= 1;
            const int tpb = kEmdThreads / G;
            const int g = tid / tpb, t = tid - g * tpb;
            const bool valid = a0 + g < mine;
            // global position in the cluster's bidder list -> (home rank, index in its list)
            int a = lo + (valid ? a0 + g : 0), hr = 0;
            if (S > 1) {
                while (hr < S - 1 && a >= ucount[hr]) { a -= ucount[hr]; ++hr; }
            }
            const int jl = *(rmt(list, hr) + a);   // idle groups look at the first bidder of the share
            const int j = hr * ns + jl;
            const float x1 = x1g[j * 3 + 0], y1 = x1g[j * 3 + 1], z1 = x1g[j * 3 + 2];
            const int wl = tpb < 32 ? tpb : 32;
            Top2 r = scan_bidder<GLOBAL>(ox, oy, oz, price, n, x1, y1, z1, tpb, t, valid);
            if (wl == 32) warp_top2_redux(r);   // whole warp, one bidder: three redux.sync instead of five shuffle rounds
            else warp_merge_top2(r, wl);
            if (tpb > 32) {  // bidder groups span several warps: finish through shared memory
                __syncthreads();
                if (lane == 0) { w_best[warp] = r.best; w_better[warp] = r.better; w_idx[warp] = r.idx; }
                __syncthreads();
                if (t == 0) {
                    const int wpb = tpb >> 5;
                    for (int w = 1; w < wpb; ++w) merge_top2(r, w_best[warp + w], w_better[warp + w], w_idx[warp + w]);
                }
            }
            if (valid && t == 0) {
                const float inc = __fadd_rn(__fsub_rn(r.best, r.better), p.eps);
                *(rmt(bid, hr) + jl) = r.idx;
                *(rmt(bid_inc, hr) + jl) = inc;
                if (r.idx >= 0) {
                    const int orank = r.idx / ns;
                    atomic_max_float(rmt(max_inc, orank) + (r.idx - orank * ns), inc);
                }
            }
        }
        EMD_STAMP(it, 2);
        EMD_NOTE(it, 7, grid_now ? 1 : 0);
        cluster.sync();  // [A] all bids and max_increments visible cluster-wide
        EMD_STAMP(it, 3);

        // ---- 4. GetMax (emd_cuda.cu:181-194): lowest bidder index within +-1e-6 (fp64) of the maximum
        for (int a = tid; a < u; a += kEmdThreads) {
            const int jl = list[a];
            const int o = bid[jl];
            if (o >= 0) {
                const int orank = o / ns, ol = o - orank * ns;
                const double bi = (double)bid_inc[jl];
                const double mi = (double)*(rmt(max_inc, orank) + ol);
                if (bi - 1e-6 <= mi && mi <= bi + 1e-6) atomicMin(rmt(winner, orank) + ol, base + jl);
            }
        }
        cluster.sync();  // [B]
        EMD_STAMP(it, 4);

        // ---- 5. Assign (emd_cuda.cu:196-215)
        for (int a = tid; a < u; a += kEmdThreads) {
            const int jl = list[a];
            const int o = bid[jl];
            if (o >= 0) {
                const int orank = o / ns, ol = o - orank * ns;
                const int w = *(rmt(winner, orank) + ol);
                if (last || w == base + jl) {
                    const float inc = bid_inc[jl];
                    int *inv = rmt(ass_inv, orank) + ol;
                    const int old = *inv;
                    if (!last && old != -1) {
                        const int hr = old / ns;
                        *(rmt(assign, hr) + (old - hr * ns)) = -1;
                    }
                    *inv = base + jl;
                    assign[jl] = o;
                    const float np = __fadd_rn(ld1<GLOBAL>(price + o), inc);
                    if (GLOBAL) price[o] = np;
                    else for (int r2 = 0; r2 < S; ++r2) *(cluster.map_shared_rank(price, r2) + o) = np;
                    *(rmt(max_inc, orank) + ol) = kNegInit;
                    *(rmt(winner, orank) + ol) = INT_MAX;
                }
            }
        }
        cluster.sync();  // [C]
        EMD_STAMP(it, 5);
        // The number of unassigned points never grows (a winner takes one point off the list and evicts at most one), so once
        // a cloud is down to a handful of bidders it stays there -- typically for hundreds of iterations at the training
        // setting (eps = 0.05, 3000 iterations).  Those iterations are pure latency in the cluster-wide form (three cluster
        // barriers, remote atomics, a 1024-thread scan for one bidder): rank 0 finishes them alone.
        if (!GLOBAL && p.solo && total_u <= kSoloMax && !last) { solo_from = it + 1; break; }
    }

    if (!GLOBAL && solo_from >= 0) {
        {   // gather the sliced state and the unassigned points in rank 0
            float *r_maxinc = cluster.map_shared_rank(F_maxinc, 0);
            int *r_winner = cluster.map_shared_rank(F_winner, 0), *r_inv = cluster.map_shared_rank(F_inv, 0);
            int *r_assign = cluster.map_shared_rank(F_assign, 0), *r_bid = cluster.map_shared_rank(F_bid, 0);
            float *r_binc = cluster.map_shared_rank(F_binc, 0);
            int *r_list = cluster.map_shared_rank(s_list, 0), *r_cnt = cluster.map_shared_rank(s_cnt, 0);
            for (int k = tid; k < ns; k += kEmdThreads) {
                r_maxinc[base + k] = max_inc[k]; r_winner[base + k] = winner[k]; r_inv[base + k] = ass_inv[k];
                r_assign[base + k] = assign[k]; r_bid[base + k] = bid[k]; r_binc[base + k] = bid_inc[k];
                if (assign[k] == -1) {
                    const int pos = atomicAdd(r_cnt, 1);
                    if (pos < kSoloMax) r_list[pos] = base + k;
                }
            }
        }
        cluster.sync();
        if (rank == 0) {
            for (int i = tid; i < 3 * n; i += kEmdThreads) F_x1[i] = x1g[i];
            __syncthreads();
            int cur = 0;
            for (int it = solo_from; it < p.iters; ++it) {
                const bool last = (it == p.iters - 1);
                const int u = min(s_cnt[cur], kSoloMax);
                if (u == 0) break;
                int *lst = s_list + cur * kSoloMax, *nxt = s_list + (cur ^ 1) * kSoloMax;
                if (tid == 0) s_cnt[cur ^ 1] = 0;
                // Bid: all u bidders in one pass, 1024 / G threads each (G = next power of two >= u, so >= 32 threads)
                {
                    const int lg = u <= 1 ? 0 : 32 - __clz(u - 1);          // log2(G)
                    const int tpb = kEmdThreads >> lg, wpb = tpb >> 5;
                    const int g = tid >> (10 - lg), t = tid & (tpb - 1);
                    const bool valid = g < u;
                    const int j = lst[valid ? g : 0];
                    const float x1 = F_x1[j * 3 + 0], y1 = F_x1[j * 3 + 1], z1 = F_x1[j * 3 + 2];
                    Top2 r = scan_bidder<GLOBAL>(ox, oy, oz, price, n, x1, y1, z1, tpb, t, valid);
                    warp_top2_redux(r);
                    if (wpb > 1) {   // the group's warps meet in shared memory; its first warp merges them
                        if (lane == 0) { w_best[warp] = r.best; w_better[warp] = r.better; w_idx[warp] = r.idx; }
                        __syncthreads();
                        if (t < 32) {
                            const bool have = lane < wpb;
                            r.best = have ? w_best[warp + lane] : kNegInit;
                            r.better = have ? w_better[warp + lane] : kNegInit;
                            r.idx = have ? w_idx[warp + lane] : -1;
                            warp_top2_redux(r);
                        }
                    }
                    if (u == 1) {
                        // a single bidder (the usual case in the long tail: an eviction chain): thread 0 runs winner
                        // selection and assignment right here, with the state transitions of the general path
                        if (tid == 0) {
                            const float inc = __fadd_rn(__fsub_rn(r.best, r.better), p.eps);
                            const int o = r.idx;
                            F_bid[j] = o; F_binc[j] = inc;
                            int push = j;
                            if (o >= 0) {
                                float mi = F_maxinc[o];
                                if (inc > mi) mi = inc;                                   // atomic_max_float
                                int w = F_winner[o];
                                const double bi = (double)inc, md = (double)mi;
                                if (bi - 1e-6 <= md && md <= bi + 1e-6 && j < w) w = j;     // GetMax
                                if (last || w == j) {                                      // Assign
                                    const int old = F_inv[o];
                                    push = -1;
                                    if (!last && old != -1) { F_assign[old] = -1; push = old; }
                                    F_inv[o] = j;
                                    F_assign[j] = o;
                                    price[o] = __fadd_rn(price[o], inc);
                                    F_maxinc[o] = kNegInit;
                                    F_winner[o] = INT_MAX;
                                } else {
                                    F_maxinc[o] = mi;
                                    F_winner[o] = w;
                                }
                            }
                            s_cnt[cur ^ 1] = push >= 0 ? 1 : 0;
                            if (push >= 0) nxt[0] = push;
                        }
                        __syncthreads();
                        cur ^= 1;
                        continue;
                    }
                    if (valid && t == 0) {
                        const float inc = __fadd_rn(__fsub_rn(r.best, r.better), p.eps);
                        F_bid[j] = r.idx; F_binc[j] = inc;
                        s_sbid[g] = r.idx; s_sinc[g] = inc;
                        if (r.idx >= 0) atomic_max_float(F_maxinc + r.idx, inc);
                    }
                }
                __syncthreads();
                // GetMax
                if (tid < u) {
                    const int o = s_sbid[tid];
                    if (o >= 0) {
                        const double bi = (double)s_sinc[tid], mi = (double)F_maxinc[o];
                        if (bi - 1e-6 <= mi && mi <= bi + 1e-6) atomicMin(F_winner + o, lst[tid]);
                    }
                }
                __syncthreads();
                // Assign; whoever stays or becomes unassigned goes on the next list
                if (tid < u) {
                    const int j = lst[tid], o = s_sbid[tid];
                    int push = j;
                    if (o >= 0) {
                        const int w = F_winner[o];
                        if (last || w == j) {
                            const float inc = s_sinc[tid];
                            const int old = F_inv[o];
                            push = -1;
                            if (!last && old != -1) { F_assign[old] = -1; push = old; }
                            F_inv[o] = j;
                            F_assign[j] = o;
                            price[o] = __fadd_rn(price[o], inc);
                            F_maxinc[o] = kNegInit;
                            F_winner[o] = INT_MAX;
                        }
                    }
                    if (push >= 0) {
                        const int pos = atomicAdd(s_cnt + (cur ^ 1), 1);
                        if (pos < kSoloMax) nxt[pos] = push;
                    }
                }
                __syncthreads();
                cur ^= 1;
            }
            // CalcDist + write-back for the whole cloud
            float lsum = 0.f;
            for (int j = tid; j < n; j += kEmdThreads) {
                const int o = F_assign[j];
                float d = 0.f;
                if (o >= 0)
                    d = sqdist_exact(x1g[j * 3 + 0] - ox[o], x1g[j * 3 + 1] - oy[o], x1g[j * 3 + 2] - oz[o]);
                lsum += __fsqrt_rn(d);
                p.dist[cb + j] = d;
                p.assignment[cb + j] = o;
                if (p.assignment_inv) p.assignment_inv[cb + j] = F_inv[j];
                if (p.max_increments) p.max_increments[cb + j] = F_maxinc[j];
                if (p.bid) p.bid[cb + j] = F_bid[j];
                if (p.bid_increments) p.bid_increments[cb + j] = F_binc[j];
                if (p.price) p.price[cb + j] = price[j];
            }
            if (p.loss_sums) {   // fused sum_j sqrt(dist) of Loss.get_emd_loss (loss/loss.py:25): one atomic per warp
#pragma unroll
                for (int o2 = 16; o2 > 0; o2 >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, o2);
                if (lane == 0) atomicAdd(p.loss_sums + cloud, lsum);
            }
        }
        cluster.sync();  // keep every CTA's shared memory alive until rank 0 is done
        return;
    }

    // ---- CalcDist (emd_cuda.cu:217-226) + write-back of the state the reference leaves in its tensors
    float lsum = 0.f;
    for (int k = tid; k < ns; k += kEmdThreads) {
        const int j = base + k;
        const int o = assign[k];
        float d = 0.f;
        if (o >= 0)
            d = sqdist_exact(x1g[j * 3 + 0] - ox[o], x1g[j * 3 + 1] - oy[o], x1g[j * 3 + 2] - oz[o]);
        lsum += __fsqrt_rn(d);
        p.dist[cb + j] = d;
        p.assignment[cb + j] = o;
        if (p.assignment_inv) p.assignment_inv[cb + j] = ass_inv[k];
        if (p.max_increments) p.max_increments[cb + j] = max_inc[k];
        if (p.bid) p.bid[cb + j] = bid[k];
        if (p.bid_increments) p.bid_increments[cb + j] = bid_inc[k];
        if (p.price) p.price[cb + j] = price[j];
    }
    if (p.loss_sums) {   // fused sum_j sqrt(dist) of Loss.get_emd_loss (loss/loss.py:25): one atomic per warp
#pragma unroll
        for (int o2 = 16; o2 > 0; o2 >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, o2);
        if (lane == 0) atomicAdd(p.loss_sums + cloud, lsum);
    }
    cluster.sync();  // keep every CTA's shared memory alive until all remote accesses are done
}

// emd_cuda_backward's NmDistanceGradKernel (emd_cuda.cu:284-300): one term per address.
// OVERWRITE = false: the reference's contract (accumulate into the caller-zeroed gradient); true: plain store.
// MEAN_LOSS: grad_dist is formed in the kernel for loss = sqrt(dist).mean(1).mean() (loss/loss.py:25) from the saved
// distances: grad_dist = ((upstream / B) / n) / (2 sqrt(dist)) -- autograd's own sequence (mean, mean(1), sqrt), including
// the infinite factor at dist == 0 that the reference's loss has.
template <bool OVERWRITE, bool MEAN_LOSS>
__global__ void __launch_bounds__(256) emd_grad_kernel(int total, int n, int b, const float *__restrict__ xyz1,
                                                       const float *__restrict__ xyz2, const float *__restrict__ grad_dist,
                                                       const float *__restrict__ upstream, const int *__restrict__ idx,
                                                       float *grad_xyz) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    const int cloud = e / n;
    const int j2 = idx[e];
    float gd;
    if (MEAN_LOSS) {
        const float up = upstream ? __ldg(upstream) : 1.0f;
        const float t = __fdiv_rn(__fdiv_rn(up, (float)b), (float)n);
        gd = __fdiv_rn(t, __fmul_rn(2.0f, __fsqrt_rn(grad_dist[e])));   // grad_dist carries the saved dist here
    } else {
        gd = grad_dist[e];
    }
    const float g = gd * 2.0f;
    const float *a = xyz1 + (size_t)e * 3;
    float *o = grad_xyz + (size_t)e * 3;
    float v[3] = {0.f, 0.f, 0.f};
    if (j2 >= 0) {   // an unassigned point (possible when iters == 0) has no term
        const float *bq = xyz2 + ((size_t)cloud * n + j2) * 3;
#pragma unroll
        for (int k = 0; k < 3; ++k) v[k] = __fmul_rn(g, __fsub_rn(a[k], bq[k]));
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) o[k] = OVERWRITE ? v[k] : __fadd_rn(o[k], v[k]);
}

// loss = mean_b( sum_j sqrt(dist[b, j]) / n ) from the per-cloud sums of the auction kernel's epilogue; one warp.
__global__ void emd_mean_loss_kernel(const float *__restrict__ sums, int b, float n, float *__restrict__ out) {
    float s1 = 0.f;
    for (int i = threadIdx.x; i < b; i += 32) s1 += __fdiv_rn(sums[i], n);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    if (threadIdx.x == 0) *out = __fdiv_rn(s1, (float)b);
}

// ---- Certificate of an (assignment, prices) pair: weak-duality bounds on the Euclidean EMD (emd_certified).
// For ANY prices p and any permutation a:  sum_j d(j, a_j)  >=  L = sum_j min_k (d_jk + p_k) - sum_k p_k,  and U = sum_j d(j, a_j)
// is the cost of a feasible matching, so L <= optimum <= U.  Nothing about the auction is assumed.  Every quantity is
// rounded towards its bound: d_jk + p_k downwards for L (|dx| rounded down, squares and sums of squares rounded down,
// __dsqrt_rd), sum_k p_k upwards; d(j, a_j) upwards for U.  The sums run in a fixed order (no float atomics): the bounds are
// reproducible bit for bit.
constexpr int kBoundThreads = 256;
constexpr int kBoundRowsPerLane = 8;                                   // bidders per warp; every lane carries all of them
constexpr int kBoundRows = (kBoundThreads / 32) * kBoundRowsPerLane;   // 64 bidders per CTA
constexpr int kBoundTile = 2048;                                       // objects staged in shared memory per pass (32 KB)

// |a - b| of two floats rounded down / up in fp64 (the exact difference of two floats does not always fit a double)
__device__ __forceinline__ double absdiff_rd(float a, float b) { return __dsub_rd((double)fmaxf(a, b), (double)fminf(a, b)); }
__device__ __forceinline__ double absdiff_ru(float a, float b) { return __dsub_ru((double)fmaxf(a, b), (double)fminf(a, b)); }
__device__ __forceinline__ double sqdist_rd(float ax, float ay, float az, float bx, float by, float bz) {
    const double dx = absdiff_rd(ax, bx), dy = absdiff_rd(ay, by), dz = absdiff_rd(az, bz);
    return __fma_rd(dz, dz, __fma_rd(dy, dy, __dmul_rd(dx, dx)));
}
__device__ __forceinline__ double sqdist_ru(float ax, float ay, float az, float bx, float by, float bz) {
    const double dx = absdiff_ru(ax, bx), dy = absdiff_ru(ay, by), dz = absdiff_ru(az, bz);
    return __fma_ru(dz, dz, __fma_ru(dy, dy, __dmul_ru(dx, dx)));
}

// CTA (blockIdx.x, cloud blockIdx.y) owns 64 bidders j: part_lo = sum over them of min_k (d_jk + p_k) rounded down,
// part_hi = sum of d(j, a_j) rounded up (0 for an assignment outside [0, n); the final kernel then reports no permutation).
// A warp holds 8 bidders, its lanes split the objects, staged through shared memory 2048 at a time.  The fp64 square root is
// taken only when the pair can lower the running minimum m: it cannot if p_k >= m or s >= t^2 with t = m - p_k rounded up
// (then sqrt(s) >= t and d + p_k >= m), and a skipped pair leaves the minimum unchanged.
__global__ void __launch_bounds__(kBoundThreads) emd_bound_rows_kernel(const float *__restrict__ xyz1, const float *__restrict__ xyz2,
                                                                       const int *__restrict__ assignment, const float *__restrict__ price,
                                                                       int n, double *__restrict__ part_lo, double *__restrict__ part_hi) {
    __shared__ float4 obj[kBoundTile];
    __shared__ double row_lo[kBoundRows], row_hi[kBoundRows];
    const int cloud = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const size_t cb = (size_t)cloud * n;
    const float *x1 = xyz1 + cb * 3, *x2 = xyz2 + cb * 3;
    const int row0 = blockIdx.x * kBoundRows + warp * kBoundRowsPerLane;
    float bx[kBoundRowsPerLane], by[kBoundRowsPerLane], bz[kBoundRowsPerLane];
    double mn[kBoundRowsPerLane];
#pragma unroll
    for (int r = 0; r < kBoundRowsPerLane; ++r) {
        const int j = min(row0 + r, n - 1);   // rows past the end repeat the last one and are not summed
        bx[r] = x1[j * 3 + 0]; by[r] = x1[j * 3 + 1]; bz[r] = x1[j * 3 + 2];
        mn[r] = __longlong_as_double(0x7ff0000000000000LL);   // +inf
    }
    for (int k0 = 0; k0 < n; k0 += kBoundTile) {
        const int cnt = min(kBoundTile, n - k0);
        __syncthreads();
        for (int i = tid; i < cnt; i += kBoundThreads) {
            const int k = k0 + i;
            obj[i] = make_float4(x2[k * 3 + 0], x2[k * 3 + 1], x2[k * 3 + 2], price ? price[cb + k] : 0.f);
        }
        __syncthreads();
        for (int i = lane; i < cnt; i += 32) {
            const float4 o = obj[i];
            const double p = (double)o.w;
#pragma unroll
            for (int r = 0; r < kBoundRowsPerLane; ++r) {
                const double s = sqdist_rd(bx[r], by[r], bz[r], o.x, o.y, o.z);
                const double t = __dsub_ru(mn[r], p);
                if (t > 0.0 && s < __dmul_ru(t, t)) mn[r] = fmin(mn[r], __dadd_rd(__dsqrt_rd(s), p));
            }
        }
    }
#pragma unroll
    for (int r = 0; r < kBoundRowsPerLane; ++r) {
        double m = mn[r];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmin(m, __shfl_xor_sync(0xffffffffu, m, o));   // exact: min is order-free
        if (lane == r) row_lo[warp * kBoundRowsPerLane + r] = m;
    }
    if (lane < kBoundRowsPerLane) {
        const int j = row0 + lane;
        double hi = 0.0;
        if (j < n) {
            const int a = assignment[cb + j];
            if (a >= 0 && a < n) hi = __dsqrt_ru(sqdist_ru(x1[j * 3 + 0], x1[j * 3 + 1], x1[j * 3 + 2], x2[a * 3 + 0], x2[a * 3 + 1], x2[a * 3 + 2]));
        }
        row_hi[warp * kBoundRowsPerLane + lane] = hi;
    }
    __syncthreads();
    if (tid == 0) {
        double lo = 0.0, hi = 0.0;
        const int rows = min(kBoundRows, n - (int)blockIdx.x * kBoundRows);
        for (int r = 0; r < rows; ++r) { lo = __dadd_rd(lo, row_lo[r]); hi = __dadd_ru(hi, row_hi[r]); }
        part_lo[(size_t)cloud * gridDim.x + blockIdx.x] = lo;
        part_hi[(size_t)cloud * gridDim.x + blockIdx.x] = hi;
    }
}

// One CTA per cloud: permutation check (a bitmap of the objects in shared memory), sum_k p_k rounded up (strided partial sums,
// then a fixed tree), the partial sums of the rows kernel in CTA order, and the per-point means.
constexpr int kBoundFinalThreads = 1024;
__global__ void __launch_bounds__(kBoundFinalThreads) emd_bound_final_kernel(const int *__restrict__ assignment, const float *__restrict__ price,
                                                                             int n, int nblk, const double *__restrict__ part_lo,
                                                                             const double *__restrict__ part_hi, double *__restrict__ bounds,
                                                                             int *__restrict__ status) {
    extern __shared__ unsigned int seen[];
    __shared__ double red[kBoundFinalThreads];
    const int cloud = blockIdx.x, tid = threadIdx.x;
    const size_t cb = (size_t)cloud * n;
    const int words = (n + 31) >> 5;
    for (int w = tid; w < words; w += kBoundFinalThreads) seen[w] = 0u;
    __syncthreads();
    int bad = 0;
    double ps = 0.0;
    for (int j = tid; j < n; j += kBoundFinalThreads) {
        const int o = assignment[cb + j];
        if (o < 0 || o >= n) {
            bad = 1;
        } else {
            const unsigned int bit = 1u << (o & 31);
            if (atomicOr(seen + (o >> 5), bit) & bit) bad = 1;   // object taken twice
        }
        if (price) ps = __dadd_ru(ps, (double)price[cb + j]);
    }
    red[tid] = ps;
    bad = __syncthreads_or(bad);
    for (int s = kBoundFinalThreads / 2; s > 0; s >>= 1) {
        if (tid < s) red[tid] = __dadd_ru(red[tid], red[tid + s]);
        __syncthreads();
    }
    if (tid == 0) {
        double lo = 0.0, hi = 0.0;
        for (int i = 0; i < nblk; ++i) {
            lo = __dadd_rd(lo, part_lo[(size_t)cloud * nblk + i]);
            hi = __dadd_ru(hi, part_hi[(size_t)cloud * nblk + i]);
        }
        bounds[2 * (size_t)cloud + 0] = __ddiv_rd(__dsub_rd(lo, red[0]), (double)n);
        bounds[2 * (size_t)cloud + 1] = bad ? __longlong_as_double(0x7ff8000000000000LL) : __ddiv_ru(hi, (double)n);
        status[cloud] = bad ? 0 : 1;
    }
}

static size_t emd_smem_bytes(int n, int S) {
    const int ns = n / S;
    return sizeof(float) * (size_t)(4 * n) + sizeof(float) * (size_t)(7 * ns) + sizeof(float) * (32 * 3 + 8 + 4);
}
static size_t emd_grid_bytes(int n) { return sizeof(float) * ((size_t)4 * n + (kGridCells + 4) + kGridCells + 8 + 8); }
static size_t emd_solo_bytes(int n) { return sizeof(float) * ((size_t)9 * n + 2 * kSoloMax + 2 + 2 * kSoloMax); }

}  // namespace psd

using namespace psd;

static std::atomic<int> g_emd_grid{1};
int psd_set_emd_grid(int enable) { return (enable == 0 || enable == 1) ? g_emd_grid.exchange(enable) : g_emd_grid.load(); }
static std::atomic<int> g_emd_solo{1};
int psd_set_emd_solo(int enable) { return (enable == 0 || enable == 1) ? g_emd_solo.exchange(enable) : g_emd_solo.load(); }

// returns cudaSuccess, or an error.  Clouds whose state fits in the (distributed) shared memory of a cluster (n <= 8192) run
// the resident kernel; larger clouds run the same auction on a stream-ordered global workspace (11 n floats per cloud).
// force_cluster: 0 = automatic, 1/2/4/8 = cluster size (test hook), negative = -cluster size AND the global-workspace form
// (test hook: parity of the GLOBAL mode at small sizes).
cudaError_t psd_launch_emd_forward(const float *xyz1, const float *xyz2, int b, int n, float *dist, int *assignment,
                                   float *price, int *assignment_inv, int *bid, float *bid_increments,
                                   float *max_increments, float eps, int iters, int force_cluster, int fresh,
                                   float *loss_sums, cudaStream_t stream, int *unsupported) {
    *unsupported = 0;
    if (b <= 0 || n <= 0) return cudaSuccess;
    int dev = 0, num_sms = 148, max_smem = 227 * 1024;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    bool global = force_cluster < 0;
    int S = 1;
    if (force_cluster != 0) {
        S = force_cluster < 0 ? -force_cluster : force_cluster;
        if (S != 1 && S != 2 && S != 4 && S != 8) return cudaErrorInvalidValue;
    } else {
        while (S < 8 && b * (S * 2) <= num_sms) S *= 2;
    }
    if (!global) {
        while (S < 8 && emd_smem_bytes(n, S) > (size_t)max_smem) S *= 2;
        if (emd_smem_bytes(n, S) > (size_t)max_smem) { global = true; S = 8; }
    }
    if ((n % S) != 0) { *unsupported = 1; return cudaSuccess; }
    EmdParams p;
    p.xyz1 = xyz1; p.xyz2 = xyz2; p.dist = dist; p.assignment = assignment; p.price = price;
    p.assignment_inv = assignment_inv; p.max_increments = max_increments; p.bid = bid; p.bid_increments = bid_increments;
    p.b = b; p.n = n; p.eps = eps; p.iters = iters; p.fresh = fresh; p.solo = 0; p.grid = 0; p.gws = nullptr;
    p.loss_sums = loss_sums;
    {
        const char *ev = getenv("PSD_EMD_GRID_MIN_U");
        p.grid_min_u = ev ? atoi(ev) : 144;   // measured optimum for cluster sizes 2, 4 and 8 (sweep 0 ... 1024 at B = 64, 32, 8)
    }
    size_t smem;
    cudaError_t e;
    if (global) {
        smem = sizeof(float) * (32 * 3 + 8 + 4);
        e = cudaMallocAsync(reinterpret_cast<void **>(&p.gws), sizeof(float) * 11 * (size_t)n * (size_t)b, stream);
        if (e != cudaSuccess) return e;
    } else {
        smem = emd_smem_bytes(n, S);
        p.grid = (smem + emd_grid_bytes(n) <= (size_t)max_smem && g_emd_grid.load()) ? 1 : 0;
        if (p.grid) smem += emd_grid_bytes(n);
        p.solo = (smem + emd_solo_bytes(n) <= (size_t)max_smem && g_emd_solo.load()) ? 1 : 0;
        if (p.solo) smem += emd_solo_bytes(n);
        e = cudaFuncSetAttribute(emd_auction_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned int)(b * S));
    cfg.blockDim = dim3(kEmdThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned int)S;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (global) {
        e = cudaLaunchKernelEx(&cfg, emd_auction_kernel<true>, p);
        const cudaError_t e2 = cudaFreeAsync(p.gws, stream);
        return e != cudaSuccess ? e : e2;
    }
    return cudaLaunchKernelEx(&cfg, emd_auction_kernel<false>, p);
}

cudaError_t psd_launch_emd_mean_loss(const float *sums, int b, int n, float *out, cudaStream_t stream) {
    emd_mean_loss_kernel<<<1, 32, 0, stream>>>(sums, b, (float)n, out);
    return cudaGetLastError();
}

// mode: 0 = accumulate grad_dist terms (reference contract), 1 = overwrite, 2 = mean-loss gradient (graddist = saved dist,
// upstream = device scalar or NULL for 1.0), overwrite
cudaError_t psd_launch_emd_backward(const float *xyz1, const float *xyz2, float *gradxyz, const float *graddist,
                                    const int *idx, int b, int n, int mode, const float *upstream, cudaStream_t stream) {
    if (b <= 0 || n <= 0) return cudaSuccess;
    const int total = b * n;
    const int blocks = (total + 255) / 256;
    if (mode == 0) emd_grad_kernel<false, false><<<blocks, 256, 0, stream>>>(total, n, b, xyz1, xyz2, graddist, nullptr, idx, gradxyz);
    else if (mode == 1) emd_grad_kernel<true, false><<<blocks, 256, 0, stream>>>(total, n, b, xyz1, xyz2, graddist, nullptr, idx, gradxyz);
    else emd_grad_kernel<true, true><<<blocks, 256, 0, stream>>>(total, n, b, xyz1, xyz2, graddist, upstream, idx, gradxyz);
    return cudaGetLastError();
}

int psd_emd_bound_max_points() { return 1 << 20; }   // the permutation bitmap of a cloud (n / 8 bytes) sits in shared memory

// bounds[B, 2] (lower, upper per point, fp64) and status[B] of (assignment, price); price may be NULL (all zero).  Two launches
// and a stream-ordered scratch of 2 B ceil(n / 64) doubles; nothing synchronises the host (capturable in a CUDA graph).
cudaError_t psd_launch_emd_dual_bound(const float *xyz1, const float *xyz2, int b, int n, const int *assignment, const float *price,
                                      double *bounds, int *status, cudaStream_t stream) {
    if (b <= 0 || n <= 0) return cudaSuccess;
    const int nblk = (n + kBoundRows - 1) / kBoundRows;
    const size_t smem = sizeof(unsigned int) * (size_t)((n + 31) / 32);
    cudaError_t e = cudaFuncSetAttribute(emd_bound_final_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    double *part = nullptr;
    e = cudaMallocAsync(reinterpret_cast<void **>(&part), sizeof(double) * 2 * (size_t)b * nblk, stream);
    if (e != cudaSuccess) return e;
    double *part_lo = part, *part_hi = part + (size_t)b * nblk;
    emd_bound_rows_kernel<<<dim3((unsigned int)nblk, (unsigned int)b), kBoundThreads, 0, stream>>>(xyz1, xyz2, assignment, price, n,
                                                                                                 part_lo, part_hi);
    e = cudaGetLastError();
    if (e == cudaSuccess) {
        emd_bound_final_kernel<<<b, kBoundFinalThreads, smem, stream>>>(assignment, price, n, nblk, part_lo, part_hi, bounds, status);
        e = cudaGetLastError();
    }
    const cudaError_t e2 = cudaFreeAsync(part, stream);
    return e != cudaSuccess ? e : e2;
}
