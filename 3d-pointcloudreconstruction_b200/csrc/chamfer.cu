// chamfer.cu -- B200-native Chamfer nearest-neighbour forward and gradient scatter.
//
// Replaces metric/chamfer3D/chamfer3D.cu of the reference (NmDistanceKernel :12-134,
// NmDistanceGradKernel :155-174 and their launchers :136-154, :176-195).  Results are bit-identical
// to the reference for finite inputs (dist AND lowest-index argmin) -- see DESIGN.md "Chamfer forward".
//
// Forward design (FP32-FMA-pipe bound, 8 algorithmic flop per directed pair):
//   * one CTA = 32*Q queries of one cloud/direction; its 4 warps hold the SAME queries in registers and
//     each scans a quarter of the targets, so an SM that hosts k CTAs puts k warps on each of its four
//     sub-partitions (grid of 1024 CTAs on 148 SMs at B=32, N=M=2048 -> 6.92 CTAs/SM, all co-resident).
//   * targets are staged per 1024-point tile in shared memory as SoA x[], y[], z[], w[] where the
//     coordinates are centred on the cloud (t - c) and w = |t - c|^2; one broadcast LDS.128 per array
//     feeds 4 targets to all lanes.
//   * FILTER: a_k = w_k - 2 (q-c).(t_k-c) = |t_k-q|^2 - |q-c|^2 costs 3 FMAs per pair, issued as packed
//     FFMA2 (two targets per instruction); the minimum over a 16-target chunk is taken with FMNMX3.
//     Per chunk and query the kernel keeps (best chunk minimum, its chunk id, second-best chunk minimum).
//   * EXACT: a rigorous rounding bound (margin = 2^-18 (|q-c| + max|t-c|)^2, derivation in DESIGN.md) says
//     the reference's argmin lies in the best chunk whenever second > best + margin; that chunk (16
//     targets) is re-evaluated with the reference's exact formula fma(dz,dz,fma(dx,dx,rn(dy*dy))) in index
//     order with strict '<'.  Otherwise (near-ties, duplicated points, non-finite input) the query takes
//     an exact full scan that also reproduces the reference's NaN/512-tile semantics.
//   => dist/idx are always produced by the exact formula; the filter only decides where to look.
#include "chamfer_nn.cuh"
#include "psd_device.h"

#ifndef PSD_GRAD_TRIGGER_EARLY
#define PSD_GRAD_TRIGGER_EARLY 1
#endif
namespace psd {

constexpr int kWarps = 16;        // one persistent CTA per SM: 4 warps on each of the four sub-partitions
constexpr int kThreads = kWarps * 32;
constexpr int kPartBytes = kWarps * kQB * 12;  // per-block partial results: (best, second, chunk) per warp and query

__device__ unsigned long long g_fallback_queries = 0ull;

struct BlockInfo {      // per block of the current flush group (shared memory)
    int blk, d, cloud, qblock;   // static part, filled once per flush group (the only integer divisions)
    float cx, cy, cz;   // centre of the filter frame
    float t2max;        // max |t-c|^2 over the target cloud
    int bad;            // non-finite / huge target seen
    int qn, tn, inval;  // ragged launches: the pair's participating queries / targets (0 / 0 for an invalid pair); else 0
};
constexpr int kPerBlockBytes = kPartBytes + (int)sizeof(BlockInfo) + 3 * kQB * 4 + kQB * 4;  // + staged queries + fallback list

// RAGGED: per-pair lengths (NNRaggedParams); blocks of the padded grid beyond them do no search.
template <int TM, bool RAGGED>
__global__ void __launch_bounds__(kThreads, 1) chamfer_nn_kernel(const std::conditional_t<RAGGED, NNRaggedParams, NNParams> p) {
    constexpr int Q = kQ, QB = kQB, C = kChunk;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *sX = reinterpret_cast<float *>(smem_raw);               // SoA target tile: x, y, z, w = |t-c|^2
    float *sY = sX + TM;
    float *sZ = sY + TM;
    float *sW = sZ + TM;
    float *part_best = sW + TM;                                   // [flush][kWarps][QB]
    float *part_second = part_best + p.flush * kWarps * QB;
    int *part_chunk = reinterpret_cast<int *>(part_second + p.flush * kWarps * QB);
    float *sq = reinterpret_cast<float *>(part_chunk + p.flush * kWarps * QB);   // [flush][3][QB] staged raw queries
    int *fb_list = reinterpret_cast<int *>(sq + p.flush * 3 * QB);               // [flush*QB]
    BlockInfo *binfo = reinterpret_cast<BlockInfo *>(fb_list + p.flush * QB);    // [flush]
    __shared__ float s_tile_wmax;
    __shared__ int s_tile_bad;
    __shared__ int s_nfb;
    __shared__ unsigned long long s_key[kWarps];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = gridDim.x;
    const int blk_begin = (int)(((long long)blockIdx.x * p.total_blocks) / G);
    const int blk_end = (int)(((long long)(blockIdx.x + 1) * p.total_blocks) / G);
    zero_fill(p);

    float cx = 0.f, cy = 0.f, cz = 0.f;   // filter-frame centre of group c_group
    int c_group = -1;
    // shared-memory resident tile: (group = dir,cloud; first target) and its statistics
    int res_group = -1, res_t0 = -1;
    float res_wmax = 0.f;
    int res_bad = 0;

    for (int fb0 = blk_begin; fb0 < blk_end; fb0 += p.flush) {
        const int nb = min(p.flush, blk_end - fb0);
        // =========================== set-up: decode the blocks and stage their queries in shared memory
        if (tid < nb) {
            BlockInfo bi;
            bi.blk = fb0 + tid;
            bi.d = bi.blk >= p.blocks_dir0 ? 1 : 0;
            const int bid = bi.d ? bi.blk - p.blocks_dir0 : bi.blk;
            const int qbn = p.dir[bi.d].qblocks;
            bi.cloud = bid / qbn;
            bi.qblock = bid - bi.cloud * qbn;
            bi.cx = bi.cy = bi.cz = 0.f; bi.t2max = 0.f; bi.bad = 0; bi.qn = bi.tn = bi.inval = 0;
            if constexpr (RAGGED) bi.inval = !ragged_lengths(p, bi.d, bi.cloud, bi.qn, bi.tn);
            binfo[tid] = bi;
        }
        __syncthreads();
        for (int i = tid; i < nb * QB; i += kThreads) {
            const int bl = i / QB, ql = i - bl * QB;
            const BlockInfo &bi = binfo[bl];
            const NNDirection &D = p.dir[bi.d];
            const float *__restrict__ qb = D.q + (long long)bi.cloud * D.q_bs;
            int j = D.q_begin + bi.qblock * QB + ql;
            const int q_last = RAGGED ? max(min(D.q_begin + D.q_count, bi.qn) - 1, 0) : D.q_begin + D.q_count - 1;
            j = j < q_last ? j : q_last;
            sq[(bl * 3 + 0) * QB + ql] = __ldg(qb + j * D.q_ps);
            sq[(bl * 3 + 1) * QB + ql] = __ldg(qb + j * D.q_ps + D.q_cs);
            sq[(bl * 3 + 2) * QB + ql] = __ldg(qb + j * D.q_ps + 2 * D.q_cs);
        }
        if (tid == 0) s_nfb = 0;
        __syncthreads();

        // =========================== stage A: filter scan, one block after the other (no barrier between
        // blocks while the target tile stays resident: warps run ahead independently)
        for (int bl = 0; bl < nb; ++bl) {
            const int d = binfo[bl].d, cloud = binfo[bl].cloud;
            const NNDirection &D = p.dir[d];
            // ragged: a block whose queries all lie beyond the pair's length (or of an invalid pair) scans nothing
            const int nt = !RAGGED ? D.nt : (D.q_begin + binfo[bl].qblock * QB < binfo[bl].qn ? binfo[bl].tn : 0);
            const float *__restrict__ tb = D.t + (long long)cloud * D.t_bs;
            const long long tps = D.t_ps, tcs = D.t_cs;
            const int group = d * 0x40000000 + cloud;

            // centre of the filter's coordinate frame: mean of up to 8 evenly spaced targets.  Any value is
            // correct (results come from the exact formula); a centred frame only keeps the margin small.
            if (group != c_group && (!RAGGED || nt > 0)) {
                float sx = 0.f, sy = 0.f, sz = 0.f;
                const int ns = nt < 8 ? nt : 8;
                const int step = nt >> 3;
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    if (s < ns) {
                        const long long k = nt < 8 ? s : s * step;
                        sx += __ldg(tb + k * tps);
                        sy += __ldg(tb + k * tps + tcs);
                        sz += __ldg(tb + k * tps + 2 * tcs);
                    }
                }
                const float inv = 1.0f / (float)ns;
                cx = sx * inv; cy = sy * inv; cz = sz * inv;
                c_group = group;
            }
            float qx[Q], qy[Q], qz[Q];  // -2 (q - c)
            float best[Q], second[Q];
            int bchunk[Q];
#pragma unroll
            for (int i = 0; i < Q; ++i) {
                qx[i] = -2.0f * (sq[(bl * 3 + 0) * QB + i * 32 + lane] - cx);
                qy[i] = -2.0f * (sq[(bl * 3 + 1) * QB + i * 32 + lane] - cy);
                qz[i] = -2.0f * (sq[(bl * 3 + 2) * QB + i * 32 + lane] - cz);
                best[i] = kBig; second[i] = kBig; bchunk[i] = 0;
            }
            float blk_wmax = 0.f;
            int blk_bad = 0;
            const bool vec_ok = (tps == 3) && (tcs == 1) && ((reinterpret_cast<unsigned long long>(tb) & 15ull) == 0ull);

            for (int t0 = 0; t0 < nt; t0 += TM) {
                const int cnt = min(TM, nt - t0);
                const int nchunks = (cnt + C - 1) / C;
                if (!(res_group == group && res_t0 == t0)) {
                    // ---- (re)load the tile: everybody must be done with the previous one
                    __syncthreads();
                    if (tid == 0) { s_tile_wmax = 0.f; s_tile_bad = 0; }
                    float wmax = 0.f;
                    int bad = 0;
                    if (vec_ok && (cnt & 7) == 0) {
                        // AoS fast path: 6 x LDG.128 = 24 floats = 8 whole points per thread and round
                        for (int g8 = tid; g8 * 8 < cnt; g8 += kThreads) {
                            const float4 *src = reinterpret_cast<const float4 *>(tb + (long long)t0 * 3) + g8 * 6;
                            float f[24];
#pragma unroll
                            for (int i = 0; i < 6; ++i) {
                                const float4 v = __ldg(src + i);
                                f[4 * i + 0] = v.x; f[4 * i + 1] = v.y; f[4 * i + 2] = v.z; f[4 * i + 3] = v.w;
                            }
                            float xs[8], ys[8], zs[8], ws[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                xs[i] = f[3 * i + 0] - cx;
                                ys[i] = f[3 * i + 1] - cy;
                                zs[i] = f[3 * i + 2] - cz;
                                ws[i] = __fmaf_rn(zs[i], zs[i], __fmaf_rn(xs[i], xs[i], ys[i] * ys[i]));
                                bad |= !(ws[i] < kLimit);
                                wmax = fmaxf(wmax, ws[i]);
                            }
                            float4 *dX = reinterpret_cast<float4 *>(sX) + g8 * 2, *dY = reinterpret_cast<float4 *>(sY) + g8 * 2;
                            float4 *dZ = reinterpret_cast<float4 *>(sZ) + g8 * 2, *dW = reinterpret_cast<float4 *>(sW) + g8 * 2;
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                dX[h] = make_float4(xs[4 * h], xs[4 * h + 1], xs[4 * h + 2], xs[4 * h + 3]);
                                dY[h] = make_float4(ys[4 * h], ys[4 * h + 1], ys[4 * h + 2], ys[4 * h + 3]);
                                dZ[h] = make_float4(zs[4 * h], zs[4 * h + 1], zs[4 * h + 2], zs[4 * h + 3]);
                                dW[h] = make_float4(ws[4 * h], ws[4 * h + 1], ws[4 * h + 2], ws[4 * h + 3]);
                            }
                        }
                        for (int k = cnt + tid; k < nchunks * C; k += kThreads) { sX[k] = 0.f; sY[k] = 0.f; sZ[k] = 0.f; sW[k] = kBig; }
                    } else {
                        // generic strides / ragged tile: 4 points per thread per round, loads issued before use
                        for (int k0 = tid; k0 < nchunks * C; k0 += 4 * kThreads) {
                            float lx[4], ly[4], lz[4];
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int k = k0 + i * kThreads;
                                const float *tp = tb + (long long)(t0 + (k < cnt ? k : 0)) * tps;
                                lx[i] = __ldg(tp); ly[i] = __ldg(tp + tcs); lz[i] = __ldg(tp + 2 * tcs);
                            }
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int k = k0 + i * kThreads;
                                if (k < nchunks * C) {
                                    float x = 0.f, y = 0.f, z = 0.f, w = kBig;
                                    if (k < cnt) {
                                        x = lx[i] - cx; y = ly[i] - cy; z = lz[i] - cz;
                                        w = __fmaf_rn(z, z, __fmaf_rn(x, x, y * y));
                                        bad |= !(w < kLimit);
                                        wmax = fmaxf(wmax, w);
                                    }
                                    sX[k] = x; sY[k] = y; sZ[k] = z; sW[k] = w;
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        wmax = fmaxf(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
                        bad |= __shfl_xor_sync(0xffffffffu, bad, o);
                    }
                    __syncthreads();  // s_tile_* reset is visible; all tile stores are done
                    if (lane == 0) {
                        atomicMax(reinterpret_cast<int *>(&s_tile_wmax), __float_as_int(wmax));  // wmax >= 0: int order == float order
                        if (bad) atomicOr(&s_tile_bad, 1);
                    }
                    __syncthreads();
                    res_group = group; res_t0 = t0;
                    res_wmax = s_tile_wmax; res_bad = s_tile_bad;
                }
                blk_wmax = fmaxf(blk_wmax, res_wmax);
                blk_bad |= res_bad;

                // software-pipelined over 4-target groups: the next group's four LDS.128 are issued before the
                // current group's 24 FFMA2, also across chunk boundaries.  TM is a template constant so the
                // four arrays are immediate offsets from one address register.
                const float4 *T4 = reinterpret_cast<const float4 *>(sX);
                constexpr int OY = TM / 4, OZ = 2 * (TM / 4), OW = 3 * (TM / 4);
                int c = warp;
                float4 X, Y, Z, W;
                if (c < nchunks) {
                    const float4 *g0 = T4 + c * (C / 4);
                    X = g0[0]; Y = g0[OY]; Z = g0[OZ]; W = g0[OW];
                }
                while (c < nchunks) {
                    float cm[Q];
                    const int cn = c + kWarps;
                    const float4 *gp = T4 + c * (C / 4);
                    const float4 *gn = T4 + cn * (C / 4);
#pragma unroll
                    for (int g = 0; g < C / 4; ++g) {
                        float4 Xn = X, Yn = Y, Zn = Z, Wn = W;
                        if (g + 1 < C / 4) {
                            Xn = gp[g + 1]; Yn = gp[g + 1 + OY]; Zn = gp[g + 1 + OZ]; Wn = gp[g + 1 + OW];
                        } else if (cn < nchunks) {
                            Xn = gn[0]; Yn = gn[OY]; Zn = gn[OZ]; Wn = gn[OW];
                        }
#pragma unroll
                        for (int i = 0; i < Q; ++i) {
                            float2 a01 = ffma2(qz[i], make_float2(Z.x, Z.y), make_float2(W.x, W.y));
                            float2 a23 = ffma2(qz[i], make_float2(Z.z, Z.w), make_float2(W.z, W.w));
                            a01 = ffma2(qy[i], make_float2(Y.x, Y.y), a01);
                            a23 = ffma2(qy[i], make_float2(Y.z, Y.w), a23);
                            a01 = ffma2(qx[i], make_float2(X.x, X.y), a01);
                            a23 = ffma2(qx[i], make_float2(X.z, X.w), a23);
                            if (g == 0) {
                                cm[i] = fminf(fmin3(a01.x, a01.y, a23.x), a23.y);
                            } else {
                                cm[i] = fmin3(cm[i], a01.x, a01.y);
                                cm[i] = fmin3(cm[i], a23.x, a23.y);
                            }
                        }
                        X = Xn; Y = Yn; Z = Zn; W = Wn;
                    }
                    const int gchunk = t0 / C + c;
#pragma unroll
                    for (int i = 0; i < Q; ++i) {
                        const float v = cm[i];
                        second[i] = fminf(second[i], fmaxf(best[i], v));
                        const bool lt = v < best[i];
                        best[i] = fminf(best[i], v);
                        bchunk[i] = lt ? gchunk : bchunk[i];
                    }
                    c = cn;
                }
            }
            // ---- park this warp's partial results for block bl (distinct slots per block: no barrier needed)
            {
                float *pb = part_best + (bl * kWarps + warp) * QB;
                float *ps = part_second + (bl * kWarps + warp) * QB;
                int *pc = part_chunk + (bl * kWarps + warp) * QB;
#pragma unroll
                for (int i = 0; i < Q; ++i) {
                    pb[i * 32 + lane] = best[i];
                    ps[i * 32 + lane] = second[i];
                    pc[i * 32 + lane] = bchunk[i];
                }
                if (tid == 0) {
                    binfo[bl].cx = cx; binfo[bl].cy = cy; binfo[bl].cz = cz;
                    binfo[bl].t2max = blk_wmax; binfo[bl].bad = blk_bad;
                }
            }
        }

        // =========================== stage B: resolve the nb*128 queries of this flush group
        __syncthreads();
        for (int i = tid; i < nb * QB; i += kThreads) {   // a warp covers 32 consecutive queries of ONE block
            const int bl = i / QB, ql = i - bl * QB;
            const BlockInfo bi = binfo[bl];
            const int cloud = bi.cloud;
            const NNDirection &D = p.dir[bi.d];
            const int j = D.q_begin + bi.qblock * QB + ql;
            const bool live = j < D.q_begin + D.q_count && (!RAGGED || j < bi.qn);
            float dres = 0.f;
            bool done = false;
            if (RAGGED && !live && j < D.q_begin + D.q_count) {
                // rows past the pair's query length, and every row of an invalid pair: dist 0 (NaN), idx -1, counted nowhere
                // (the NaN goes into the pair's sums)
                dres = bi.inval ? __int_as_float(0x7fc00000) : 0.f;
                D.dist[(long long)cloud * D.nq + j] = dres;
                D.idx[(long long)cloud * D.nq + j] = -1;
            }
            if (live) {
                const int nt = RAGGED ? bi.tn : D.nt;
                const float *__restrict__ tb = D.t + (long long)cloud * D.t_bs;
                const long long tps = D.t_ps, tcs = D.t_cs;
                float b1 = kBig, b2 = kBig;
                int bc = 0;
#pragma unroll
                for (int w = 0; w < kWarps; ++w) {
                    const float v = part_best[(bl * kWarps + w) * QB + ql];
                    b2 = fminf(b2, fminf(part_second[(bl * kWarps + w) * QB + ql], fmaxf(b1, v)));
                    if (v < b1) { b1 = v; bc = part_chunk[(bl * kWarps + w) * QB + ql]; }
                }
                const float x1 = sq[(bl * 3 + 0) * QB + ql], y1 = sq[(bl * 3 + 1) * QB + ql], z1 = sq[(bl * 3 + 2) * QB + ql];
                const float ux = x1 - bi.cx, uy = y1 - bi.cy, uz = z1 - bi.cz;
                const float qq = __fmaf_rn(uz, uz, __fmaf_rn(ux, ux, uy * uy));
                // margin = 26u * min(S, S') with 15% slack (u = 2^-24; derivation in DESIGN.md):
                //   S  = (|q-c| + max|t-c|)^2 bounds every target,
                //   S' = (2|q-c| + rho)^2 bounds the targets that can compete (within rho of the query).
                const float qn = sqrtf(qq);
                const float r = qn + sqrtf(bi.t2max);
                const float S = r * r;
                const float rho = sqrtf(fmaxf(b1 + qq, 0.f) + 2.4e-6f * S);
                const float r2 = 2.0f * qn + rho;
                const float Seff = fminf(S, r2 * r2);
                const float margin = __fmaf_rn(Seff, 1.8e-6f, 1e-36f);
                const bool ok = !bi.bad && (S < 4.0f * kLimit) && (b2 > b1 + margin);
                if (ok) {
                    const int k0 = bc * C;
                    const int k1 = min(k0 + C, nt);
                    float dv[C];
                    if (tps == 3 && tcs == 1 && k1 - k0 == C && ((reinterpret_cast<unsigned long long>(tb) & 15ull) == 0ull)) {
                        // AoS, 16-byte aligned chunk (16 points = 192 B): 12 x LDG.128 in flight at once
                        const float4 *src = reinterpret_cast<const float4 *>(tb + (long long)k0 * 3);
                        float f[3 * C];
#pragma unroll
                        for (int u = 0; u < 3 * C / 4; ++u) {
                            const float4 v = __ldg(src + u);
                            f[4 * u] = v.x; f[4 * u + 1] = v.y; f[4 * u + 2] = v.z; f[4 * u + 3] = v.w;
                        }
#pragma unroll
                        for (int u = 0; u < C; ++u) dv[u] = sqdist_exact(f[3 * u] - x1, f[3 * u + 1] - y1, f[3 * u + 2] - z1);
                    } else {
#pragma unroll
                        for (int u = 0; u < C; ++u) dv[u] = exact_d(tb, tps, tcs, min(k0 + u, k1 - 1), x1, y1, z1);
                    }
                    float dbest = dv[0];
                    int ibest = k0;
#pragma unroll
                    for (int u = 1; u < C; ++u) {
                        if (k0 + u < k1 && dv[u] < dbest) { dbest = dv[u]; ibest = k0 + u; }
                    }
                    D.dist[(long long)cloud * D.nq + j] = dbest;
                    D.idx[(long long)cloud * D.nq + j] = ibest;
                    dres = dbest;
                    done = true;
                } else {
                    fb_list[atomicAdd(&s_nfb, 1)] = i;
                }
            }
            if (p.sums != nullptr || p.fs_count != nullptr) {   // fused epilogues, one atomic per warp
                float ws = (done || RAGGED) ? dres : 0.f;
                int wc = (done && dres < p.fs_thr) ? 1 : 0;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    ws += __shfl_xor_sync(0xffffffffu, ws, o);
                    wc += __shfl_xor_sync(0xffffffffu, wc, o);
                }
                if (lane == 0) {
                    if (p.sums) atomicAdd(p.sums + cloud * 2 + D.slot, ws);
                    if (p.fs_count && wc) atomicAdd(p.fs_count + cloud * 2 + D.slot, wc);
                }
            }
        }
        __syncthreads();

        // ---- exact full scan for the flagged queries, the whole CTA per query.  Reference semantics incl. NaN:
        // within a 512-target tile the first element is taken unconditionally and NaN never replaces or is
        // replaced (chamfer3D.cu:36); a tile result replaces the running result only if strictly smaller (:126).
        const int nfb = s_nfb;
        for (int f = 0; f < nfb; ++f) {   // 4 independent targets per thread and round
            const int i = fb_list[f];
            const int bl = i / QB, ql = i - bl * QB;
            const BlockInfo bi = binfo[bl];
            const int cloud = bi.cloud;
            const NNDirection &D = p.dir[bi.d];
            const int j = D.q_begin + bi.qblock * QB + ql;
            const int nt = RAGGED ? bi.tn : D.nt;
            const float *__restrict__ tb = D.t + (long long)cloud * D.t_bs;
            const long long tps = D.t_ps, tcs = D.t_cs;
            const float x1 = sq[(bl * 3 + 0) * QB + ql], y1 = sq[(bl * 3 + 1) * QB + ql], z1 = sq[(bl * 3 + 2) * QB + ql];
            const bool nan_possible = bi.bad || !(fabsf(x1) < 1e18f) || !(fabsf(y1) < 1e18f) || !(fabsf(z1) < 1e18f);
            unsigned long long key = ~0ull;
            for (int kb = tid; kb < nt; kb += 4 * kThreads) {
                float dd[4], dts[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int k = min(kb + u * kThreads, nt - 1);
                    dd[u] = exact_d(tb, tps, tcs, k, x1, y1, z1);
                    dts[u] = nan_possible ? exact_d(tb, tps, tcs, k & ~(kRefTile - 1), x1, y1, z1) : 0.f;
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int k = kb + u * kThreads;
                    if (k < nt && !(dd[u] != dd[u]) && !(dts[u] != dts[u])) {
                        const unsigned long long kk = pack_key(dd[u], k);
                        key = kk < key ? kk : key;
                    }
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long other = shfl_xor_u64(key, o);
                key = other < key ? other : key;
            }
            if (lane == 0) s_key[warp] = key;
            __syncthreads();
            if (tid == 0) {
                unsigned long long kmin = s_key[0];
#pragma unroll
                for (int w = 1; w < kWarps; ++w) kmin = s_key[w] < kmin ? s_key[w] : kmin;
                const float d0 = exact_d(tb, tps, tcs, 0, x1, y1, z1);
                float dres;
                int ires;
                if (d0 != d0) { dres = d0; ires = 0; }   // tile 0 poisoned: stays NaN, index 0
                else { dres = __uint_as_float((unsigned int)(kmin >> 32)); ires = (int)(kmin & 0xffffffffu); }
                D.dist[(long long)cloud * D.nq + j] = dres;
                D.idx[(long long)cloud * D.nq + j] = ires;
                if (p.sums) atomicAdd(p.sums + cloud * 2 + D.slot, dres);
                if (p.fs_count && dres < p.fs_thr) atomicAdd(p.fs_count + cloud * 2 + D.slot, 1);
            }
            __syncthreads();
        }
        if (nfb > 0 && tid == 0) atomicAdd(&g_fallback_queries, (unsigned long long)nfb);
        __syncthreads();  // partial-result slots, staged queries and fb_list are reused by the next flush group
    }
}

// ------------------------------------------------------------------------------------------------
// Backward: replaces both NmDistanceGradKernel launches (chamfer3D.cu:155-195) with one kernel.
// One term per (direction, cloud, point): g = 2*graddist; v = g*(a - b[idx]) with the subtraction
// rounded before the multiply, exactly as the reference's SASS (FADD, FMUL, no FMA);
//   own-point term: grad_a[j]   += v   (one term per address and direction)
//   scatter term  : grad_b[idx] -= v   aggregated inside the warp first: lanes that hit the same target
//                   (__match_any_sync) are summed by the lowest lane of the group, one atomic per axis.
// Two forms:
//   OVERWRITE = false  the reference's contract (chamfer3D.cu:177-178): accumulate into caller-zeroed buffers, every
//                      term an atomic.
//   OVERWRITE = true   the gradients need no initialisation: a first launch STORES the own-point terms (every element of
//                      both gradients is written exactly once), a second launch adds the scatter terms.
// Clouds and their gradients are addressed through (point, component) strides, so the generator's native
// [B,3,N] layout (train.py:160-163) needs no transpose copy in either direction.
// ------------------------------------------------------------------------------------------------
struct GradParams {
    const float *xyz1, *xyz2;
    float *g1, *g2;
    const float *gd1, *gd2;
    const int *idx1, *idx2;
    int b, n, m;
    long long total1;  // b*n
    long long total;   // b*(n+m)
    long long ps1, cs1, ps2, cs2;   // point / component stride (floats) of cloud 1 and 2; the gradients use the same
    // mean-loss mode (gd1 == gd2 == nullptr): graddist1[e] = *upstream / cnt1, graddist2[e] = *upstream / cnt2 -- what
    // autograd hands to the reference's backward for loss = mean(dist1) + mean(dist2) (loss/loss.py:36)
    const float *upstream;
    float cnt1, cnt2;
};

struct GradTerm {
    bool d2;            // direction 2 (cloud 2's points are the queries)
    long long own;      // float offset of component 0 of the own point in its cloud / gradient
    long long tgt;      // float offset of component 0 of the matched point in the other cloud / gradient
    float v[3];
};

__device__ __forceinline__ GradTerm grad_term(const GradParams &p, long long gid) {
    GradTerm t;
    t.d2 = gid >= p.total1;
    const long long e = t.d2 ? gid - p.total1 : gid;  // flat (cloud, point) index in its direction
    const int na = t.d2 ? p.m : p.n, nb = t.d2 ? p.n : p.m;
    const float *a = t.d2 ? p.xyz2 : p.xyz1;
    const float *bq = t.d2 ? p.xyz1 : p.xyz2;
    const long long psa = t.d2 ? p.ps2 : p.ps1, csa = t.d2 ? p.cs2 : p.cs1;
    const long long psb = t.d2 ? p.ps1 : p.ps2, csb = t.d2 ? p.cs1 : p.cs2;
    const float *gd = t.d2 ? p.gd2 : p.gd1;
    const int *idx = t.d2 ? p.idx2 : p.idx1;
    const long long cloud = p.total < 0x7fffffffLL ? (long long)((int)e / na) : e / na;
    const int j = (int)(e - cloud * na);
    const int j2 = __ldg(idx + e);
    const float gdv = gd ? __ldg(gd + e) : __fdiv_rn(p.upstream ? __ldg(p.upstream) : 1.0f, t.d2 ? p.cnt2 : p.cnt1);
    const float g = gdv * 2.0f;
    t.own = cloud * 3 * na + j * psa;
    t.tgt = cloud * 3 * nb + j2 * psb;
#pragma unroll
    for (int k = 0; k < 3; ++k) t.v[k] = __fmul_rn(g, __fsub_rn(__ldg(a + t.own + k * csa), __ldg(bq + t.tgt + k * csb)));
    return t;
}

// ragged backward: per-pair lengths of xyz1 / xyz2 (device int [b], NULL = n / m)
struct GradRaggedParams : GradParams {
    const int *len1, *len2;
};

// The term of (direction, cloud, point) gid in a ragged backward: 1 = a term (grad_term); 0 = the point lies at or beyond its
// cloud's length (nothing is read); 2 = the pair has a length outside [1, n] / [1, m] (t.own is set and t.v is NaN: the
// point's gradient row becomes NaN, and there is no scatter term).
__device__ __forceinline__ int grad_term_ragged(const GradRaggedParams &p, long long gid, GradTerm &t) {
    const bool d2 = gid >= p.total1;
    const long long e = d2 ? gid - p.total1 : gid;
    const int na = d2 ? p.m : p.n;
    const long long cloud = e / na;
    const int j = (int)(e - cloud * na);
    const int l1 = p.len1 ? __ldg(p.len1 + cloud) : p.n, l2 = p.len2 ? __ldg(p.len2 + cloud) : p.m;
    const bool ok = l1 >= 1 && l1 <= p.n && l2 >= 1 && l2 <= p.m;
    if (ok && j >= (d2 ? l2 : l1)) return 0;
    if (ok) { t = grad_term(p, gid); return 1; }
    t.d2 = d2;
    t.own = cloud * 3 * na + j * (d2 ? p.ps2 : p.ps1);
    t.v[0] = t.v[1] = t.v[2] = __int_as_float(0x7fc00000);
    return 2;
}

// o[0], o[cs], o[2 cs] += (vx, vy, vz).  For the reference layout (cs == 1: three adjacent floats) the 8-byte aligned pair goes
// out as ONE vector atomic (red.global.add.v2.f32, sm_90+): two instructions per term instead of three -- the kernel is bound by
// the atomic issue rate of the SMs (786 k scalar atomics at config 2), not by bandwidth.  Each element is still added atomically.
__device__ __forceinline__ void atomic_add3(float *o, long long cs, float vx, float vy, float vz) {
    if (cs == 1) {
        if ((reinterpret_cast<unsigned long long>(o) & 7ull) == 0ull) {
            atomicAdd(reinterpret_cast<float2 *>(o), make_float2(vx, vy));
            atomicAdd(o + 2, vz);
        } else {
            atomicAdd(o, vx);
            atomicAdd(reinterpret_cast<float2 *>(o + 1), make_float2(vy, vz));
        }
    } else {
        atomicAdd(o, vx);
        atomicAdd(o + cs, vy);
        atomicAdd(o + 2 * cs, vz);
    }
}

// warp-aggregated scatter of one term per lane (inactive lanes carry unique negative targets and zero values)
template <bool OVERWRITE>
__device__ __forceinline__ void grad_scatter(const GradParams &p, bool active, const GradTerm &t, int lane) {
    if (!OVERWRITE && active) {
        atomic_add3((t.d2 ? p.g2 : p.g1) + t.own, t.d2 ? p.cs2 : p.cs1, t.v[0], t.v[1], t.v[2]);
    }
    // (the direction is warp-uniform only if total1 % 32 == 0, so the direction bit is folded into the match key)
    const unsigned long long mkey = ((unsigned long long)t.tgt << 1) | (unsigned long long)(t.d2 ? 1 : 0);
    const unsigned int peers = __match_any_sync(0xffffffffu, mkey);
    const int leader = __ffs(peers) - 1;
    float sx = t.v[0], sy = t.v[1], sz = t.v[2];
    // the lowest lane of every group adds its peers' terms in lane order; the loop trip count is the
    // largest group size minus one (zero for clouds without shared nearest neighbours in the warp).
    unsigned int rest = (lane == leader) ? (peers & ~(1u << lane)) : 0u;
    while (__any_sync(0xffffffffu, rest != 0u)) {
        const int src = rest ? __ffs(rest) - 1 : lane;
        const float ox = __shfl_sync(0xffffffffu, t.v[0], src);
        const float oy = __shfl_sync(0xffffffffu, t.v[1], src);
        const float oz = __shfl_sync(0xffffffffu, t.v[2], src);
        if (rest) { sx += ox; sy += oy; sz += oz; rest &= rest - 1u; }
    }
    if (active && lane == leader) {
        atomic_add3((t.d2 ? p.g1 : p.g2) + t.tgt, t.d2 ? p.cs1 : p.cs2, -sx, -sy, -sz);
    }
}

// MODE 0: accumulate (own-point and scatter terms as atomics, caller-zeroed buffers)
// MODE 2 / 3: overwrite as TWO plain launches (2 = store own-point terms, 3 = scatter atomics): stream order is the barrier.
// (A single cooperative launch with a grid-wide barrier in between was measured SLOWER on B200: 11.2 us against 9.4 us for the
// two launches and 8.1 us for zero fill + MODE 0 at config 2, tools/grad_forms.py -- and it would have to wait for most of
// the GPU when several steps are in flight.  The fast path is MODE 0 on buffers that the forward kernel zero-filled.)
// RAGGED (MODE 0 only): per-pair lengths (GradRaggedParams); points at or beyond them have no term.
template <int MODE, bool RAGGED>
__global__ void __launch_bounds__(256) chamfer_grad_kernel(const std::conditional_t<RAGGED, GradRaggedParams, GradParams> p) {
    static_assert(!RAGGED || MODE == 0, "the ragged backward accumulates");
    constexpr bool OVERWRITE = MODE != 0;
    const long long nthreads = (long long)gridDim.x * blockDim.x;   // a multiple of 32
    const long long gid0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const bool active0 = gid0 < p.total;
    if (MODE == 0 && PSD_GRAD_TRIGGER_EARLY) pdl_trigger();   // the next forward launch may be scheduled as the SMs drain (it waits before its first global access)
    if constexpr (RAGGED) {
        for (long long base = gid0 - lane; base < p.total; base += nthreads) {   // warp-uniform trip count
            GradTerm t;
            t.d2 = false; t.own = 0; t.tgt = -1 - (long long)lane; t.v[0] = t.v[1] = t.v[2] = 0.f;
            const int kind = base + lane < p.total ? grad_term_ragged(p, base + lane, t) : 0;
            if (kind == 2) {   // invalid pair: NaN own row, then an inactive lane for the scatter
                atomic_add3((t.d2 ? p.g2 : p.g1) + t.own, t.d2 ? p.cs2 : p.cs1, t.v[0], t.v[1], t.v[2]);
                t.tgt = -1 - (long long)lane; t.v[0] = t.v[1] = t.v[2] = 0.f;
            }
            grad_scatter<false>(p, kind == 1, t, lane);
        }
        if (!PSD_GRAD_TRIGGER_EARLY) pdl_trigger();
        return;
    }
    GradTerm t0;
    t0.d2 = false; t0.own = 0; t0.tgt = -1 - (long long)lane; t0.v[0] = t0.v[1] = t0.v[2] = 0.f;
    if (active0) t0 = grad_term(p, gid0);
    if (MODE == 2) {
        auto store_own = [&](const GradTerm &t) {
            float *o = (t.d2 ? p.g2 : p.g1) + t.own;
            const long long csa = t.d2 ? p.cs2 : p.cs1;
            o[0] = t.v[0]; o[csa] = t.v[1]; o[2 * csa] = t.v[2];
        };
        if (active0) store_own(t0);
        for (long long gid = gid0 + nthreads; gid < p.total; gid += nthreads) store_own(grad_term(p, gid));
        return;
    }
    grad_scatter<OVERWRITE>(p, active0, t0, lane);
    for (long long base = gid0 - lane + nthreads; base < p.total; base += nthreads) {   // warp-uniform trip count
        const bool active = base + lane < p.total;
        GradTerm t;
        t.d2 = false; t.own = 0; t.tgt = -1 - (long long)lane; t.v[0] = t.v[1] = t.v[2] = 0.f;
        if (active) t = grad_term(p, base + lane);   // the second visit is served by L1 / L2
        grad_scatter<OVERWRITE>(p, active, t, lane);
    }
    if (MODE == 0 && !PSD_GRAD_TRIGGER_EARLY) pdl_trigger();
}

// loss = sum_b sums[b,0] / cnt1 + sum_b sums[b,1] / cnt2 -- the epilogue of Loss.get_chamfer_loss (loss/loss.py:36) on
// the per-cloud sums that the forward kernels accumulate; one warp, fixed summation order.
__global__ void chamfer_mean_loss_kernel(const float *__restrict__ sums, int b, float cnt1, float cnt2, float *__restrict__ out) {
    float s1 = 0.f, s2 = 0.f;
    for (int i = threadIdx.x; i < b; i += 32) { s1 += sums[2 * i]; s2 += sums[2 * i + 1]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
    if (threadIdx.x == 0) *out = __fdiv_rn(s1, cnt1) + __fdiv_rn(s2, cnt2);
}

}  // namespace psd

// ------------------------------------------------------------------------------------------------
// host launchers (called by psd_capi.cu)
// ------------------------------------------------------------------------------------------------
using namespace psd;

// test / measurement switches (process-wide, atomics: safe to flip from any thread)
static std::atomic<int> g_nn_variant{0};   // 0 = auto, 1 = FFMA kernel (this file), 3 = tensor-core kernel
static std::atomic<float *> g_tc_dbg{nullptr};   // one-shot debug dump target of the tensor-core kernel (psd_debug_tc_filter)
static std::atomic<int> g_tc_dbg_ld{0};
static std::atomic<long long *> g_tc_prof{nullptr};

bool psd_nn_tc_supported(const NNParams &p);                                               // chamfer_nn_tc.cu
cudaError_t psd_launch_nn_tc(const NNParams &p, DeviceState *ds, cudaStream_t stream, float *dbg, int dbg_ld, long long *prof, int b,
                             bool ragged, const int *len1, const int *len2);
void psd_set_tc_prof(long long *prof) { g_tc_prof.store(prof); }
cudaError_t psd_read_chamfer_stats_tc(unsigned long long *fallback, int reset);
void psd_set_tc_debug(float *dbg, int ld) { g_tc_dbg_ld.store(ld); g_tc_dbg.store(dbg); }

int psd_set_nn_variant(int v) {
    if (v == 0 || v == 1 || v == 3) return g_nn_variant.exchange(v);
    return g_nn_variant.load();
}

// layout: bit 0 = xyz1 is [B,3,N], bit 1 = xyz2 is [B,3,M] (else [B,N,3] / [B,M,3])
static inline void layout_strides(int layout, int bit, int npts, long long &ps, long long &cs) {
    if (layout & bit) { ps = 1; cs = npts; } else { ps = 3; cs = 1; }
}

cudaError_t psd_launch_chamfer_forward(const float *xyz1, const float *xyz2, int b, int n, int m, int layout,
                                       float *dist1, float *dist2, int *idx1, int *idx2, float *sums, float fs_thr,
                                       int *fs_count, int q_begin, int q_count, cudaStream_t stream, float *zero_buf,
                                       long long zero_floats, bool ragged, const int *len1, const int *len2) {
    if (zero_floats <= 0) zero_buf = nullptr;
    auto only_zero = [&]() { return zero_buf ? cudaMemsetAsync(zero_buf, 0, sizeof(float) * (size_t)zero_floats, stream) : cudaSuccess; };
    if (b <= 0 || n <= 0 || m <= 0) return only_zero();
    cudaError_t derr = cudaSuccess;
    DeviceState *ds = device_state(&derr);
    if (ds == nullptr) return derr;
    const int num_sms = ds->num_sms, max_smem = ds->max_smem;
    NNParams p;
    const int QB = kQB;
    auto fill = [&](NNDirection &D, const float *q, int nq, int qbit, const float *t, int nt, int tbit, float *dist, int *idx, int slot) {
        D.q = q; D.t = t; D.nq = nq; D.nt = nt; D.dist = dist; D.idx = idx; D.slot = slot;
        layout_strides(layout, qbit, nq, D.q_ps, D.q_cs);
        layout_strides(layout, tbit, nt, D.t_ps, D.t_cs);
        D.q_bs = 3LL * nq; D.t_bs = 3LL * nt;
        int qb0 = q_begin < 0 ? 0 : q_begin;
        if (qb0 > nq) qb0 = nq;
        int qc = (q_count < 0) ? nq - qb0 : q_count;
        if (qb0 + qc > nq) qc = nq - qb0;
        D.q_begin = qb0; D.q_count = qc;
        D.qblocks = (qc + QB - 1) / QB;
        D.ntt = 1; D.ws = nullptr;
    };
    fill(p.dir[0], xyz1, n, 1, xyz2, m, 2, dist1, idx1, 0);
    fill(p.dir[1], xyz2, m, 2, xyz1, n, 1, dist2, idx2, 1);
    const long long blocks = (long long)b * (p.dir[0].qblocks + p.dir[1].qblocks);
    if (blocks == 0) return only_zero();
    if (blocks > 0x3fffffffLL) return cudaErrorInvalidConfiguration;
    p.zero_buf = zero_buf; p.zero_floats = zero_floats;
    p.pdl_trigger = 0;
    p.blocks_dir0 = b * p.dir[0].qblocks;
    p.total_blocks = (int)blocks;
    p.sums = sums; p.fs_count = fs_count; p.fs_thr = fs_thr;
    p.tile = 0; p.flush = 0;
    // Tensor-core filter (chamfer_nn_tc.cu) for every launch of at least two units per SM.
    // Measured (tools/nn_variants.py): 41.5 vs 55.8 us at B=32 N=M=2048, 70.5 vs 105.8 us at B=64, 20.3 vs 22.5 us at
    // B=32 N=M=1024; launches of < 2 units per SM are latency-bound and stay on the FFMA kernel (8.9 vs 7.5 us at B=8 N=512).
    const int variant = g_nn_variant.load();
    if ((variant == 3 || (variant == 0 && blocks >= 2LL * num_sms)) && psd_nn_tc_supported(p)) {
        if (ragged) return psd_launch_nn_tc(p, ds, stream, nullptr, 0, nullptr, b, true, len1, len2);
        float *dbg = g_tc_dbg.exchange(nullptr);
        return psd_launch_nn_tc(p, ds, stream, dbg, g_tc_dbg_ld.load(), g_tc_prof.load(), b, false, nullptr, nullptr);
    }
    // persistent grid: one CTA per SM, each takes a contiguous range of 128-query blocks
    const int grid = blocks < num_sms ? (int)blocks : num_sms;
    const int per_cta = (int)((blocks + grid - 1) / grid);
    int tile = 1024;
    const int tmax = n > m ? n : m;
    while (tile < tmax && tile < 4096) tile *= 2;
    const size_t fixed = (size_t)tile * 16 + 2048;  // tile arrays + static shared memory + slack
    const size_t per_block = (size_t)kPerBlockBytes;
    int flush = (int)(((size_t)max_smem - fixed) / per_block);
    if (flush > per_cta) flush = per_cta;
    if (flush < 1) flush = 1;
    p.tile = tile; p.flush = flush;
    const size_t smem = (size_t)tile * 16 + (size_t)flush * per_block + 64;
    {
        std::lock_guard<std::mutex> lock(state_mutex());
        if (!ds->attr_nn) {
            cudaError_t e = cudaSuccess;
            for (auto k : {chamfer_nn_kernel<1024, false>, chamfer_nn_kernel<2048, false>, chamfer_nn_kernel<4096, false>})
                if (e == cudaSuccess) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem - 1024);
            for (auto k : {chamfer_nn_kernel<1024, true>, chamfer_nn_kernel<2048, true>, chamfer_nn_kernel<4096, true>})
                if (e == cudaSuccess) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem - 1024);
            if (e != cudaSuccess) return e;
            ds->attr_nn = true;
        }
    }
    if (ragged) {
        NNRaggedParams pr;
        static_cast<NNParams &>(pr) = p;
        pr.qlen[0] = len1; pr.tlen[0] = len2;   // direction 0: xyz1 -> xyz2
        pr.qlen[1] = len2; pr.tlen[1] = len1;
        if (tile == 1024) chamfer_nn_kernel<1024, true><<<grid, kThreads, smem, stream>>>(pr);
        else if (tile == 2048) chamfer_nn_kernel<2048, true><<<grid, kThreads, smem, stream>>>(pr);
        else chamfer_nn_kernel<4096, true><<<grid, kThreads, smem, stream>>>(pr);
        return cudaGetLastError();
    }
    if (tile == 1024) chamfer_nn_kernel<1024, false><<<grid, kThreads, smem, stream>>>(p);
    else if (tile == 2048) chamfer_nn_kernel<2048, false><<<grid, kThreads, smem, stream>>>(p);
    else chamfer_nn_kernel<4096, false><<<grid, kThreads, smem, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t psd_launch_chamfer_mean_loss(const float *sums, int b, int n, int m, float *out, cudaStream_t stream) {
    chamfer_mean_loss_kernel<<<1, 32, 0, stream>>>(sums, b, (float)((long long)b * n), (float)((long long)b * m), out);
    return cudaGetLastError();
}

// overwrite = 0: accumulate into caller-zeroed gradients (the reference's contract); 1: the gradients need no initialisation
cudaError_t psd_launch_chamfer_backward(const float *xyz1, const float *xyz2, float *gradxyz1, float *gradxyz2,
                                        const float *graddist1, const float *graddist2, const int *idx1, const int *idx2,
                                        int b, int n, int m, int layout, int overwrite, cudaStream_t stream, const float *upstream,
                                        bool ragged, const int *len1, const int *len2) {
    if (b <= 0 || (n <= 0 && m <= 0)) return cudaSuccess;
    if (n <= 0 || m <= 0) {   // one cloud is empty: no pair exists, nothing to accumulate
        if (!overwrite) return cudaSuccess;
        cudaError_t e = n > 0 ? cudaMemsetAsync(gradxyz1, 0, sizeof(float) * 3 * (size_t)b * n, stream) : cudaSuccess;
        if (e == cudaSuccess && m > 0) e = cudaMemsetAsync(gradxyz2, 0, sizeof(float) * 3 * (size_t)b * m, stream);
        return e;
    }
    GradParams p;
    p.upstream = upstream; p.cnt1 = (float)((long long)b * n); p.cnt2 = (float)((long long)b * m);
    p.xyz1 = xyz1; p.xyz2 = xyz2; p.g1 = gradxyz1; p.g2 = gradxyz2; p.gd1 = graddist1; p.gd2 = graddist2;
    p.idx1 = idx1; p.idx2 = idx2; p.b = b; p.n = n; p.m = m;
    p.total1 = (long long)b * n;
    p.total = (long long)b * (n + m);
    layout_strides(layout, 1, n, p.ps1, p.cs1);
    layout_strides(layout, 2, m, p.ps2, p.cs2);
    const long long blocks = (p.total + 255) / 256;
    if (blocks > 0x7fffffffLL) return cudaErrorInvalidConfiguration;
    if (ragged) {   // (accumulate form only)
        GradRaggedParams pr;
        static_cast<GradParams &>(pr) = p;
        pr.len1 = len1; pr.len2 = len2;
        chamfer_grad_kernel<0, true><<<(unsigned int)blocks, 256, 0, stream>>>(pr);
        return cudaGetLastError();
    }
    if (!overwrite) {
        // A PLAIN launch: as a programmatic dependent of the forward kernel the 512 small CTAs are placed as the forward's CTAs
        // exit -- eight per SM on the first SMs to drain, none on the last ones -- and the kernel runs on half of the GPU
        // (38.9 instead of 38.3 us per step).  It still triggers its own successor (the next forward launch, one CTA per SM).
        chamfer_grad_kernel<0, false><<<(unsigned int)blocks, 256, 0, stream>>>(p);
        return cudaGetLastError();
    }
    // two plain launches: stream order is the barrier between the stores and the atomics
    chamfer_grad_kernel<2, false><<<(unsigned int)blocks, 256, 0, stream>>>(p);
    chamfer_grad_kernel<3, false><<<(unsigned int)blocks, 256, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t psd_read_chamfer_stats(unsigned long long *fallback, int reset) {
    cudaError_t e = cudaMemcpyFromSymbol(fallback, g_fallback_queries, sizeof(unsigned long long));
    if (e != cudaSuccess) return e;
    if (reset) {
        const unsigned long long z = 0;
        e = cudaMemcpyToSymbol(g_fallback_queries, &z, sizeof(z));
        if (e != cudaSuccess) return e;
    }
    unsigned long long fg = 0;
    e = psd_read_chamfer_stats_tc(&fg, reset);
    *fallback += fg;
    return e;
}
