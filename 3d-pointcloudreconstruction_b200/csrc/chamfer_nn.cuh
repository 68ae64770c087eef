// chamfer_nn.cuh -- launch description shared by the two Chamfer NN forward kernels
// (chamfer.cu: FFMA kernel for small launches; chamfer_nn_tc.cu: tensor-core kernel).
#pragma once
#include <type_traits>

#include "psd_common.cuh"

namespace psd {

constexpr int kQ = 4;             // queries per lane
constexpr int kQB = 32 * kQ;      // queries per block (every warp of the CTA holds the same 128 queries)
constexpr int kChunk = 16;        // targets per filter chunk
constexpr float kBig = 1e30f;     // padding value for w[]; larger than any admissible filter value
constexpr float kLimit = 1e18f;   // |t-c|^2, |q-c|^2 above this (or NaN) route the query to the exact scan
constexpr int kRefTile = 512;     // the reference's tile (chamfer3D.cu:13), only observable with NaN inputs

struct NNDirection {
    const float *q;      // query cloud base
    const float *t;      // target cloud base
    long long q_ps, q_cs, q_bs;  // query strides in floats: point, component, batch
    long long t_ps, t_cs, t_bs;
    float *dist;         // [B, nq]
    int *idx;            // [B, nq]
    int nq, nt;
    int q_begin, q_count;  // query slice handled by this launch
    int qblocks;           // 128-query blocks per cloud for this direction
    int slot;              // 0/1: column in sums[B,2] / fs_count[B,2]
    // tensor-core kernel only: the targets are cut into ntt tiles of 2048 (a unit = one query block x one tile).  With
    // ntt > 1 every unit merges its exact (distance, index) into ws[cloud*nq + j] with a 64-bit atomicMin and a
    // finalize kernel unpacks dist / idx; with ntt == 1 (ws == nullptr) the kernel writes dist / idx itself.
    int ntt;
    unsigned long long *ws;
};

struct NNParams {
    NNDirection dir[2];
    int blocks_dir0;    // blocks belonging to dir[0]
    int total_blocks;
    int tile;           // targets per shared-memory tile (multiple of 1024)
    int flush;          // blocks whose partial results fit in shared memory between two resolve phases
    float *sums;        // optional [B,2]
    int *fs_count;      // optional [B,2]
    float fs_thr;
    // optional: a buffer the launch also zero-fills (the gradient buffers of the backward that follows on the stream), so
    // that a training step needs no separate memset
    float *zero_buf;
    long long zero_floats;
    // tensor-core kernel: signal near the end of a CTA that the next kernel on the stream may be launched (psd_common.cuh,
    // PSD_PDL).  Off for launches that share the GPU with other launches (psd_chamfer_tc_ctas): a successor CTA that is resident
    // and waiting for its predecessor would hold an SM that another stream's launch could use.
    int pdl_trigger;
};

// Ragged launches (the RAGGED instantiations of both NN kernels): pair c takes part with the first qlen[d][c] queries and
// tlen[d][c] targets of direction d (device int [B]; NULL = the padded size).  The work grid stays that of the padded sizes.
struct NNRaggedParams : NNParams {
    const int *qlen[2], *tlen[2];
};

// participating queries / targets of pair `cloud` in direction d; a pair with a length outside [1, padded size] in either
// cloud is invalid and gets qn = tn = 0
__device__ __forceinline__ bool ragged_lengths(const NNRaggedParams &p, int d, int cloud, int &qn, int &tn) {
    const NNDirection &D = p.dir[d];
    qn = p.qlen[d] ? __ldg(p.qlen[d] + cloud) : D.nq;
    tn = p.tlen[d] ? __ldg(p.tlen[d] + cloud) : D.nt;
    const bool ok = qn >= 1 && qn <= D.nq && tn >= 1 && tn <= D.nt;
    if (!ok) { qn = 0; tn = 0; }
    return ok;
}

// grid-wide zero fill of p.zero_buf, a few stores per thread, issued before anything else in the forward kernels
__device__ __forceinline__ void zero_fill(const NNParams &p) {
    if (p.zero_buf == nullptr) return;
    const long long nth = (long long)gridDim.x * blockDim.x, t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (((reinterpret_cast<unsigned long long>(p.zero_buf) & 15ull) == 0ull) && (p.zero_floats & 3) == 0) {
        float4 *z = reinterpret_cast<float4 *>(p.zero_buf);
        for (long long i = t0; i < (p.zero_floats >> 2); i += nth) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
        for (long long i = t0; i < p.zero_floats; i += nth) p.zero_buf[i] = 0.f;
    }
}

// exact squared distance of query (x1,y1,z1) to target k of a cloud with generic strides
__device__ __forceinline__ float exact_d(const float *__restrict__ tb, long long tps, long long tcs, int k, float x1,
                                         float y1, float z1) {
    const float *tp = tb + (long long)k * tps;
    return sqdist_exact(__ldg(tp) - x1, __ldg(tp + tcs) - y1, __ldg(tp + 2 * tcs) - z1);
}

}  // namespace psd
