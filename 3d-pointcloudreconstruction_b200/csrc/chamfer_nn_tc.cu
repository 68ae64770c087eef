// chamfer_nn_tc.cu -- Chamfer NN forward with the FILTER on the 5th-generation tensor cores (tcgen05 / TMEM).
//
// Same contract and the same exactness scheme as chamfer.cu (reference: metric/chamfer3D/chamfer3D.cu:12-154):
// dist/idx always come from the reference's exact formula; a filter only decides where to look.  Here the filter
//     a_k = |t_k - c|^2 - 2 (q - c).(t_k - c)            ( = |t_k - q|^2 - |q - c|^2 )
// is a [128 queries] x [256 targets] x K=16 FP16 GEMM per tile: ONE tcgen05.mma.kind::f16 issued by one thread.
// fp32-class accuracy comes from (1) a per-cloud power-of-two scale s that brings max|t-c| into [0.5,1) -- exact in
// fp32, keeps every term inside the fp16 exponent range -- and (2) splitting every operand into two fp16 terms
// (hi + lo, 22 significand bits) and |t-c|^2 into three, laid out along K so that the cross terms line up:
//     A row (query) : [qh qh ql]x [qh qh ql]y [qh qh ql]z  1  1  1  0 0 0 0      q' = -2 s (q - c) = qh + ql
//     B row (target): [th tl th]x [th tl th]y [th tl th]z  w1 w2 w3 0 0 0 0      t' = s (t - c) = th + tl, |t'|^2 = w1+w2+w3
// (products of two 11-bit significands are exact in the fp32 accumulator; the dropped ql*tl terms and the split
// residues are bounded by 3*2^-22 |q'||t'|).  Measured on B200 (tools/ubench_umma.cu): kind::f16 M128 N128 K16 issues
// every 64 cycles, kind::tf32 K8 only every 96, independent of the shared-memory layout -- hence fp16 and one
// instruction per tile (N = 256: 128 cycles).  Accumulators live in TMEM (2 buffers of 256 columns).
//
// One persistent CTA per SM, three concurrent roles (no CTA-wide barrier in the steady state):
//   * warps 0-7   SCANNERS: warp w reads TMEM lanes 32*(w%4).. (one thread = one query row, so the running minimum
//                 needs no cross-lane traffic) with tcgen05.ld.32x32b.x32, 64 columns at a time, and keeps per 32-target
//                 chunk (best chunk minimum, its chunk id, second best): 16 min instructions + 6 ALU ops per 32 pairs
//                 instead of 96 FFMA + 16 FMNMX3 in the FFMA kernel.  ALTERNATING (PSD_TC_SCAN_ALT, default): warp w takes
//                 all 256 columns of the tiles of TMEM buffer w/4, i.e. every other tile, so that the two warps of a
//                 sub-partition work half a period apart; the A/B build PSD_TC_SCAN_ALT=0 is the lock-step form (columns
//                 128*(w/4).. of EVERY tile: both warps wait, load and reduce at the same time) -- 35.0 vs 33.0 us.
//   * warp  8     MMA issuer: waits for operands (ready mbarrier) and a free TMEM buffer (empty mbarrier), issues one
//                 tcgen05.mma per tile and commits it to the buffer's full mbarrier.
//   * warps 9-15  HELPERS: stage the operands two units ahead (raw coordinates -> scaled split fp16, K-major core
//                 matrices, double-buffered A and B), and resolve the unit the scanners just finished: merge the
//                 partial results, margin test, exact rescan of the best chunk from raw targets kept in shared
//                 memory, fused loss-sum / F-score epilogue.  Queries that fail the margin test go to a per-CTA
//                 list and take an exact full scan, one warp per query, by all warps at the end (raw targets from
//                 shared memory when their cloud is still resident).
// A unit is a block of 128 queries of one cloud/direction; a CTA owns a contiguous range of units.
#include <cuda_fp16.h>
#include "chamfer_nn.cuh"
#include "psd_device.h"

namespace psd {
namespace tc {

#ifndef PSD_TC_SCAN_WARPS
#define PSD_TC_SCAN_WARPS 8                     // 8 (two per sub-partition, 128 columns each); A/B builds: 16 (four, 64 columns each)
#endif
#ifndef PSD_TC_SETMAXNREG
#define PSD_TC_SETMAXNREG (PSD_TC_SCAN_WARPS == 16)
#endif
#ifndef PSD_TC_STAGE_FIRST
#define PSD_TC_STAGE_FIRST 0   // A/B build: helpers stage the operands of unit ul + 2 BEFORE they resolve unit ul.  The MMA thread's operand waits
#endif                         // go away (4.7 k -> 2.1 k cycles in CTAs that build a second B operand), the launch time does not move (32.8 vs 32.4 us)
#ifndef PSD_TC_TAIL_FAST
#define PSD_TC_TAIL_FAST 1     // deferred exact scans at the end of the kernel: one-barrier form when every warp has at most one part of one query
#endif
#ifndef PSD_TC_ALT_UNROLL
#define PSD_TC_ALT_UNROLL 2
#endif
#ifndef PSD_TC_SCAN_ALT
#define PSD_TC_SCAN_ALT 1      // scanner warp (r, c) takes ALL 256 columns of the tiles of TMEM buffer c (the two warps of a
#endif                         // sub-partition work half a period apart instead of sharing every tile in lock-step)
constexpr int kScanWarps = PSD_TC_SCAN_WARPS;   // warp w reads TMEM lanes 32*(w%4).., column group w/4 of every tile
constexpr int kMmaWarp = kScanWarps;            // warp index of the MMA issuer
#ifndef PSD_TC_HELP_WARPS
#define PSD_TC_HELP_WARPS 7
#endif
constexpr int kHelpWarps = PSD_TC_HELP_WARPS;                   // 24 (16) warps in all, 80 (128) registers per thread at launch
constexpr int kHelpThreads = kHelpWarps * 32;
constexpr int kHelp0 = (kScanWarps + 1) * 32;   // first helper thread
constexpr int kThreadsTC = (kScanWarps + 1 + kHelpWarps) * 32;   // 768
constexpr int kColGroups = kScanWarps / 4;      // column groups of a tile (one scanner warp per lane quarter and group)
#ifndef PSD_TC_TILE_N
#define PSD_TC_TILE_N 256
#endif
constexpr int kAltUnroll = PSD_TC_ALT_UNROLL;
constexpr int kTileN = PSD_TC_TILE_N;           // targets per MMA tile = TMEM buffer width (columns): 256, or 128 (four buffers) in A/B builds
constexpr int kBufs = 512 / kTileN;             // TMEM buffers: all 512 columns.  Two 256-column tiles beat four 128-column
                                                // ones (37.4 vs 41.5 us at B=32, N=M=2048): the mbarrier / tcgen05.commit round
                                                // trip per tile (~300-400 cycles, tools/ubench_pipe.cu) is paid half as often
static_assert(kTileN == 256 || ((kTileN == 128 || kTileN == 160) && PSD_TC_SCAN_ALT), "tile width");
// TMEM buffer and mbarrier phase of the g-th tile of a CTA's stream (kBufs = 2 or 4: masks; 3 buffers of 160 columns: mul-shift division)
__device__ __forceinline__ int div3(int g) { return (int)(((unsigned long long)(unsigned)g * 0xAAAAAAABull) >> 33); }
__device__ __forceinline__ int buf_of(int g) { return kBufs == 3 ? g - 3 * div3(g) : (g & (kBufs - 1)); }
__device__ __forceinline__ int phase_of(int g) { return kBufs == 3 ? (div3(g) & 1) : ((g >> (kBufs == 4 ? 2 : 1)) & 1); }
constexpr int kBRows = ((2048 + kTileN - 1) / kTileN) * kTileN;   // rows of a B operand buffer: kMaxT rounded up to whole tiles
[[maybe_unused]] constexpr int kGroupCols = PSD_TC_SCAN_ALT ? kTileN : kTileN / kColGroups; // columns per tile and scanner warp: kGroupCols / 64 tmem_ld64_wait each
constexpr int kCh = 32;                         // targets per filter chunk (one tcgen05.ld.x32)
constexpr int kMaxT = 2048;                     // targets resident in shared memory (B operand: 32 B per target)
constexpr float kPadW = 32768.0f;               // padding |t'|^2 (fp16-exact), above every admissible filter value
constexpr float kQMax = 4096.0f;                // scaled |q-c| above this sends the query to the exact scan: keeps |a| <= 3 + 3.5*kQMax < kPadW

// shared-memory carve-up (bytes)
constexpr int kOffB = 0;                                  // [2][kMaxT/8][2][8][16 B]
constexpr int kOffA = kOffB + 2 * kBRows * 32;            // [2][16][2][8][16 B]
constexpr int kOffRaw = kOffA + 2 * kQB * 32;             // [2][3][kMaxT] raw target coordinates (SoA), by B buffer
constexpr int kOffPart = kOffRaw + 2 * 3 * kMaxT * 4;     // [2][kColGroups][3][128]
constexpr int kOffSq = kOffPart + 2 * kColGroups * 3 * kQB * 4;    // [3][3][128] raw queries, by unit mod 3
constexpr int kFbCap = 512;                               // deferred exact-scan list (entries: unit << 8 | query)
constexpr int kOffFb = kOffSq + 3 * 3 * kQB * 4;
constexpr int kOffFq = kOffFb + kFbCap * 4;                // [3][kFbCap] raw coordinates of the deferred queries
constexpr int kOffStat = kOffFq + 3 * kFbCap * 4;             // [32] wmax, [32] bad, [32] cmax (one per warp), [2] group resident in sraw[i]
constexpr int kOffBar = kOffStat + 3 * 32 * 4 + 16;       // 8 mbarriers (8-byte aligned)
constexpr int kOffMisc = kOffBar + 16 * 8;                // tmem base, nfb, abort
constexpr int kSmemTC = kOffMisc + 64;
static_assert(kOffBar % 8 == 0 && kOffA % 128 == 0 && kOffRaw % 16 == 0 && kOffPart % 16 == 0 && kHelpWarps <= 8 && kThreadsTC / 32 <= 32 &&
              kSmemTC <= 227 * 1024, "shared-memory carve-up");

__device__ unsigned long long g_fallback_queries_tc = 0ull;

// ---- PTX wrappers -------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok;
}
#ifndef PSD_TC_SPIN
#define PSD_TC_SPIN 0          // A/B builds: bit 0 = the MMA thread busy-polls (test_wait) instead of try_wait, bit 1 = the scanners too
#endif
__device__ __forceinline__ uint32_t mbar_test_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{ .reg .pred p; mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok;
}
// Bounded wait: a protocol bug must not hang the GPU.  After ~10 s (2e10 cycles: far beyond any legitimate wait, also
// under compute-sanitizer) the kernel traps: the stream gets a sticky launch failure, so the next CUDA call of the
// wrappers (and torch's next synchronise) raises instead of returning garbage dist / idx.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, volatile int *abort_flag) {
    if (mbar_try_wait(bar, parity)) return;
    long long t0 = 0;
    for (unsigned spins = 1;; ++spins) {
        if (mbar_try_wait(bar, parity)) return;   // try_wait suspends the warp in hardware for a bounded time
        if ((spins & 63u) == 0u) {
            if (*abort_flag) return;
            const long long now = clock64();
            if (t0 == 0) t0 = now;
            if (now - t0 > 20000000000LL) { *abort_flag = 1; __trap(); }
        }
    }
}
#ifndef PSD_TC_POLL_LANE0
#define PSD_TC_POLL_LANE0 0
#endif
// busy-polling form of mbar_wait (A/B builds)
__device__ __forceinline__ void mbar_spin(uint32_t bar, uint32_t parity, volatile int *abort_flag) {
    long long t0 = 0;
    for (unsigned spins = 1;; ++spins) {
        if (mbar_test_wait(bar, parity)) return;
        if ((spins & 1023u) == 0u) {
            if (*abort_flag) return;
            const long long now = clock64();
            if (t0 == 0) t0 = now;
            if (now - t0 > 20000000000LL) { *abort_flag = 1; __trap(); }
        }
    }
}
// warp-wide wait: every lane polls, or (A/B build) lane 0 polls and the warp reconverges behind it
__device__ __forceinline__ void mbar_wait_warp(uint32_t bar, uint32_t parity, volatile int *abort_flag) {
    if (PSD_TC_POLL_LANE0) {
        if ((threadIdx.x & 31) == 0) mbar_wait(bar, parity, abort_flag);
        __syncwarp();
    } else if (PSD_TC_SPIN & 2) {
        mbar_spin(bar, parity, abort_flag);
    } else {
        mbar_wait(bar, parity, abort_flag);
    }
}
__device__ __forceinline__ void cp_async4(void *smem_dst, const float *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void help_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kHelpThreads) : "memory"); }
// x -> (hi, lo) fp16 pair with hi + lo = x up to 2^-22 |x| (or 2^-25 absolute in the subnormal range)
__device__ __forceinline__ void split_h(float x, unsigned short &hi, unsigned short &lo) {
    const __half h = __float2half_rn(x);
    const __half l = __float2half_rn(x - __half2float(h));
    hi = __half_as_ushort(h); lo = __half_as_ushort(l);
}
// the same for two values at once with the PACKED conversion (F2FP.F16.F32.PACK_AB: one full-rate instruction for two
// values; the scalar F2F.F16.F32 runs on the slow conversion path and bounded the operand build: 9 per target row)
__device__ __forceinline__ void split_h2(float a, float b, unsigned short &ah, unsigned short &al, unsigned short &bh, unsigned short &bl) {
    const __half2 h = __floats2half2_rn(a, b);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
    ah = __half_as_ushort(__low2half(h)); bh = __half_as_ushort(__high2half(h));
    al = __half_as_ushort(__low2half(l)); bl = __half_as_ushort(__high2half(l));
}
__device__ __forceinline__ uint32_t pack2(unsigned short a, unsigned short b) { return (uint32_t)a | ((uint32_t)b << 16); }
// K-major, no swizzle: core matrix = 8 rows x 16 B (128 contiguous bytes, 8 fp16 per row); LBO = distance between
// the two core matrices of the K=16 slice (128 B), SBO = distance between 8-row groups (256 B).  Version 1 (sm_100).
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3ffffu) >> 4) | ((uint64_t)(128u >> 4) << 16) | ((uint64_t)(256u >> 4) << 32) |
           (1ull << 46);
}
// kind::f16, D = F32, A/B = F16 (format 0), both K-major, M = 128, N = kTileN
constexpr uint32_t kIdesc = (1u << 4) | ((uint32_t)(kTileN >> 3) << 17) | ((128u >> 4) << 24);
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile("{ .reg .pred p; setp.ne.b32 p, %4, 0; tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p; }"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(kIdesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// two tcgen05.ld of 32 consecutive columns each of this thread's TMEM lane (a, then b) AND the wait for them in ONE
// asm statement: the destination registers are written asynchronously until tcgen05.wait::ld, so the compiler must
// never see them as defined in between (a spill or a move there would read stale data).
__device__ __forceinline__ void tmem_ld64_wait(uint32_t taddr, uint32_t (&a)[32], uint32_t (&b)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%64];\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%65];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]), "=r"(a[4]), "=r"(a[5]), "=r"(a[6]), "=r"(a[7]), "=r"(a[8]), "=r"(a[9]), "=r"(a[10]), "=r"(a[11]), "=r"(a[12]), "=r"(a[13]), "=r"(a[14]), "=r"(a[15]), "=r"(a[16]), "=r"(a[17]), "=r"(a[18]), "=r"(a[19]), "=r"(a[20]), "=r"(a[21]), "=r"(a[22]), "=r"(a[23]), "=r"(a[24]), "=r"(a[25]), "=r"(a[26]), "=r"(a[27]), "=r"(a[28]), "=r"(a[29]), "=r"(a[30]), "=r"(a[31]),
          "=r"(b[0]), "=r"(b[1]), "=r"(b[2]), "=r"(b[3]), "=r"(b[4]), "=r"(b[5]), "=r"(b[6]), "=r"(b[7]), "=r"(b[8]), "=r"(b[9]), "=r"(b[10]), "=r"(b[11]), "=r"(b[12]), "=r"(b[13]), "=r"(b[14]), "=r"(b[15]), "=r"(b[16]), "=r"(b[17]), "=r"(b[18]), "=r"(b[19]), "=r"(b[20]), "=r"(b[21]), "=r"(b[22]), "=r"(b[23]), "=r"(b[24]), "=r"(b[25]), "=r"(b[26]), "=r"(b[27]), "=r"(b[28]), "=r"(b[29]), "=r"(b[30]), "=r"(b[31])
        : "r"(taddr), "r"(taddr + 32u)
        : "memory");
}
// Software-pipelined form (PSD_TC_PIPE_LD): ONE tcgen05.ld of 32 columns, and the wait as a separate statement, so that the load
// of the next 32 columns is in flight while the previous 32 are reduced (two 32-register landing zones: the same 64 registers
// as the combined form).  The landing registers are outputs of the load statement and in/outputs of the wait statement: the
// compiler has no reason to touch them in between (nothing else is live but the other landing zone and a few scalars; the
// SASS is checked for moves out of a landing zone between LDTM and the wait, and the GPU tests compare every bit).
#ifndef PSD_TC_PIPE_LD
#define PSD_TC_PIPE_LD 0       // measured: 35.8 us against 35.1 us for the combined load + wait (profiles/r2_tc_ab.txt)
#endif
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&a)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]), "=r"(a[4]), "=r"(a[5]), "=r"(a[6]), "=r"(a[7]), "=r"(a[8]), "=r"(a[9]), "=r"(a[10]), "=r"(a[11]), "=r"(a[12]), "=r"(a[13]), "=r"(a[14]), "=r"(a[15]), "=r"(a[16]), "=r"(a[17]), "=r"(a[18]), "=r"(a[19]), "=r"(a[20]), "=r"(a[21]), "=r"(a[22]), "=r"(a[23]), "=r"(a[24]), "=r"(a[25]), "=r"(a[26]), "=r"(a[27]), "=r"(a[28]), "=r"(a[29]), "=r"(a[30]), "=r"(a[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_wait_ld(uint32_t (&a)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]), "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]),
                   "+r"(a[16]), "+r"(a[17]), "+r"(a[18]), "+r"(a[19]), "+r"(a[20]), "+r"(a[21]), "+r"(a[22]), "+r"(a[23]), "+r"(a[24]), "+r"(a[25]), "+r"(a[26]), "+r"(a[27]), "+r"(a[28]), "+r"(a[29]), "+r"(a[30]), "+r"(a[31])
                 :: "memory");
}
// minimum of 32 filter values: 15 FMNMX3 + 1 FMNMX, four independent chains
__device__ __forceinline__ float min32(const uint32_t (&r)[32]) {
    float m[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        m[i] = fmin3(__uint_as_float(r[8 * i]), __uint_as_float(r[8 * i + 1]), __uint_as_float(r[8 * i + 2]));
        m[i] = fmin3(m[i], __uint_as_float(r[8 * i + 3]), __uint_as_float(r[8 * i + 4]));
        m[i] = fmin3(m[i], __uint_as_float(r[8 * i + 5]), __uint_as_float(r[8 * i + 6]));
    }
    float v = fmin3(m[0], m[1], m[2]);
    v = fmin3(v, m[3], __uint_as_float(r[7]));
    v = fmin3(v, __uint_as_float(r[15]), __uint_as_float(r[23]));
    return fminf(v, __uint_as_float(r[31]));
}

struct Unit {
    int d, cloud, qblock;
    int ttile, t0, nt;     // target tile of the unit: index, first target, number of targets (<= kMaxT)
    int qn, tn, inval;     // ragged launches only: the pair's participating queries / targets (0 / 0 for an invalid pair)
};
template <class P> constexpr bool kRagged = std::is_same_v<P, NNRaggedParams>;
// Ragged launches: the pair's lengths (reload) and the unit's target count.  A unit whose query block or target tile starts
// at or beyond the lengths, or whose pair is invalid, gets nt = 0: the MMA thread, the scanners and the helpers all derive
// their tile count from nt, so every role skips it by the same rule and the barrier phases stay in step.
__device__ __forceinline__ void ragged_unit(const NNRaggedParams &p, Unit &u, bool reload) {
    const NNDirection &D = p.dir[u.d];
    if (reload) u.inval = !ragged_lengths(p, u.d, u.cloud, u.qn, u.tn);
    u.nt = min(kMaxT, u.tn - u.t0);
    if (u.nt < 0 || D.q_begin + u.qblock * kQB >= u.qn) u.nt = 0;
}
// unit order inside a direction: cloud, target tile, query block -- consecutive units of a CTA share a B operand
template <class P>
__device__ __forceinline__ Unit decode_unit(const P &p, int blk) {
    Unit u;
    u.d = blk >= p.blocks_dir0 ? 1 : 0;
    const NNDirection &D = p.dir[u.d];
    const int bid = u.d ? blk - p.blocks_dir0 : blk;
    const int per_cloud = D.qblocks * D.ntt;
    u.cloud = bid / per_cloud;
    const int rem = bid - u.cloud * per_cloud;
    u.ttile = D.ntt == 1 ? 0 : rem / D.qblocks;   // (single-tile launches: one division less per decode)
    u.qblock = rem - u.ttile * D.qblocks;
    u.t0 = u.ttile * kMaxT;
    u.nt = min(kMaxT, D.nt - u.t0);
    if constexpr (kRagged<P>) ragged_unit(p, u, true);
    return u;
}
// unit blk -> unit blk + 1 without the integer divisions of decode_unit (they cost the single MMA thread ~500 cycles per unit)
template <class P>
__device__ __forceinline__ void advance_unit(const P &p, Unit &u, int blk_next) {
    if (blk_next == p.blocks_dir0) { u = decode_unit(p, blk_next); return; }   // direction switch
    const NNDirection &D = p.dir[u.d];
    if (++u.qblock == D.qblocks) {
        u.qblock = 0;
        const int cloud = u.cloud;
        if (++u.ttile == D.ntt) { u.ttile = 0; ++u.cloud; }
        u.t0 = u.ttile * kMaxT;
        u.nt = min(kMaxT, D.nt - u.t0);
        if constexpr (kRagged<P>) ragged_unit(p, u, u.cloud != cloud);
    } else if constexpr (kRagged<P>) {
        ragged_unit(p, u, false);
    }
}
// last query of the unit's cloud that its query loads may touch (they are clamped to it); ragged: the last participating one
template <class P>
__device__ __forceinline__ int query_last(const P &p, const Unit &u) {
    const NNDirection &D = p.dir[u.d];
    if constexpr (kRagged<P>) return max(min(D.q_begin + D.q_count, u.qn) - 1, 0);
    return D.q_begin + D.q_count - 1;
}
__device__ __forceinline__ int group_of(const NNParams &p, const Unit &u) { return u.d * 0x40000000 + u.cloud * p.dir[u.d].ntt + u.ttile; }
__device__ __forceinline__ const float *targets_of(const NNParams &p, const Unit &u) {
    const NNDirection &D = p.dir[u.d];
    return D.t + (long long)u.cloud * D.t_bs + (long long)u.t0 * D.t_ps;
}
// store one query's exact result: directly, or merged over the target tiles through the 64-bit workspace
__device__ __forceinline__ void store_result(const NNDirection &D, const Unit &u, int j, float dist, int idx_local) {
    if (D.ws) atomicMin(D.ws + (long long)u.cloud * D.nq + j, pack_key(dist, u.t0 + idx_local));
    else { D.dist[(long long)u.cloud * D.nq + j] = dist; D.idx[(long long)u.cloud * D.nq + j] = u.t0 + idx_local; }
}

struct Frame {        // filter frame of one unit (identical in every helper thread)
    float cx, cy, cz, cs, wmax;   // centre, power-of-two scale, max |t'|^2
    int bad, bsel;                // non-finite target seen; B / raw-target buffer
};

// Exact full scan for a query on the deferred list.  fallback_scan: one warp scans part `part` of `nsplit` of the targets
// and returns the packed (distance, index) minimum (identical in every lane); raw targets come from shared memory when the
// query's cloud/direction is still resident in sraw, else from global memory.  fallback_write: one thread stores the
// result.  Reference semantics incl. NaN: within a 512-target tile the first element is taken unconditionally and NaN
// never replaces or is replaced (chamfer3D.cu:36); a tile result replaces the running result only if strictly smaller (:126).
struct FbQuery {
    Unit u;
    int j, nt, res;
    float x1, y1, z1;
    bool nan_possible;
    const float *bx, *by, *bz;   // generic view of the targets: component base pointers and point stride
    long long ps;
};
template <class P>
__device__ __forceinline__ FbQuery fallback_query(const P &p, int blk_begin, int e, const float *sraw, const int *s_rawgroup,
                                                  const float *fq) {   // fq: the query's coordinates in the list (x, y, z kFbCap apart)
    FbQuery q;
    q.u = decode_unit(p, blk_begin + ((e & 0x3fffffff) >> 8));
    const NNDirection &D = p.dir[q.u.d];
    q.nt = q.u.nt;
    q.j = D.q_begin + q.u.qblock * kQB + (e & 0xff);
    q.x1 = fq[0]; q.y1 = fq[kFbCap]; q.z1 = fq[2 * kFbCap];   // (kept at resolve time: no global round trip in the tail)
    q.nan_possible = ((e >> 30) & 1) || !(fabsf(q.x1) < 1e18f) || !(fabsf(q.y1) < 1e18f) || !(fabsf(q.z1) < 1e18f);
    const int grp = group_of(p, q.u);
    q.res = s_rawgroup[0] == grp ? 0 : (s_rawgroup[1] == grp ? 1 : -1);
    if (q.res >= 0) { q.bx = sraw + (q.res * 3) * kMaxT; q.by = q.bx + kMaxT; q.bz = q.by + kMaxT; q.ps = 1; }
    else { q.bx = targets_of(p, q.u); q.by = q.bx + D.t_cs; q.bz = q.by + D.t_cs; q.ps = D.t_ps; }
    return q;
}
__device__ __forceinline__ unsigned long long fallback_scan(const FbQuery &q, int part, int nsplit, int lane) {
    const float x1 = q.x1, y1 = q.y1, z1 = q.z1;
    const int nt = q.nt;
    unsigned long long key = ~0ull;
    if (q.res >= 0 && !q.nan_possible) {
        // resident cloud, finite data: 4 targets per lane and step straight from the SoA copy (3 x LDS.128), running
        // (distance, index) minimum in index order with strict '<' -- no NaN can occur
        float dbest = 3.0e38f;
        int ibest = 0x7fffffff;
        for (int k0 = 4 * lane + 128 * part; k0 < nt; k0 += 128 * nsplit) {
            const float4 xa = *reinterpret_cast<const float4 *>(q.bx + k0), ya = *reinterpret_cast<const float4 *>(q.by + k0),
                         za = *reinterpret_cast<const float4 *>(q.bz + k0);
            const float d0 = sqdist_exact(xa.x - x1, ya.x - y1, za.x - z1), d1 = sqdist_exact(xa.y - x1, ya.y - y1, za.y - z1);
            const float d2 = sqdist_exact(xa.z - x1, ya.z - y1, za.z - z1), d3 = sqdist_exact(xa.w - x1, ya.w - y1, za.w - z1);
            if (d0 < dbest) { dbest = d0; ibest = k0; }
            if (k0 + 1 < nt && d1 < dbest) { dbest = d1; ibest = k0 + 1; }
            if (k0 + 2 < nt && d2 < dbest) { dbest = d2; ibest = k0 + 2; }
            if (k0 + 3 < nt && d3 < dbest) { dbest = d3; ibest = k0 + 3; }
        }
        if (ibest != 0x7fffffff) key = pack_key(dbest, ibest);
    } else {
        for (int kb = lane + 256 * part; kb < nt; kb += 256 * nsplit) {
            float dd[8], dts[8];
#pragma unroll
            for (int q8 = 0; q8 < 8; ++q8) {
                const long long k = min(kb + q8 * 32, nt - 1);
                dd[q8] = sqdist_exact(q.bx[k * q.ps] - x1, q.by[k * q.ps] - y1, q.bz[k * q.ps] - z1);
                const long long kt = k & ~(long long)(kRefTile - 1);
                dts[q8] = q.nan_possible ? sqdist_exact(q.bx[kt * q.ps] - x1, q.by[kt * q.ps] - y1, q.bz[kt * q.ps] - z1) : 0.f;
            }
#pragma unroll
            for (int q8 = 0; q8 < 8; ++q8) {
                const int k = kb + q8 * 32;
                if (k < nt && !(dd[q8] != dd[q8]) && !(dts[q8] != dts[q8])) {
                    const unsigned long long kk = pack_key(dd[q8], k);
                    key = kk < key ? kk : key;
                }
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = shfl_xor_u64(key, o);
        key = other < key ? other : key;
    }
    return key;
}
__device__ __forceinline__ void fallback_write(const NNParams &p, const FbQuery &q, unsigned long long key) {
    const NNDirection &D = p.dir[q.u.d];
    if (D.ws) {   // merged over the target tiles; the finalize kernel applies the tile-0 NaN rule and the epilogues
        if (key != ~0ull) atomicMin(D.ws + (long long)q.u.cloud * D.nq + q.j, key + (unsigned long long)q.u.t0);
        return;
    }
    const float d0 = sqdist_exact(q.bx[0] - q.x1, q.by[0] - q.y1, q.bz[0] - q.z1);
    float dres;
    int ires;
    if (d0 != d0) { dres = d0; ires = 0; }   // tile 0 poisoned: stays NaN, index 0
    else { dres = __uint_as_float((unsigned int)(key >> 32)); ires = (int)(key & 0xffffffffu); }
    D.dist[(long long)q.u.cloud * D.nq + q.j] = dres;
    D.idx[(long long)q.u.cloud * D.nq + q.j] = ires;
    if (p.sums) atomicAdd(p.sums + q.u.cloud * 2 + D.slot, dres);
    if (p.fs_count && dres < p.fs_thr) atomicAdd(p.fs_count + q.u.cloud * 2 + D.slot, 1);
}
// one warp per query (used by the helpers when the list has to be flushed in the middle of the kernel)
template <class P>
__device__ __forceinline__ void run_fallbacks(const P &p, int blk_begin, const int *fb_list, const float *fb_q, int nfb, int wi, int nw,
                                              int lane, const float *sraw, const int *s_rawgroup) {
    for (int fi = wi; fi < nfb; fi += nw) {
        const FbQuery q = fallback_query(p, blk_begin, fb_list[fi], sraw, s_rawgroup, fb_q + fi);
        const unsigned long long key = fallback_scan(q, 0, 1, lane);
        if (lane == 0) fallback_write(p, q, key);
    }
}

// DBG: instrumented build -- dumps every filter value to dbg[(unit*128 + row) * dbg_ld + target] when dbg != nullptr
// (calibration / bring-up) and writes phase clocks to prof (tools/tc_phase_clocks.py) when prof != nullptr.
// RAGGED: per-pair lengths (NNRaggedParams); the units of the padded grid that lie beyond them do no search.
template <bool DBG, bool RAGGED>
__global__ void __launch_bounds__(kThreadsTC, 1) chamfer_nn_tc_kernel(const std::conditional_t<RAGGED, NNRaggedParams, NNParams> p,
                                                                     float *dbg, int dbg_ld, long long *prof) {
    extern __shared__ __align__(128) unsigned char smem[];
    float *sraw = reinterpret_cast<float *>(smem + kOffRaw);
    float *part = reinterpret_cast<float *>(smem + kOffPart);
    float *sq = reinterpret_cast<float *>(smem + kOffSq);
    int *fb_list = reinterpret_cast<int *>(smem + kOffFb);
    float *fb_q = reinterpret_cast<float *>(smem + kOffFq);
    int *s_nfb = reinterpret_cast<int *>(smem + kOffMisc) + 1;
    float *s_wstat = reinterpret_cast<float *>(smem + kOffStat);
    int *s_bstat = reinterpret_cast<int *>(smem + kOffStat) + 32;
    float *s_cstat = reinterpret_cast<float *>(smem + kOffStat) + 64;
    int *s_rawgroup = reinterpret_cast<int *>(smem + kOffStat) + 96;   // cloud/direction whose raw targets sraw[i] holds
    uint32_t *s_tmem = reinterpret_cast<uint32_t *>(smem + kOffMisc);
    volatile int *s_abort = reinterpret_cast<volatile int *>(smem + kOffMisc) + 2;
    const uint32_t sB_addr = smem_u32(smem + kOffB), sA_addr = smem_u32(smem + kOffA);
    const uint32_t bar0 = smem_u32(smem + kOffBar);
    const uint32_t bar_full = bar0, bar_empty = bar0 + 8 * kBufs, bar_ready = bar0 + 16 * kBufs, bar_part = bar_ready + 16;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = gridDim.x;
    const int blk_begin = (int)(((long long)blockIdx.x * p.total_blocks) / G);
    const int blk_end = (int)(((long long)(blockIdx.x + 1) * p.total_blocks) / G);
    const int nunits = blk_end - blk_begin;
    // optional phase clocks (tools/tc_phase_clocks.py): 64 slots per CTA
    long long *pf = (DBG && prof) ? prof + (long long)blockIdx.x * 64 : nullptr;
    auto stamp = [&](int slot) { if (DBG && pf && slot < 56) pf[slot] = clock64(); };
    // timeline of CTA 0 (tools/tc_timeline.py): 8 rows of 64 tiles behind the per-CTA slots -- the prof buffer holds gridDim.x * 64 + 512
    // entries.  Rows: 0 MMA issued, 1 committed; scanner warp 0 (even tiles): 2 tile seen full, 3 buffer released, 4 reduction done;
    // scanner warp 4 (odd tiles): 5, 6, 7 the same (lock-step build: warp 0 only, 6 / 7 = first pair of loads issued / landed).
    long long *tl = (DBG && prof && blockIdx.x == 0) ? prof + (long long)gridDim.x * 64 : nullptr;
    auto tstamp = [&](int rowi, int g) { if (DBG && tl && g < 64) tl[rowi * 64 + g] = clock64(); };
    if (tid == 0) stamp(0);

    if (tid == 0) {
        for (int i = 0; i < kBufs; ++i) { mbar_init(bar_full + 8 * i, 1); mbar_init(bar_empty + 8 * i, PSD_TC_SCAN_ALT ? 4 : kScanWarps); }
        for (int i = 0; i < 2; ++i) { mbar_init(bar_ready + 8 * i, 1); mbar_init(bar_part + 8 * i, kScanWarps); }
        *s_abort = 0;
        *s_nfb = 0;
        s_rawgroup[0] = -1; s_rawgroup[1] = -1;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kMmaWarp) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;
    if (tid == 0) stamp(1);
    pdl_wait();      // everything above is set-up without global accesses: it overlaps the previous kernel's drain (PSD_PDL)
    zero_fill(p);

    // The B operand of a cloud/direction is built from its raw targets in sraw[bsel] (already landed and visible to the team) in
    // two steps.  frame_of: centre and power-of-two scale (one pass over the targets by a team of tn threads -- tt = index in
    // the team, tw = warp index in the team -- with the team's own barrier).  build_rows: the scaled split fp16 rows of targets
    // [k0, k1) (rows beyond nt are padding), accumulating the thread's max |t'|^2 and its bad flag.
    auto frame_of = [&](int nt, int bsel, int tt, int tn, int tw, auto &&team_bar, Frame &fr, int &bad) {
        const float *rx = sraw + (bsel * 3) * kMaxT, *ry = rx + kMaxT, *rz = ry + kMaxT;
        float cx, cy, cz;
        {   // centre of the filter frame: mean of up to 8 evenly spaced targets (any value is correct)
            float sx = 0.f, sy = 0.f, sz = 0.f;
            const int ns = nt < 8 ? nt : 8;
            const int step = nt >> 3;
#pragma unroll
            for (int s8 = 0; s8 < 8; ++s8) {
                if (s8 < ns) {
                    const int k = nt < 8 ? s8 : s8 * step;
                    sx += rx[k]; sy += ry[k]; sz += rz[k];
                }
            }
            const float inv = 1.0f / (float)ns;
            cx = sx * inv; cy = sy * inv; cz = sz * inv;
        }
        // extent around the centre -> power-of-two scale
        float cmax = 0.f;
        bad = 0;
#pragma unroll 4
        for (int k = tt; k < nt; k += tn) {
            const float ax = fabsf(rx[k] - cx), ay = fabsf(ry[k] - cy), az = fabsf(rz[k] - cz);
            bad |= !(ax < 1e18f) | !(ay < 1e18f) | !(az < 1e18f);
            cmax = fmaxf(cmax, fmaxf(ax, fmaxf(ay, az)));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
        if (lane == 0) s_cstat[tw] = cmax;
        team_bar();
        cmax = 0.f;
        for (int w = 0; w < tn / 32; ++w) cmax = fmaxf(cmax, s_cstat[w]);
        float cs;
        {
            int e = (int)((__float_as_uint(cmax) >> 23) & 0xffu);   // biased exponent; 0 for cmax == 0 / subnormal
            // Clouds smaller than 2^-60: the reference's own distances are subnormal there and round on an ABSOLUTE grid
            // (2^-149), which the relative margin below does not cover -> every query of the cloud takes the exact scan.
            bad |= e < 67;
            e = e < 27 ? 27 : (e > 227 ? 227 : e);                   // keep s within [2^-101, 2^99]
            cs = cmax > 0.f ? __uint_as_float((uint32_t)(253 - e) << 23) : 1.0f;   // 2^(126 - e): s*cmax in [0.5, 1)
        }
        fr.cx = cx; fr.cy = cy; fr.cz = cz; fr.cs = cs; fr.bsel = bsel;
        fr.wmax = -1.f;   // statistics are picked up later (pick_stats)
    };
    auto build_rows = [&](int nt, const Frame &fr, int k0, int k1, int tt, int tn, float &wmax, int &bad) {
        const float *rx = sraw + (fr.bsel * 3) * kMaxT, *ry = rx + kMaxT, *rz = ry + kMaxT;
        unsigned char *sBb = smem + kOffB + fr.bsel * (kBRows * 32);
#pragma unroll 2
        for (int k = k0 + tt; k < k1; k += tn) {
            uint4 v0 = make_uint4(0u, 0u, 0u, 0u), v1 = v0;
            if (k < nt) {
                const float x = (rx[k] - fr.cx) * fr.cs, y = (ry[k] - fr.cy) * fr.cs, z = (rz[k] - fr.cz) * fr.cs;
                const float w = __fmaf_rn(z, z, __fmaf_rn(x, x, y * y));
                bad |= !(w < 4.0f);
                wmax = fmaxf(wmax, w);
                unsigned short xh, xl, yh, yl, zh, zl, w1, w2;
                split_h2(x, y, xh, xl, yh, yl);
                split_h2(z, w, zh, zl, w1, w2);          // |t'|^2 = w1 + w2 + w3: the first two terms are w's own (hi, lo)
                const float wr2 = (w - __half2float(__ushort_as_half(w1))) - __half2float(__ushort_as_half(w2));
                const unsigned short w3 = __half_as_ushort(__float2half_rn(wr2));
                v0 = make_uint4(pack2(xh, xl), pack2(xh, yh), pack2(yl, yh), pack2(zh, zl));
                v1 = make_uint4(pack2(zh, w1), pack2(w2, w3), 0u, 0u);
            } else {
                v1.x = pack2(0, __half_as_ushort(__float2half_rn(kPadW)));
            }
            unsigned char *dst = sBb + (k >> 3) * 256 + (k & 7) * 16;
            *reinterpret_cast<uint4 *>(dst) = v0;
            *reinterpret_cast<uint4 *>(dst + 128) = v1;
        }
    };
    auto publish_stats = [&](int tw, float wmax, int bad) {   // per-warp statistics for pick_stats (after the team's next barrier)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            wmax = fmaxf(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
            bad |= __shfl_xor_sync(0xffffffffu, bad, o);
        }
        if (lane == 0) { s_wstat[tw] = wmax; s_bstat[tw] = bad; }
    };
    // whole operand by one team (steady state: the helpers)
    auto build_b = [&](int nt, int bsel, int tt, int tn, int tw, auto &&team_bar, Frame &fr) {
        int bad = 0;
        float wmax = 0.f;
        frame_of(nt, bsel, tt, tn, tw, team_bar, fr, bad);
        build_rows(nt, fr, 0, ((nt + kTileN - 1) / kTileN) * kTileN, tt, tn, wmax, bad);
        publish_stats(tw, wmax, bad);
    };
    auto pick_stats = [&](int nwarps, Frame &fr) {
        float wmax = 0.f;
        int bad = 0;
        for (int w = 0; w < nwarps; ++w) { wmax = fmaxf(wmax, s_wstat[w]); bad |= s_bstat[w]; }
        fr.wmax = wmax; fr.bad = bad;
    };

    // ---------------- prologue: the B operand of the first unit is built by the WHOLE CTA (everybody is idle anyway).
    // (Building it tile by tile behind the scan -- helpers produce 256 rows, signal, the MMA thread and the scanners start -- was
    // measured slower, 36.9 vs 35.5 us: a tile by 224 threads with its own proxy fence + barrier + arrive costs ~1.1 k cycles,
    // more than the scan of a tile, so the first unit ran at the producers' pace.)
    Frame fr0 = {0.f, 0.f, 0.f, 1.f, 0.f, 0, 0};
    int group0 = -1;
    float pq1 = 0.f, pq2 = 0.f, pq3 = 0.f;   // helpers, threads < 128: raw query of the unit being staged, loaded early
    if (nunits > 0) {
        const Unit u = decode_unit(p, blk_begin);
        const NNDirection &D = p.dir[u.d];
        group0 = group_of(p, u);
        const float *__restrict__ tb = targets_of(p, u);
#pragma unroll
        for (int comp = 0; comp < 3; ++comp)
            for (int k = tid; k < u.nt; k += kThreadsTC) cp_async4(sraw + comp * kMaxT + k, tb + k * D.t_ps + comp * D.t_cs);
        if (tid >= kHelp0 && tid - kHelp0 < kQB) {
            // the queries of unit 0 travel together with its targets: one global round trip on the critical path, not two
            int j = D.q_begin + u.qblock * kQB + (tid - kHelp0);
            const int q_last = query_last(p, u);
            j = j < q_last ? j : q_last;
            const float *qp = D.q + (long long)u.cloud * D.q_bs + j * D.q_ps;
            pq1 = __ldg(qp); pq2 = __ldg(qp + D.q_cs); pq3 = __ldg(qp + 2 * D.q_cs);
        }
        if (tid == 0) stamp(6);
        cp_async_wait_all();
        __syncthreads();
        if (tid == 0) stamp(7);
        build_b(u.nt, 0, tid, kThreadsTC, warp, [] { __syncthreads(); }, fr0);
        fence_async_smem();
        __syncthreads();
        pick_stats(kThreadsTC / 32, fr0);
        if (tid == 0) s_rawgroup[0] = group0;
    }
    if (tid == 0) stamp(5);

    // Register budget (24 warps x 80 at launch = 61 440): the scanners need their 64 landing registers and little else, the
    // helpers' resolve wants more than 80 -- 16 x 32 x 72 + 8 x 32 x 96 = 61 440.  Whole warpgroups (4 consecutive warps)
    // change together: 0-15 scanners, 16-23 MMA issuer + helpers; everybody returns to 80 before the common tail.
    if (warp < kScanWarps) {
        if (PSD_TC_SETMAXNREG) asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
        // ================================================= scanners
        const int r = warp & 3, c = warp >> 2;       // TMEM lane quarter; tile parity (alternating form) / column group of every tile (lock-step)
        const int row = r * 32 + lane;
        const uint32_t tlane = tmem_base + ((uint32_t)(r * 32) << 16);
        int g0 = 0;
        long long a59 = 0;
        Unit u = decode_unit(p, blk_begin);
        for (int ul = 0; ul < nunits; ++ul) {
            if (ul > 0) advance_unit(p, u, blk_begin + ul);
            const int ntiles = (u.nt + kTileN - 1) / kTileN;
            // A unit without tiles (ragged launches) has no MMA to pace the scanners: without this wait they could park its
            // partials in the slot of unit ul - 2 and arrive on that slot's barrier before the helpers have resolved unit
            // ul - 2.  Its operands are staged (bar_ready) only after that resolve.
            if (RAGGED && ntiles == 0) mbar_wait_warp(bar_ready + 8 * (ul & 1), (ul >> 1) & 1, s_abort);
            float best = kBig, second = kBig;
            int bchunk = 0;
            auto chunk = [&](const uint32_t (&v)[32], int cid) {
                const float m = min32(v);
                second = fminf(second, fmaxf(best, m));
                const bool lt = m < best;
                best = fminf(best, m);
                bchunk = lt ? cid : bchunk;
            };
            // Alternating form (default): warp (r, c) visits the tiles whose index in the CTA's stream is c mod 2 and reduces all of
            // their columns, four pairs of loads per visit; the TMEM buffer goes back to the MMA thread as soon as the last pair has
            // landed.  The two warps of a sub-partition are then about half a period apart -- one reduces while the other loads or
            // waits for its buffer's next tile -- instead of waiting, loading and reducing at the same time.  Lock-step form
            // (PSD_TC_SCAN_ALT=0): every warp takes its column group of EVERY tile.
#if PSD_TC_SCAN_ALT
            static_assert(kScanWarps == 8, "alternating scanners: two warps per sub-partition, warp c takes the tiles that are c mod 2");
            for (int t = (g0 ^ c) & 1; t < ntiles; t += 2) {
                const int gg = g0 + t;
                const int b = buf_of(gg);
                const long long w0 = DBG ? clock64() : 0;
                mbar_wait_warp(bar_full + 8 * b, phase_of(gg), s_abort);
                if (DBG) a59 += clock64() - w0;
                if (DBG && r == 0 && lane == 0) tstamp(2 + 3 * c, gg);
                tc_fence_after();
                const uint32_t ta = tlane + (uint32_t)(b * kTileN);
                const int cid0 = (t * kTileN) / kCh;
                uint32_t ra[32], rb[32];
                constexpr int kPairs = kTileN / 64;
                constexpr bool kTail32 = (kTileN % 64) == 32;   // 160-column tiles: two pairs of loads + one single
                auto release = [&]() {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_empty + 8 * b);
                    if (DBG && r == 0 && lane == 0) tstamp(3 + 3 * c, gg);
                };
#pragma unroll kAltUnroll
                for (int l = 0; l < kPairs; ++l) {   // (fully unrolled at 256 columns, ptxas hoists all eight loads and spills the landing zones)
                    tmem_ld64_wait(ta + 64 * l, ra, rb);
                    if (!kTail32 && l == kPairs - 1) release();
                    if (DBG && dbg) {
                        float *o = dbg + ((long long)(blk_begin + ul) * kQB + row) * dbg_ld + t * kTileN + 64 * l;
#pragma unroll
                        for (int i = 0; i < 32; ++i) { o[i] = __uint_as_float(ra[i]); o[32 + i] = __uint_as_float(rb[i]); }
                    }
                    chunk(ra, cid0 + 2 * l);
                    chunk(rb, cid0 + 2 * l + 1);
                }
                if (kTail32) {
                    tmem_ld32(ta + 64 * kPairs, ra);
                    tmem_wait_ld(ra);
                    release();
                    if (DBG && dbg) {
                        float *o = dbg + ((long long)(blk_begin + ul) * kQB + row) * dbg_ld + t * kTileN + 64 * kPairs;
#pragma unroll
                        for (int i = 0; i < 32; ++i) o[i] = __uint_as_float(ra[i]);
                    }
                    chunk(ra, cid0 + 2 * kPairs);
                }
                if (DBG && tl && r == 0) { if (__float_as_uint(best) != 0x7fc00123u && lane == 0) tstamp(4 + 3 * c, gg); }
            }
#else
            for (int t = 0; t < ntiles; ++t) {
                const int gg = g0 + t;
                const int b = buf_of(gg);
                const long long w0 = DBG ? clock64() : 0;
                mbar_wait_warp(bar_full + 8 * b, phase_of(gg), s_abort);
                if (DBG) a59 += clock64() - w0;
                if (DBG && tid == 0) tstamp(2, gg);
                tc_fence_after();
                const int col0 = c * kGroupCols;                       // first column of this warp's share of the tile
                const uint32_t ta = tlane + (uint32_t)(b * kTileN + col0);
                const int cid0 = (t * kTileN + col0) / kCh;            // chunk id of the first 32 columns
                uint32_t ra[32], rb[32];
                if (PSD_TC_PIPE_LD && !(DBG && dbg)) {
                    // 32 columns at a time, the next load in flight behind the reduction of the previous one
                    constexpr int kLd = kGroupCols / 32;
                    tmem_ld32(ta, ra);
                    tmem_wait_ld(ra);
#pragma unroll
                    for (int l = 0; l < kLd; l += 2) {
                        tmem_ld32(ta + 32 * (l + 1), rb);
                        chunk(ra, cid0 + l);
                        tmem_wait_ld(rb);
                        if (l + 2 < kLd) {
                            tmem_ld32(ta + 32 * (l + 2), ra);
                        } else {
                            // every column of this warp's share is in registers: hand the TMEM buffer back before the last min work
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(bar_empty + 8 * b);
                        }
                        chunk(rb, cid0 + l + 1);
                        if (l + 2 < kLd) tmem_wait_ld(ra);
                    }
                } else {
#pragma unroll
                    for (int l = 0; l < kGroupCols / 64; ++l) {
                        if (DBG && tl && l == 0 && tid == 0) tstamp(6, gg);
                        tmem_ld64_wait(ta + 64 * l, ra, rb);
                        if (DBG && tl && l == 0 && warp == 0) {   // (the compare makes the stamp wait for the landed registers)
                            if (ra[0] != 0x7fc00123u && rb[31] != 0x7fc00123u && lane == 0) tstamp(7, gg);
                        }
                        if (l == kGroupCols / 64 - 1) {
                            // every column of this warp's share is in registers: hand the TMEM buffer back before the remaining min work
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(bar_empty + 8 * b);
                            if (DBG && tid == 0) tstamp(3, gg);
                        }
                        if (DBG && dbg) {
                            float *o = dbg + ((long long)(blk_begin + ul) * kQB + row) * dbg_ld + t * kTileN + col0 + 64 * l;
#pragma unroll
                            for (int i = 0; i < 32; ++i) { o[i] = __uint_as_float(ra[i]); o[32 + i] = __uint_as_float(rb[i]); }
                        }
                        chunk(ra, cid0 + 2 * l);
                        chunk(rb, cid0 + 2 * l + 1);
                    }
                }
                if (DBG && tl && warp == 0) { if (__float_as_uint(best) != 0x7fc00123u && lane == 0) tstamp(4, gg); }
            }
#endif
            g0 += ntiles;
            {   // park this warp's partial results (double-buffered by unit parity) and tell the helpers
                float *pp = part + ((ul & 1) * kColGroups + c) * 3 * kQB;
                pp[row] = best; pp[kQB + row] = second; reinterpret_cast<int *>(pp)[2 * kQB + row] = bchunk;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_part + 8 * (ul & 1));
            if (tid == 0) stamp(8 + ul * 6);
        }
        if (DBG && pf && tid == 0) pf[59] = a59;
        if (PSD_TC_SETMAXNREG) asm volatile("setmaxnreg.inc.sync.aligned.u32 80;");
    } else if (warp == kMmaWarp) {
        if (PSD_TC_SETMAXNREG) asm volatile("setmaxnreg.inc.sync.aligned.u32 96;");
        // ================================================= MMA issuer: ONE thread runs the whole loop (an elected
        // issue inside a warp-wide loop costs ~270 cycles per tile on B200, a single-thread loop 64: tools/ubench_umma.cu)
        if (lane == 0) {
            int g = 0, grp = -1, bsel = 1;
            long long a56 = 0, a57 = 0, a61 = 0, a62 = 0;   // DBG: wait / issue cycle totals
            Unit u = decode_unit(p, blk_begin);
            for (int ul = 0; ul < nunits; ++ul) {
                if (ul > 0) advance_unit(p, u, blk_begin + ul);
                const int ntiles = (u.nt + kTileN - 1) / kTileN;
                if (group_of(p, u) != grp) { grp = group_of(p, u); bsel ^= 1; }
                long long w0 = DBG ? clock64() : 0;
                mbar_wait(bar_ready + 8 * (ul & 1), (ul >> 1) & 1, s_abort);
                if (DBG) a56 += clock64() - w0;
                tc_fence_after();
                const uint64_t adesc = umma_desc(sA_addr + (uint32_t)(ul & 1) * (kQB * 32));
                uint64_t bdesc = umma_desc(sB_addr + (uint32_t)bsel * (kBRows * 32));
                for (int t = 0; t < ntiles; ++t, ++g) {
                    const int b = buf_of(g);
                    w0 = DBG ? clock64() : 0;
                    if (PSD_TC_SPIN & 1) mbar_spin(bar_empty + 8 * b, phase_of(g) ^ 1, s_abort);
                    else mbar_wait(bar_empty + 8 * b, phase_of(g) ^ 1, s_abort);
                    if (DBG) a57 += clock64() - w0;
                    tc_fence_after();
                    const long long w1 = DBG ? clock64() : 0;
                    if (DBG && tl && g < 64) tl[g] = w1;
                    umma_f16(tmem_base + (uint32_t)(b * kTileN), adesc, bdesc, 0u);
                    const long long w2 = DBG ? clock64() : 0;
                    umma_commit(bar_full + 8 * b);
                    if (DBG) { const long long w3 = clock64(); a61 += w2 - w1; a62 += w3 - w2; if (tl && g < 64) tl[64 + g] = w3; }
                    bdesc += (uint64_t)((kTileN * 32) >> 4);   // next 128 targets: start-address field, 16-byte units
                }
            }
            if (DBG && pf) { pf[56] = a56; pf[57] = a57; pf[58] = clock64(); pf[61] = a61; pf[62] = a62; }
        }
        __syncwarp();
        if (PSD_TC_SETMAXNREG) asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
    } else {
        if (PSD_TC_SETMAXNREG) asm volatile("setmaxnreg.inc.sync.aligned.u32 96;");
        // ================================================= helpers
        const int ht = tid - kHelp0, hw = warp - (kScanWarps + 1);
        int st_group = group0, st_bsel = 0;  // cloud/direction of the most recently staged B operand; its buffer
        Frame fr_st = fr0;                   // frame of the most recently staged unit
        bool need_b = false;

        // does staging unit ul replace the B operand?  (uniform)
        auto stage_changes_group = [&](const Unit &u) { return group_of(p, u) != st_group; };
        // stage, part 1: put the global loads of unit ul in flight -- its 128 raw queries into registers and, if its
        // cloud/direction is not the staged one, its raw targets into sraw[other buffer] by cp.async.
        auto stage_issue = [&](int ul, const Unit &u) {
            const NNDirection &D = p.dir[u.d];
            if (ht < kQB && ul > 0) {   // (unit 0's queries were loaded in the prologue)
                int j = D.q_begin + u.qblock * kQB + ht;
                const int q_last = query_last(p, u);
                j = j < q_last ? j : q_last;
                const float *qp = D.q + (long long)u.cloud * D.q_bs + j * D.q_ps;
                pq1 = __ldg(qp); pq2 = __ldg(qp + D.q_cs); pq3 = __ldg(qp + 2 * D.q_cs);
            }
            const int group = group_of(p, u);
            need_b = group != st_group;
            if (need_b) {
                st_group = group;
                st_bsel ^= 1;
                const int nt = u.nt;
                const float *__restrict__ tb = targets_of(p, u);
                const long long tps = D.t_ps, tcs = D.t_cs;
                float *rx = sraw + (st_bsel * 3) * kMaxT;
#pragma unroll
                for (int comp = 0; comp < 3; ++comp)
                    for (int k = ht; k < nt; k += kHelpThreads) cp_async4(rx + comp * kMaxT + k, tb + k * tps + comp * tcs);
            }
        };
        // stage, part 2: build the operands of unit ul in shared memory and signal the MMA warp.
        auto stage_finish = [&](int ul, const Unit &u) {
            if (need_b) {
                cp_async_wait_all();
                help_bar();   // every helper's raw targets have landed
                build_b(u.nt, st_bsel, ht, kHelpThreads, hw, [] { help_bar(); }, fr_st);
                if (ht == 0) s_rawgroup[st_bsel] = st_group;
            }
            if (ht < kQB) {
                float *sqp = sq + (ul % 3) * 3 * kQB;
                sqp[ht] = pq1; sqp[kQB + ht] = pq2; sqp[2 * kQB + ht] = pq3;
                const float sc = -2.0f * fr_st.cs;
                const float x = (pq1 - fr_st.cx) * sc, y = (pq2 - fr_st.cy) * sc, z = (pq3 - fr_st.cz) * sc;
                unsigned short xh, xl, yh, yl, zh, zl, uh, ul_;
                split_h2(x, y, xh, xl, yh, yl);
                split_h2(z, 0.f, zh, zl, uh, ul_);
                const unsigned short one = 0x3c00;
                unsigned char *dst = smem + kOffA + (ul & 1) * (kQB * 32) + (ht >> 3) * 256 + (ht & 7) * 16;
                *reinterpret_cast<uint4 *>(dst) = make_uint4(pack2(xh, xh), pack2(xl, yh), pack2(yh, yl), pack2(zh, zh));
                *reinterpret_cast<uint4 *>(dst + 128) = make_uint4(pack2(zl, one), pack2(one, one), 0u, 0u);
            }
            fence_async_smem();
            help_bar();
            if (ht == 0) mbar_arrive(bar_ready + 8 * (ul & 1));
            if (fr_st.wmax < 0.f) pick_stats(kHelpWarps, fr_st);
        };

        // resolve unit ul.  Warp hw owns the queries [hw*kQW, hw*kQW + kQW) of the unit:
        //   A  lane = query: merge the two scanner partials, margin test
        //   B  4 lanes per query: exact rescan of the best chunk (32 targets) from the raw targets in shared memory
        //   C  queries that fail the margin test go to the deferred list (exact full scan at the end of the kernel)
        constexpr int kQW = (kQB + kHelpWarps - 1) / kHelpWarps;   // 19
        auto resolve = [&](int ul, const Unit &u, const Frame &fr) {
            const NNDirection &D = p.dir[u.d];
            const int nt = u.nt;
            const float *pp = part + (ul & 1) * kColGroups * 3 * kQB;
            const float *sqp = sq + (ul % 3) * 3 * kQB;
            const float *rx = sraw + (fr.bsel * 3) * kMaxT, *ry = rx + kMaxT, *rz = ry + kMaxT;
            const int q0 = hw * kQW;
            const int nqw = min(kQW, kQB - q0);
            // ---- A
            const int ql = q0 + (lane < nqw ? lane : 0);
            const int j = D.q_begin + u.qblock * kQB + ql;
            // (ragged: a unit without targets -- a tile beyond the pair's targets in multi-tile mode -- has nothing to search)
            const bool live = lane < nqw && j < D.q_begin + D.q_count && (!RAGGED || (j < u.qn && u.nt > 0));
            float b1 = kBig, b2 = kBig;
            int bc = 0;
#pragma unroll
            for (int w = 0; w < kColGroups; ++w) {
                const float v = pp[w * 3 * kQB + ql];
                b2 = fminf(b2, fminf(pp[w * 3 * kQB + kQB + ql], fmaxf(b1, v)));
                if (v < b1) { b1 = v; bc = reinterpret_cast<const int *>(pp)[w * 3 * kQB + 2 * kQB + ql]; }
            }
            const float x1 = sqp[ql], y1 = sqp[kQB + ql], z1 = sqp[2 * kQB + ql];
            const float ux = (x1 - fr.cx) * fr.cs, uy = (y1 - fr.cy) * fr.cs, uz = (z1 - fr.cz) * fr.cs;   // scaled frame
            const float qq = __fmaf_rn(uz, uz, __fmaf_rn(ux, ux, uy * uy));
            // Filter error bound (u = 2^-24).  RELATIVE part E_r = 15u*S: frame 2u, |t'|^2 3u, operand splits 6u
            // (3*2^-22 |q'||t'| and |q'||t'| <= S/2), tensor-core accumulation 4u (measured total on B200: <= 4.1u,
            // tools/tc_calibrate.py).  ABSOLUTE part: the lo term of a split is an fp16 SUBNORMAL whenever |x| < 1/4
            // (2^-12 |x| < 2^-14), so hi + lo = x only up to 2^-25 per coordinate (and |t'|^2's three terms up to 2^-25):
            // E_a <= 2^-25 (sqrt(3) (|q'| + |t'|) + 1) with |q'| = 2|u|, |t'| <= |u| + rho for every target that can compete.
            // The reference's argmin lies in the best chunk if second > best + 2 E_r + 10u*S + 2 E_a:
            //   S  = (|u| + max|t'|)^2 bounds every target,
            //   S' = (2|u| + rho)^2 bounds the targets that can compete (within rho of the query),
            //   margin = 40u min(S, S') + 2^-24 (1 + 5.2|u| + 1.74 rho)       [coded with 25 % slack on the absolute part].
            // Without the absolute part a query close to the frame centre (S' ~ 1e-5) trusted filter values whose fp16 operand
            // error was 100x its margin: found by tests/test_gpu_tc_hypothesis.py, reproduced on the CPU by
            // tools/tc_filter_model.py (6 591 wrong chunks in 129 k adversarial queries without the term, 0 with it; the
            // exact-scan fallback rate on U[0,1)^3 is unchanged).
            const float qn = sqrtf(qq);
            const float rr = qn + sqrtf(fr.wmax);
            const float S = rr * rr;
            const float rho = sqrtf(fmaxf(b1 + qq, 0.f) + 2.0e-6f * S);
            const float r2 = 2.0f * qn + rho;
            const float Seff = fminf(S, r2 * r2);
            const float margin = __fmaf_rn(Seff, 2.5e-6f, 1.5e-7f * (0.5f + __fmaf_rn(2.6f, qn, 0.9f * rho)));
            const bool ok = live && !fr.bad && (qn < kQMax) && (b2 > b1 + margin);
            float ws = 0.f;   // fused epilogue accumulators of this lane
            int wc = 0;
            if constexpr (RAGGED) {
                // rows past the pair's query length, and every row of an invalid pair: dist 0 (NaN), idx -1, counted nowhere
                // (the NaN goes into the pair's sums); the multi-tile mode leaves them to the finalize kernel
                if (lane < nqw && j < D.q_begin + D.q_count && !live && D.ws == nullptr) {
                    const float dz = u.inval ? __int_as_float(0x7fc00000) : 0.f;
                    D.dist[(long long)u.cloud * D.nq + j] = dz;
                    D.idx[(long long)u.cloud * D.nq + j] = -1;
                    ws += dz;
                }
            }
            if (DBG && ht == 0) stamp(12 + ul * 6);
            // ---- B
#pragma unroll
            for (int it = 0; it < (kQW * 4 + 31) / 32; ++it) {
                const int lt = it * 32 + lane;
                const int qi = lt >> 2, sub = lt & 3;          // qi < 24: a valid source lane
                const bool okq = __shfl_sync(0xffffffffu, (int)ok, qi) != 0;
                const int bcq = __shfl_sync(0xffffffffu, bc, qi);
                const float xq = __shfl_sync(0xffffffffu, x1, qi), yq = __shfl_sync(0xffffffffu, y1, qi),
                            zq = __shfl_sync(0xffffffffu, z1, qi);
                const int jq = __shfl_sync(0xffffffffu, j, qi);
                int k0 = bcq * kCh + sub * 8;
                const bool act = okq && k0 < nt;
                k0 = act ? k0 : 0;
                const float4 xa = *reinterpret_cast<const float4 *>(rx + k0), xb = *reinterpret_cast<const float4 *>(rx + k0 + 4);
                const float4 ya = *reinterpret_cast<const float4 *>(ry + k0), yb = *reinterpret_cast<const float4 *>(ry + k0 + 4);
                const float4 za = *reinterpret_cast<const float4 *>(rz + k0), zb = *reinterpret_cast<const float4 *>(rz + k0 + 4);
                const float tx[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
                const float ty[8] = {ya.x, ya.y, ya.z, ya.w, yb.x, yb.y, yb.z, yb.w};
                const float tz[8] = {za.x, za.y, za.z, za.w, zb.x, zb.y, zb.z, zb.w};
                float dbest = 3.0e38f;
                int ibest = 0x7fffffff;
                if (act) {
                    dbest = sqdist_exact(tx[0] - xq, ty[0] - yq, tz[0] - zq);
                    ibest = k0;
#pragma unroll
                    for (int i = 1; i < 8; ++i) {
                        const float dv = sqdist_exact(tx[i] - xq, ty[i] - yq, tz[i] - zq);
                        if (k0 + i < nt && dv < dbest) { dbest = dv; ibest = k0 + i; }
                    }
                }
                // quad merge: smaller distance wins, equal distances -> lower index (sub-ranges are index-ordered)
#pragma unroll
                for (int o = 1; o <= 2; o <<= 1) {
                    const float od = __shfl_xor_sync(0xffffffffu, dbest, o);
                    const int oi = __shfl_xor_sync(0xffffffffu, ibest, o);
                    if (od < dbest || (od == dbest && oi < ibest)) { dbest = od; ibest = oi; }
                }
                if (okq && sub == 0) {
                    store_result(D, u, jq, dbest, ibest);
                    ws += dbest;
                    wc += dbest < p.fs_thr ? 1 : 0;
                }
            }
            if (DBG && ht == 0) stamp(13 + ul * 6);
            // ---- C: the exact full scan of a query that failed the margin test is deferred to the end of the kernel
            if (live && !ok) {
                const int slot = atomicAdd(s_nfb, 1);
                fb_list[slot] = (ul << 8) | ql | (fr.bad ? (1 << 30) : 0);
                fb_q[slot] = x1; fb_q[kFbCap + slot] = y1; fb_q[2 * kFbCap + slot] = z1;
            }
            if ((p.sums != nullptr || p.fs_count != nullptr) && D.ws == nullptr) {   // fused epilogues, one atomic per warp
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    ws += __shfl_xor_sync(0xffffffffu, ws, o);
                    wc += __shfl_xor_sync(0xffffffffu, wc, o);
                }
                if (lane == 0) {
                    if (p.sums) atomicAdd(p.sums + u.cloud * 2 + D.slot, ws);
                    if (p.fs_count && wc) atomicAdd(p.fs_count + u.cloud * 2 + D.slot, wc);
                }
            }
        };

        Frame f0 = fr_st, f1 = fr_st;     // frames of unit ul and ul + 1
        Unit u0 = decode_unit(p, blk_begin), u1 = u0, u2 = u0;   // units ul, ul + 1, ul + 2 (advanced without divisions)
        if (nunits > 0) { stage_issue(0, u0); stage_finish(0, u0); f0 = fr_st; }
        if (nunits > 1) { advance_unit(p, u1, blk_begin + 1); stage_issue(1, u1); stage_finish(1, u1); f1 = fr_st; }
        u2 = u1;
        if (ht == 0) stamp(2);
        long long a60 = 0;
        for (int ul = 0; ul < nunits; ++ul) {
            // Loads of unit ul+2 go in flight before the resolve work.  Its raw targets may only be prefetched here when
            // their buffer is not the one resolve(ul) still reads: units ul and ul+1 of the same cloud/direction.
            const bool stage_next = ul + 2 < nunits;
            bool issued = false;
            if (stage_next) {
                advance_unit(p, u2, blk_begin + ul + 2);
                if (!stage_changes_group(u2) || f0.bsel == f1.bsel) { stage_issue(ul + 2, u2); issued = true; }
            }
            const long long w0 = DBG ? clock64() : 0;
            mbar_wait_warp(bar_part + 8 * (ul & 1), (ul >> 1) & 1, s_abort);   // scanners parked unit ul; its MMAs are complete
            if (DBG) a60 += clock64() - w0;
            if (ht == 0) stamp(9 + ul * 6);
            // (A/B build PSD_TC_STAGE_FIRST) operands first: unit ul's MMAs are complete, so its A buffer is free, and (issued) the
            // staging touches nothing that resolve(ul) reads.  Staged behind the resolve, the operands of unit ul + 2 arrive ~0.8 k
            // cycles before the MMA thread needs them -- and ~3.9 k cycles too late whenever the unit starts a new cloud/direction
            // (B operand build, ~4.7 k cycles): all of the slowest CTAs of a launch are such CTAs (tools/tc_cta_balance.py).  With
            // the operands first those waits disappear, but the helpers' extra work still ends the CTA later: no gain.
            bool staged = false;
            Frame f2 = f1;
            if (PSD_TC_STAGE_FIRST && stage_next && issued) { stage_finish(ul + 2, u2); f2 = fr_st; staged = true; }
            resolve(ul, u0, f0);
            if (ht == 0) stamp(10 + ul * 6);
            help_bar();   // every helper is done with part/sq/sraw of unit ul before anything is restaged
            {   // deferred exact scans: flush when the next unit could overflow the list
                const int nfb = *s_nfb;
                if (nfb > kFbCap - kQB) {
                    run_fallbacks(p, blk_begin, fb_list, fb_q, nfb, hw, kHelpWarps, lane, sraw, s_rawgroup);
                    if (ht == 0) atomicAdd(&g_fallback_queries_tc, (unsigned long long)nfb);
                    help_bar();
                    if (ht == 0) *s_nfb = 0;
                    help_bar();
                }
            }
            f0 = f1;
            if (stage_next) {
                if (!staged) {
                    if (!issued) stage_issue(ul + 2, u2);
                    stage_finish(ul + 2, u2);
                    f2 = fr_st;
                }
                f1 = f2;
            }
            u0 = u1; u1 = u2;
            if (ht == 0) stamp(11 + ul * 6);
        }
        if (DBG && pf && ht == 0) pf[60] = a60;
        if (PSD_TC_SETMAXNREG) asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
    }

    // ---------------- the deferred exact scans of this CTA, by every warp: with few queries (the usual 0-3) each query is
    // split over up to four warps whose partial minima meet in a shared-memory atomicMin
    if (p.pdl_trigger) pdl_trigger();   // the next kernel on the stream may be launched; it waits (pdl_wait) until this grid has completed
    tc_fence_before();
    __syncthreads();
    if (tid == 0) stamp(3);
    {
        const int nfb = *s_nfb;
        constexpr int kW = kThreadsTC / 32;
        const int nsplit = nfb * 4 <= kW ? 4 : (nfb * 2 <= kW ? 2 : 1);
        unsigned long long *s_keys = reinterpret_cast<unsigned long long *>(part);   // partial results are dead by now
        if (PSD_TC_TAIL_FAST && nfb * nsplit <= kW) {
            // the usual case (at most one part of one query per warp): the warp keeps its query in registers across ONE barrier,
            // every part writes its own slot (no initialisation, no atomics), and part 0 of a query merges and stores -- one
            // decode + one round trip for the query's coordinates and one CTA barrier less than the general form below
            const bool mine = warp < nfb * nsplit;
            const int fi = warp / nsplit, pt = warp - fi * nsplit;
            FbQuery q;
            if (mine) {
                q = fallback_query(p, blk_begin, fb_list[fi], sraw, s_rawgroup, fb_q + fi);
                const unsigned long long key = fallback_scan(q, pt, nsplit, lane);
                if (lane == 0) s_keys[warp] = key;
            }
            __syncthreads();
            if (mine && pt == 0 && lane == 0) {
                unsigned long long key = s_keys[warp];
                for (int i = 1; i < nsplit; ++i) { const unsigned long long o = s_keys[warp + i]; key = o < key ? o : key; }
                fallback_write(p, q, key);
            }
        } else {
            for (int i = tid; i < nfb; i += kThreadsTC) s_keys[i] = ~0ull;
            __syncthreads();
            for (int item = warp; item < nfb * nsplit; item += kW) {
                const int fi = item / nsplit;
                const FbQuery q = fallback_query(p, blk_begin, fb_list[fi], sraw, s_rawgroup, fb_q + fi);
                const unsigned long long key = fallback_scan(q, item - fi * nsplit, nsplit, lane);
                if (lane == 0) atomicMin(s_keys + fi, key);
            }
            __syncthreads();
            for (int fi = tid; fi < nfb; fi += kThreadsTC) {
                const FbQuery q = fallback_query(p, blk_begin, fb_list[fi], sraw, s_rawgroup, fb_q + fi);
                fallback_write(p, q, s_keys[fi]);
            }
        }
        if (nfb > 0 && tid == 0) atomicAdd(&g_fallback_queries_tc, (unsigned long long)nfb);
    }
    if (tid == 0) stamp(4);
    if (warp == kMmaWarp)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
}

}  // namespace tc
}  // namespace psd

using namespace psd;

// Finalize kernel of the multi-tile mode: unpack the merged (distance, index) keys, apply the reference's tile-0 NaN rule
// (a NaN distance to target 0 poisons the result: chamfer3D.cu:36,126) and the fused loss-sum / F-score epilogue.
namespace psd {
namespace tc {
// RAGGED: rows past the pair's query length get dist 0, idx -1 and are not counted; every row of an invalid pair gets NaN, -1.
template <bool RAGGED>
__global__ void __launch_bounds__(256) chamfer_nn_tc_finalize_kernel(const std::conditional_t<RAGGED, NNRaggedParams, NNParams> p,
                                                                     int b) {
    const long long n0 = p.dir[0].ws ? (long long)b * p.dir[0].q_count : 0;
    const long long n1 = p.dir[1].ws ? (long long)b * p.dir[1].q_count : 0;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = gid < n0 + n1;
    const int d = (active && gid >= n0) ? 1 : 0;
    const NNDirection &D = p.dir[d];
    float dres = 0.f;
    int cloud = -1;
    bool counted = active;
    if (active) {
        const long long e = d ? gid - n0 : gid;
        cloud = (int)(e / D.q_count);
        const int j = D.q_begin + (int)(e - (long long)cloud * D.q_count);
        const unsigned long long key = D.ws[(long long)cloud * D.nq + j];
        D.ws[(long long)cloud * D.nq + j] = ~0ull;   // the library-owned workspace is always left clean for the next launch
        int qn = 0, tn = 0;
        bool ok = true;
        if constexpr (RAGGED) ok = ragged_lengths(p, d, cloud, qn, tn);
        int ires;
        if (RAGGED && j >= qn) {   // (the query row itself is never read)
            dres = ok ? 0.f : __int_as_float(0x7fc00000);
            ires = -1;
            counted = false;
        } else {
            const float *qp = D.q + (long long)cloud * D.q_bs + (long long)j * D.q_ps;
            const float d0 = exact_d(D.t + (long long)cloud * D.t_bs, D.t_ps, D.t_cs, 0, __ldg(qp), __ldg(qp + D.q_cs), __ldg(qp + 2 * D.q_cs));
            if (d0 != d0) { dres = d0; ires = 0; }
            else { dres = __uint_as_float((unsigned int)(key >> 32)); ires = (int)(key & 0xffffffffu); }
        }
        D.dist[(long long)cloud * D.nq + j] = dres;
        D.idx[(long long)cloud * D.nq + j] = ires;
    }
    if (p.sums != nullptr || p.fs_count != nullptr) {
        // warp-aggregated when the whole warp sits in one cloud/direction, else one atomic per thread
        const int key2 = active ? cloud * 2 + D.slot : -1;
        const int k0 = __shfl_sync(0xffffffffu, key2, 0);
        const bool uniform = __all_sync(0xffffffffu, key2 == k0);
        float ws = active ? dres : 0.f;
        int wc = (counted && dres < p.fs_thr) ? 1 : 0;
        if (uniform) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { ws += __shfl_xor_sync(0xffffffffu, ws, o); wc += __shfl_xor_sync(0xffffffffu, wc, o); }
            if ((threadIdx.x & 31) == 0 && k0 >= 0) {
                if (p.sums) atomicAdd(p.sums + k0, ws);
                if (p.fs_count && wc) atomicAdd(p.fs_count + k0, wc);
            }
        } else if (active) {
            if (p.sums) atomicAdd(p.sums + key2, ws);
            if (p.fs_count && wc) atomicAdd(p.fs_count + key2, wc);
        }
    }
}
}  // namespace tc
}  // namespace psd

// The tensor-core kernel takes every shape: target clouds of more than 2048 points are cut into tiles (multi-tile mode).
bool psd_nn_tc_supported(const NNParams &p) {
    const long long t0 = (p.dir[0].nt + tc::kMaxT - 1) / tc::kMaxT, t1 = (p.dir[1].nt + tc::kMaxT - 1) / tc::kMaxT;
    return (long long)p.blocks_dir0 * t0 + (long long)(p.total_blocks - p.blocks_dir0) * t1 < 0x3fffffffLL;
}

// Throughput-oriented callers that keep several launches in flight (a pipelined training loop) can give every launch a part
// of the GPU: a CTA then owns twice as many units and its serial prologue and tail amortise, while a launch on another stream
// fills the other SMs.  0 = one CTA per SM.
static std::atomic<int> g_tc_max_ctas{0};
int psd_set_tc_max_ctas(int n) { return n >= 0 ? g_tc_max_ctas.exchange(n) : g_tc_max_ctas.load(); }

// Merge workspace of the multi-tile mode: one grow-only buffer per (device, stream), owned by the library and ALWAYS left
// filled with all-ones keys (the finalize kernel resets what it reads), so a launch costs neither an allocation nor a
// memset.  Launches on one stream are ordered, launches on different streams get different buffers.  While `stream` is
// being captured into a CUDA graph the launch takes a graph-owned allocation instead (cudaMallocAsync + memset +
// cudaFreeAsync nodes, *temp = true): a graph must never hold a library pointer that a later launch may free.
static cudaError_t acquire_merge_ws(DeviceState *ds, cudaStream_t stream, size_t elems, unsigned long long **out, bool *temp,
                                    MergeWorkspace **slot_out) {
    *temp = false; *slot_out = nullptr;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaError_t e = cudaStreamIsCapturing(stream, &cap);
    if (e != cudaSuccess) return e;
    if (cap != cudaStreamCaptureStatusNone) {
        // a graph must not hold a pointer that a later, larger launch may free: graph-owned memory for this launch
        e = cudaMallocAsync(reinterpret_cast<void **>(out), elems * sizeof(unsigned long long), stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(*out, 0xff, elems * sizeof(unsigned long long), stream);
        *temp = true;
        return e;
    }
    std::lock_guard<std::mutex> lock(state_mutex());
    MergeWorkspace *hit = nullptr, *victim = &ds->merge[0];
    for (MergeWorkspace &w : ds->merge) {
        if (w.used && w.stream == stream) { hit = &w; break; }
        if (!w.used) { if (victim->used) victim = &w; }
        else if (victim->used && w.last_use < victim->last_use) victim = &w;
    }
    if (hit && hit->elems >= elems && !hit->dirty) {
        hit->last_use = ++ds->merge_clock;
        *out = hit->ptr; *slot_out = hit;
        return cudaSuccess;
    }
    MergeWorkspace *w = hit ? hit : victim;
    if (w->used && (w->elems < elems || w != hit)) {
        // growing, or evicting another stream's buffer: whatever still uses it must have finished
        e = (w == hit) ? cudaStreamSynchronize(stream) : cudaDeviceSynchronize();
        if (e != cudaSuccess) return e;
        cudaFree(w->ptr);
        *w = MergeWorkspace();
    }
    if (w->ptr == nullptr) {
        e = cudaMalloc(reinterpret_cast<void **>(&w->ptr), elems * sizeof(unsigned long long));
        if (e != cudaSuccess) { *w = MergeWorkspace(); return e; }
        w->elems = elems;
        w->dirty = true;
    }
    if (w->dirty) {
        e = cudaMemsetAsync(w->ptr, 0xff, w->elems * sizeof(unsigned long long), stream);
        if (e != cudaSuccess) return e;
        w->dirty = false;
    }
    w->used = true; w->stream = stream; w->last_use = ++ds->merge_clock;
    *out = w->ptr; *slot_out = w;
    return cudaSuccess;
}

// ragged: per-pair lengths len1 / len2 of xyz1 / xyz2 (device int [b], NULL = n / m), see NNRaggedParams
cudaError_t psd_launch_nn_tc(const NNParams &p_in, DeviceState *ds, cudaStream_t stream, float *dbg, int dbg_ld, long long *prof, int b,
                             bool ragged, const int *len1, const int *len2) {
    {
        std::lock_guard<std::mutex> lock(state_mutex());
        if (!ds->attr_tc) {
            cudaError_t e = cudaFuncSetAttribute(tc::chamfer_nn_tc_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::kSmemTC);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(tc::chamfer_nn_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::kSmemTC);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(tc::chamfer_nn_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::kSmemTC);
            if (e != cudaSuccess) return e;
            ds->attr_tc = true;
        }
    }
    NNParams p = p_in;
    // target tiles; directions with more than one tile (and at least one query) merge through the 64-bit workspace [B, nq]
    unsigned long long *ws = nullptr;
    size_t ws_elems = 0;
    bool need_ws[2];
    for (int d = 0; d < 2; ++d) {
        p.dir[d].ntt = (p.dir[d].nt + tc::kMaxT - 1) / tc::kMaxT;
        need_ws[d] = p.dir[d].ntt > 1 && p.dir[d].q_count > 0;
        if (need_ws[d]) ws_elems += (size_t)b * p.dir[d].nq;
    }
    bool ws_temp = false;
    MergeWorkspace *ws_slot = nullptr;
    if (ws_elems) {
        cudaError_t e = acquire_merge_ws(ds, stream, ws_elems, &ws, &ws_temp, &ws_slot);
        if (e != cudaSuccess) return e;
    }
    {
        unsigned long long *w = ws;
        for (int d = 0; d < 2; ++d) {
            p.dir[d].ws = need_ws[d] ? w : nullptr;
            if (need_ws[d]) w += (size_t)b * p.dir[d].nq;
        }
    }
    const int blocks0 = p.blocks_dir0 * p.dir[0].ntt;
    const int blocks1 = (p.total_blocks - p.blocks_dir0) * p.dir[1].ntt;
    p.blocks_dir0 = blocks0;
    p.total_blocks = blocks0 + blocks1;
    int grid = p.total_blocks < ds->num_sms ? p.total_blocks : ds->num_sms;
    const int cap = g_tc_max_ctas.load();
    if (cap > 0 && grid > cap) grid = cap;
    p.pdl_trigger = (cap > 0 && grid == cap) ? 0 : 1;
    NNRaggedParams pr;
    static_cast<NNParams &>(pr) = p;
    pr.qlen[0] = len1; pr.tlen[0] = len2;   // direction 0: xyz1 -> xyz2
    pr.qlen[1] = len2; pr.tlen[1] = len1;
    cudaError_t e;
    if (ragged) e = psd_launch_pdl(p.pdl_trigger != 0, tc::chamfer_nn_tc_kernel<false, true>, dim3(grid), dim3(tc::kThreadsTC), tc::kSmemTC, stream, pr, (float *)nullptr, 0, (long long *)nullptr);
    else if (dbg || prof) e = psd_launch_pdl(p.pdl_trigger != 0, tc::chamfer_nn_tc_kernel<true, false>, dim3(grid), dim3(tc::kThreadsTC), tc::kSmemTC, stream, p, dbg, dbg_ld, prof);
    else e = psd_launch_pdl(p.pdl_trigger != 0, tc::chamfer_nn_tc_kernel<false, false>, dim3(grid), dim3(tc::kThreadsTC), tc::kSmemTC, stream, p, (float *)nullptr, 0, (long long *)nullptr);
    if (ws_elems) {
        if (e == cudaSuccess) {
            const long long total = (p.dir[0].ws ? (long long)b * p.dir[0].q_count : 0) + (p.dir[1].ws ? (long long)b * p.dir[1].q_count : 0);
            if (total > 0) {
                if (ragged) tc::chamfer_nn_tc_finalize_kernel<true><<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(pr, b);
                else tc::chamfer_nn_tc_finalize_kernel<false><<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(p, b);
                e = cudaGetLastError();
            }
        }
        if (ws_temp) {
            const cudaError_t e2 = cudaFreeAsync(ws, stream);
            if (e == cudaSuccess) e = e2;
        } else if (e != cudaSuccess && ws_slot) {
            std::lock_guard<std::mutex> lock(state_mutex());
            ws_slot->dirty = true;   // a failed launch may have left keys behind: refill before the next use
        }
    }
    return e;
}

cudaError_t psd_read_chamfer_stats_tc(unsigned long long *fallback, int reset) {
    cudaError_t e = cudaMemcpyFromSymbol(fallback, tc::g_fallback_queries_tc, sizeof(unsigned long long));
    if (e != cudaSuccess) return e;
    if (reset) {
        const unsigned long long z = 0;
        e = cudaMemcpyToSymbol(tc::g_fallback_queries_tc, &z, sizeof(z));
    }
    return e;
}
