// Kernel 2 (tensor-core contraction path, sm_100a): the bilinear contractions of the decoder on tcgen05 with TMEM
// accumulators, fp32-accurate through an error-compensated 3xTF32 split.
//
//   reference: weighted_R = T.tensordot(relation_probs, R, axes=[[1],[2]])   learning/models/decoders/Bilinear.py:33
//              weightedC  (same)                                             learning/models/decoders/BilinearPlusSP.py:37
//              weightedC1/C2 = T.dot(relation_probs, C1.T / C2.T)            BilinearPlusSP.py:35-36, SelectionalPreferences.py:31-32
//              batched_tensordot / batched_dot consumers                     Bilinear.py:58-59,68-69,78-79
//              and T.grad through them                                       learning/Optimizers.py:27
//
// Three GEMM-shaped contractions per step, none of which may materialise [B, d*d] in HBM (64 KiB per example at d=128):
//   forward / backward-recompute  M_b = sum_k q_bk C[:,:,k]      D[b, n]  = sum_k P[b,k]  Cf[n,k]     -> v = M R, w = M^T L
//   backward dq                   dq_bk = <dM_b, C[:,:,k]>        D[b, k]  = sum_n G[b,n]  Cf[n,k]     (G = a R^T + L Y2^T, rank 2)
//   backward dC                   dC[n,k] = sum_b dM_b[n] q_bk    D[n, k]  = sum_b G[b,n]  q[b,k]
// fp32 parity: every operand x is split x = hi + lo and each k-step issues hi.hi + hi.lo + lo.hi with fp32 accumulation in
// TMEM (dropped lo.lo ~ 2^-22 relative).  The forward / recompute and dq contractions split into FP16 pairs (kind::f16,
// K = 16 per MMA: the same 64 cycles per instruction as a K = 8 kind::tf32 MMA, profiles/microbench/mma_power.cu, so half
// the MMAs): an fp16 has the 11-bit significand of a TF32, and its narrow exponent is handled by scaling every operand
// tensor by an exact power of two chosen from its measured |max| (so that |x| s < 2^12: no overflow; a value whose lo part
// falls into the fp16 subnormals is still exact to 2^-37 of the tensor's maximum), undone in the epilogue.  So does the dC
// contraction (k_tc_dc2), except its fallback for B % 4 != 0 (k_tc_dc), which splits into TF32 pairs (kind::tf32).
//
// The M-side (A) operand lives in TMEM (TS mode): the threads that own a TMEM lane (= an example row b, or an output row
// n) write their row with tcgen05.st - q rows once per segment for the forward, the generated operand G stage by stage for
// the backward - and only the small N-side (B) operand streams through shared memory.  B operands are pre-split and
// pre-arranged in HBM as the exact shared-memory image of the no-swizzle K-major canonical layout (float4 planes
// T[kq][row]; LBO = rows*16 B, SBO = 128 B), so a stage is filled by ONE 1-D bulk copy (cp.async.bulk -> UBLKCP)
// completing on an mbarrier.
//
// Sizes follow the measured MMA cadence (profiles/microbench/RESULTS.md): one tcgen05.mma cannot issue faster than every
// ~45 cycles, so every MMA here has N >= 112 accumulator columns (56 / 64 cycles, at the floor 128*N/256): the forward
// streams 128-row chunks (one N = 128 MMA per k-step and split term), the backward reduces over 64-row stages against the
// NK = K rounded up to 16 relation columns.  Work is dealt over the SMs by the balanced schedule of rae_internal.h
// (TcSched): every CTA gets the same number of MMAs; its range is cut into per-tile segments.
//
// Warp roles (all kernels): the row-owning workers (epilogue / operand generators) are warps 0 .. NW-1 (worker warp w
// touches TMEM lanes 32*(w%4)..+31 as the hardware requires); then NW = MMA issuer (one elected thread), NW+1 = bulk-copy
// producer, NW+2 = TMEM allocator, NW+3 = idle.  The order matters: a scheduler partition issues from its HIGHEST warp id
// first (B300_MICROARCH.md), and the MMA issuer must never wait behind the instruction-heavy workers it shares a partition
// with - as warp 1 it did, and the MMAs and the epilogue arithmetic ran one after the other instead of side by side.
#include <cuda_fp16.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "rae_common.cuh"
#include "rae_internal.h"

namespace rae {

namespace {

// optional in-kernel timeline (build with -DRAE_TRACE, never part of the shipped library): SM cycle counter of CTA-local
// milestones, [CTA][TC_TRACE_STRIDE] slots; forward kernel slots 0.., dq 16.., dC 32.., recompute pass 64.. (the forward
// kernel's slots + 64), dq segment / selectional-preference stamps 96.., dC segment values 80.. (see profiles/trace_tc.py)
#ifdef RAE_TRACE
constexpr int TC_TRACE_STRIDE = 128;
__device__ unsigned long long* g_tc_trace = nullptr;
// knock-out switches of the MEASUREMENT build only (profiles/trace_tc.py): 1 = the producer arrives without copying after
// the first fills, 2 = the MMA thread commits without issuing MMAs, 4 = the row-owning warps skip their arithmetic
__device__ int g_tc_knock = 0;
#define TC_KNOCK(bit) ((g_tc_knock & (bit)) != 0)
#define TC_TRACE_INIT() unsigned long long* const tc_trace_ptr_ = g_tc_trace
#define TC_TRACE(slot)                                                                                         \
    do {                                                                                                       \
        if (tc_trace_ptr_ != nullptr && (slot) < TC_TRACE_STRIDE) tc_trace_ptr_[(size_t)blockIdx.x * TC_TRACE_STRIDE + (slot)] = clock64(); \
    } while (0)
// a value instead of a clock (segment count, tile-end flag)
#define TC_TRACE_VAL(slot, v)                                                                                  \
    do {                                                                                                       \
        if (tc_trace_ptr_ != nullptr) tc_trace_ptr_[(size_t)blockIdx.x * TC_TRACE_STRIDE + (slot)] = (unsigned long long)(v); \
    } while (0)
// the forward kernel's slot base: 0 for the forward pass, 64 for the recompute pass (the one without C1 / C2 rows)
#define TC_TRACE_BASE(with_sp) const int tc_tb_ = (with_sp) ? 0 : 64
// this CTA's segment count and whether one of its segments ends a tile (its range holds the tile's last unit)
#define TC_TRACE_SEGS(sch, slot_n, slot_end)                                                                   \
    do {                                                                                                       \
        TcSegIter si_(p.segs, (sch).upt, blockIdx.x);                                                          \
        TcSeg sg_;                                                                                             \
        int n_ = 0, e_ = 0;                                                                                    \
        while (si_.next(sg_)) { ++n_; e_ |= sg_.u1 == (sch).upt; }                                             \
        TC_TRACE_VAL(slot_n, n_);                                                                              \
        TC_TRACE_VAL(slot_end, e_);                                                                            \
    } while (0)
// wall-clock stamp (ns, synchronised across SMs): kernel duration and the SM clock actually held under tensor load
#define TC_TRACE_NS(slot)                                                                                      \
    do {                                                                                                       \
        if (tc_trace_ptr_ != nullptr) {                                                                        \
            unsigned long long ns_;                                                                            \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns_));                                            \
            tc_trace_ptr_[(size_t)blockIdx.x * TC_TRACE_STRIDE + (slot)] = ns_;                                \
        }                                                                                                      \
    } while (0)
#else
#define TC_KNOCK(bit) false
#define TC_TRACE_VAL(slot, v) do { } while (0)
#define TC_TRACE_BASE(with_sp) do { } while (0)
#define TC_TRACE_SEGS(sch, slot_n, slot_end) do { } while (0)
#define TC_TRACE_NS(slot) do { } while (0)
#define TC_TRACE_INIT() do { } while (0)
#define TC_TRACE(slot) do { } while (0)
#endif

constexpr int TC_M = 128;          // rows per CTA tile (TMEM lanes)
constexpr int TC_N = 128;          // forward: B-operand rows per chunk = accumulator columns per MMA
constexpr int TC_H = 64;           // forward: half chunk, the unit one epilogue group consumes
constexpr int TC_TSTAGES = 3;      // forward: accumulator stages in TMEM (3 x 128 columns; the packed FP16 P operand needs <= 112)
constexpr int TC_NC = 32;          // backward: reduction rows per operand chunk in HBM ([c32][hi/lo][8][NK])
constexpr int TC_SR = 64;          // backward: reduction rows per pipeline stage (two chunks)
constexpr int TC_BSTAGES = 3;      // backward: B-operand shared-memory stages
constexpr int TC_FWD_WORKERS = 8;      // forward: epilogue warps (0..7)
constexpr int TC_BWD_WORKERS = 16;     // backward: generator warps (0..15)
constexpr int TC_FWD_THREADS = 384;    // 8 epilogue + 4 control warps
constexpr int TC_BWD_THREADS = 640;    // 16 generator + 4 control warps
constexpr uint32_t TC_FWD_ACOL = 384;  // forward: first TMEM column of the resident P operand (hi, then lo)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_g2s_pieces(uint8_t* dst_smem, const uint8_t* src_gmem, uint32_t bytes, uint64_t* bar) {
    constexpr uint32_t PIECE = 1u << 16;    // one instruction per stage: each bulk copy costs ~85 cycles + bytes / 130 B per cycle (profiles/microbench)
    for (uint32_t off = 0; off < bytes; off += PIECE) bulk_g2s(dst_smem + off, src_gmem + off, min(PIECE, bytes - off), bar);
}
// one lane of a converged warp (the loops around it stay warp-uniform, so descriptor math lives in uniform registers)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T, kind::tf32 (TS mode: A rows = TMEM lanes, one 32-bit element per column)
__device__ __forceinline__ void tc_mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// 32 lanes x 32 columns of fp32 accumulators -> 32 registers per thread (thread t = lane base + t)
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
// 8 registers per thread -> 32 lanes x 8 columns of TMEM (thread t writes lane base + t)
__device__ __forceinline__ void tc_st8(uint32_t taddr, const float (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
                 "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
                 "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
                 : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 consecutive floats of one accumulator row -> global memory; 16-byte stores when the row is 16-byte aligned
__device__ __forceinline__ void store_row32(float* o, const float (&t)[32], int nvalid, bool vec) {
    if (vec) {
#pragma unroll
        for (int x = 0; x < 32; x += 4)
            if (x < nvalid) *reinterpret_cast<float4*>(o + x) = make_float4(t[x], t[x + 1], t[x + 2], t[x + 3]);
    } else {
#pragma unroll
        for (int x = 0; x < 32; ++x)
            if (x < nvalid) o[x] = t[x];
    }
}

// shared-memory matrix descriptor, K-major, no swizzle: core matrix = 8 rows x 16 B (128 B contiguous);
// LBO = byte distance between the two 16-byte K-halves of one MMA k-step, SBO = byte distance between 8-row groups
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
    d |= (uint64_t)1 << 46;     // descriptor version (Blackwell)
    return d;                   // layout_type = 0 (SWIZZLE_NONE), base_offset = 0
}
// descriptor with the start address advanced by `bytes` (the address field is the low 14 bits, in 16-byte units)
__device__ __forceinline__ uint64_t desc_advance(uint64_t desc, uint32_t bytes) { return desc + (uint64_t)(bytes >> 4); }
// instruction descriptor: D = F32, A = B = TF32, both K-major, dense, no negate
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ float tf32_hi(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
// hot-loop split (operand generators, 16 warps per SM, instruction-bound): hi = round-to-nearest-away TF32 of a FINITE x as
// two integer ops (cvt.rna.tf32 compiles to three: it also guards inf / nan), lo = x - hi (exact) with its low 13 bits
// cleared (truncation: |error| < 2^-23 |x|, below the dropped lo*lo term)
__device__ __forceinline__ void split8(const float (&x)[8], float (&hi)[8], float (&lo)[8]) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        hi[u] = __uint_as_float((__float_as_uint(x[u]) + 0x1000u) & 0xffffe000u);
        lo[u] = __uint_as_float(__float_as_uint(x[u] - hi[u]) & 0xffffe000u);
    }
}
__device__ __forceinline__ void split4(const float (&x)[4], float4& hi, float4& lo) {
    hi.x = tf32_hi(x[0]); hi.y = tf32_hi(x[1]); hi.z = tf32_hi(x[2]); hi.w = tf32_hi(x[3]);
    lo.x = tf32_hi(x[0] - hi.x); lo.y = tf32_hi(x[1] - hi.y); lo.z = tf32_hi(x[2] - hi.z); lo.w = tf32_hi(x[3] - hi.w);
}

// instruction descriptor: D = F32, A = B = F16, both K-major, dense, no negate (kind::f16)
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void tc_mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// FP16 pair split of two (already scaled) values: hi = rn_f16(x), lo = rn_f16(x - hi); element 0 in the low half-word
__device__ __forceinline__ void split_h2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn(x0, x1);
    const __half2 l = __floats2half2_rn(x0 - __low2float(h), x1 - __high2float(h));
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}
__device__ __forceinline__ void tc_st8u(uint32_t taddr, const uint32_t (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
                 "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
__device__ __forceinline__ void tc_st4u(uint32_t taddr, const uint32_t (&v)[4]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3])
                 : "memory");
}
// power-of-two scale s with amax * s < 2^12 (amax given as the bits of a non-negative float; 1 for zero / denormal)
__host__ __device__ __forceinline__ float pow2_scale(uint32_t amax_bits) {
    const int e = (int)((amax_bits >> 23) & 255u) - 127;      // amax < 2^(e+1)
    if (((amax_bits >> 23) & 255u) == 0u) return 1.f;
    int se = 11 - e;
    se = se < -100 ? -100 : (se > 100 ? 100 : se);
    union { uint32_t u; float f; } cv;
    cv.u = (uint32_t)(se + 127) << 23;
    return cv.f;
}
constexpr float TC_QSCALE = 4096.f;        // q in [0, 1] -> [0, 2^12]
// device scalars of the tensor path (TcState::scal, uint32 words)
// (TS_AMAX_SP: the selectional-preference stage images of the dC kernel, a + G2 L | c + G1 R)
enum TcScal { TS_AMAX_C = 0, TS_AMAX_L = 1, TS_AMAX_R = 2, TS_AMAX_A = 3, TS_AMAX_CV = 4, TS_AMAX_Y2 = 5, TS_AMAX_SP = 6, TS_N = 8 };

// Global load that stays where it is written: a run of these is issued back to back (ptxas keeps volatile asm in program
// order and cannot fold the consumers in between), so a thread's 32-64 row loads cost ONE memory latency.  Plain loads were
// scheduled in batches of 7 with the conversions in between (register reuse): 8 serialised L2 latencies per prologue.
__device__ __forceinline__ float ldg_stream(const float* p) {
    float v;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}

// the same for data this kernel also writes (no read-only path)
__device__ __forceinline__ float ldg_ordered(const float* p) {
    float v;
    asm volatile("ld.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
    return v;
}

// segments of a CTA's range under the balanced schedule (rae_internal.h)
struct TcSeg { int tile, u0, u1, slot; };
// A CTA's range comes from the schedule's table (tc_init: tc_seg_table), one int4 per CTA: first unit, end unit, slot of
// the first segment.  Every role of every CTA reads its entry instead of evaluating the closed form: the divisions of
// tcs_start / tcs_first, run by all 12-20 warps of a CTA at its start, cost thousands of cycles per CTA.  Only the first
// segment can start inside a tile; every later one starts its tile, so this CTA is the tile's first and writes slot 0.
struct TcSegIter {
    int upt, cur, end, slot;
    __device__ __forceinline__ TcSegIter(const int4* segs, int upt_, int x) : upt(upt_) {
        const int4 e = __ldg(segs + x);
        cur = e.x; end = e.y; slot = e.z;
    }
    __device__ __forceinline__ bool next(TcSeg& g) {
        if (cur >= end) return false;
        g.tile = cur / upt;
        g.u0 = cur - g.tile * upt;
        const int len = min(upt - g.u0, end - cur);
        g.u1 = g.u0 + len;
        g.slot = slot;
        slot = 0;
        cur += len;
        return true;
    }
};

// row n of the dense operand Cf -> source [K]-vector (nullptr = zero padding row)
//   n <  n_bil_rows : C[i, j, :] with i = n / DP, j = n % DP
//   then DP rows of C1[j,:] and DP rows of C2[j,:]; anything beyond is padding
__device__ __forceinline__ const float* cf_row(const float* C, const float* C1, const float* C2, int d, int K, int DP,
                                               int n_bil_rows, int n) {
    if (n < n_bil_rows) {
        const int i = n / DP, j = n - i * DP;
        return (i < d && j < d && C != nullptr) ? C + ((size_t)i * d + j) * K : nullptr;
    }
    const int m = n - n_bil_rows;
    const int which = m / DP, j = m - which * DP;
    if (j >= d || which > 1) return nullptr;
    const float* src = which == 0 ? C1 : C2;
    return src != nullptr ? src + (size_t)j * K : nullptr;
}

// ------------------------------------------------------------------------------------------------------------
// operand preparation (per step; the dense parameters change every step)
// ------------------------------------------------------------------------------------------------------------
// |max| over the dense decoder tensors -> scal[TS_AMAX_C] (bits of a non-negative float: integer max is order-free, so the
// atomic is deterministic)
__global__ void __launch_bounds__(256) k_tc_absmax(const float* __restrict__ C, size_t nC, const float* __restrict__ C1, size_t n1,
                                                   const float* __restrict__ C2, size_t n2, uint32_t* __restrict__ out) {
    pdl_enter();
    __shared__ uint32_t red[8];
    uint32_t m = 0;
    const size_t stride = (size_t)gridDim.x * blockDim.x, t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    auto scan = [&](const float* p, size_t n) {
        if (p == nullptr || n == 0) return;
        if ((n & 3) == 0 && (reinterpret_cast<uintptr_t>(p) & 15) == 0) {
            const float4* p4 = reinterpret_cast<const float4*>(p);
            for (size_t i = t0; i < n / 4; i += stride) {
                const float4 v = p4[i];
                m = max(max(m, __float_as_uint(fabsf(v.x))), max(__float_as_uint(fabsf(v.y)), max(__float_as_uint(fabsf(v.z)), __float_as_uint(fabsf(v.w)))));
            }
        } else {
            for (size_t i = t0; i < n; i += stride) m = max(m, __float_as_uint(fabsf(p[i])));
        }
    };
    scan(C, nC);
    scan(C1, n1);
    scan(C2, n2);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(kFull, m, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) m = max(m, red[w]);
        atomicMax(out, m);
    }
}

// FP16 pair operands of the dense tensors, scaled by s_C = pow2_scale(|max|):
// blockIdx.y == 0: forward B operand [chunk of 128 rows n][hi/lo][kq 0..KQ8-1][row] x 16 B = relations 8 kq .. 8 kq + 7 of row n
// blockIdx.y == 1: dq B operand, Cf transposed: [stage of 128 rows n][hi/lo][oct 0..15][krow 0..NK-1] x 16 B = rows
//                  128 st + 8 oct + 0..7 at relation krow
__global__ void __launch_bounds__(256) k_tc_prep_c(const float* __restrict__ C, const float* __restrict__ C1,
                                                   const float* __restrict__ C2, int d, int K, int KQ8, int DP, int n_bil_rows,
                                                   int n_rows_fwd, uint4* __restrict__ out, int NK, int n_rows_bwd,
                                                   uint4* __restrict__ out2, const uint32_t* __restrict__ scal) {
    pdl_enter();
    const float sC = pow2_scale(scal[TS_AMAX_C]);
    if (blockIdx.y == 1) {
        const size_t total2 = (size_t)(n_rows_bwd / 8) * NK;
        for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total2; idx += (size_t)gridDim.x * blockDim.x) {
            const int krow = (int)(idx % NK);
            const int oct_g = (int)(idx / NK);
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float* s0 = cf_row(C, C1, C2, d, K, DP, n_bil_rows, 8 * oct_g + 2 * u);
                const float* s1 = cf_row(C, C1, C2, d, K, DP, n_bil_rows, 8 * oct_g + 2 * u + 1);
                const float x0 = (s0 != nullptr && krow < K) ? s0[krow] * sC : 0.f;
                const float x1 = (s1 != nullptr && krow < K) ? s1[krow] * sC : 0.f;
                split_h2(x0, x1, hi[u], lo[u]);
            }
            const int st = oct_g / 16, oct = oct_g - st * 16;
            uint4* base = out2 + (size_t)st * 2 * 16 * NK;
            base[(size_t)oct * NK + krow] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            base[(size_t)(16 + oct) * NK + krow] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
        return;
    }
    const size_t total = (size_t)n_rows_fwd * KQ8;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int kq = (int)(idx % KQ8);
        const int n = (int)(idx / KQ8);
        const float* src = cf_row(C, C1, C2, d, K, DP, n_bil_rows, n);
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int k = 8 * kq + 2 * u;
            const float x0 = (src != nullptr && k < K) ? src[k] * sC : 0.f;
            const float x1 = (src != nullptr && k + 1 < K) ? src[k + 1] * sC : 0.f;
            split_h2(x0, x1, hi[u], lo[u]);
        }
        const int chunk = n / TC_N, r = n - chunk * TC_N;
        uint4* base = out + (size_t)chunk * 2 * KQ8 * TC_N;
        base[(size_t)kq * TC_N + r] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        base[(size_t)(KQ8 + kq) * TC_N + r] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
}

// blockIdx.y == 0: dC B operand, q transposed: [chunk of 32 examples][hi/lo][bq 0..7][krow 0..NK-1] = (q[32c+4bq+0..3][krow]),
//                  nbc chunks (an even number: the kernels consume two per stage; examples >= B are zero)
// blockIdx.y == 1: L = A[a1], R = A[a2] (A[a1] with the model-C quirk) -> ev, one warp per example
// blockIdx.y == 2: P operand of the forward / recompute contraction (k_tc_bilinear): per 128-example tile
//                  [hi/lo][kq 0..NK/8-1][row 0..127] x 16 B = the FP16 pairs of q[b][8 kq .. 8 kq + 7] scaled by 2^12, i.e. TMEM
//                  columns 4 kq .. 4 kq + 3 of the row's P planes (one B-operand stage per tile, bulk-copied per segment)
// blockIdx.y == 3: the two-tile dC kernel's operand (below)
__global__ void __launch_bounds__(256) k_tc_prep_qt(const float* __restrict__ q, int B, int K, int NK, int nbc, float4* __restrict__ out,
                                                    const float* __restrict__ A, const int32_t* __restrict__ a1,
                                                    const int32_t* __restrict__ a2, int d, int dp, int quirk, float* __restrict__ ev,
                                                    uint32_t* __restrict__ scal, uint4* __restrict__ out4, uint4* __restrict__ pimg) {
    pdl_enter();
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < 2) scal[TS_AMAX_L + threadIdx.x] = 0u;   // the transposes that follow accumulate
    if (blockIdx.y == 2) {
        const int KQ8 = NK / 8;
        const size_t totalp = (size_t)((B + TC_M - 1) / TC_M) * KQ8 * TC_M;
        for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < totalp; idx += (size_t)gridDim.x * blockDim.x) {
            const int r = (int)(idx % TC_M);
            const int kq = (int)((idx / TC_M) % KQ8);
            const size_t tile = idx / ((size_t)TC_M * KQ8);
            const int b = (int)tile * TC_M + r;
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int k = 8 * kq + 2 * u;
                const float x0 = (b < B && k < K) ? q[(size_t)b * K + k] * TC_QSCALE : 0.f;
                const float x1 = (b < B && k + 1 < K) ? q[(size_t)b * K + k + 1] * TC_QSCALE : 0.f;
                split_h2(x0, x1, hi[u], lo[u]);
            }
            uint4* base = pimg + tile * 2 * KQ8 * TC_M;
            base[(size_t)kq * TC_M + r] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            base[(size_t)(KQ8 + kq) * TC_M + r] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
        return;
    }
    if (blockIdx.y == 3) {
        // FP16 pair operand of the two-tile dC kernel: [stage of 64 examples][hi/lo][oct 0..7][krow 0..NK-1] x 16 B = examples
        // 64 st + 8 oct + 0..7 at relation krow, q scaled by 2^12
        const size_t total4 = (size_t)(nbc / 2) * 8 * NK;
        for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total4; idx += (size_t)gridDim.x * blockDim.x) {
            const int krow = (int)(idx % NK);
            const int oct = (int)((idx / NK) % 8);
            const int st = (int)(idx / ((size_t)8 * NK));
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int b = st * 64 + 8 * oct + 2 * u;
                const float x0 = (b < B && krow < K) ? q[(size_t)b * K + krow] * TC_QSCALE : 0.f;
                const float x1 = (b + 1 < B && krow < K) ? q[(size_t)(b + 1) * K + krow] * TC_QSCALE : 0.f;
                split_h2(x0, x1, hi[u], lo[u]);
            }
            uint4* base = out4 + (size_t)st * 2 * 8 * NK;
            base[(size_t)oct * NK + krow] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            base[(size_t)(8 + oct) * NK + krow] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
        return;
    }
    if (blockIdx.y == 1) {
        const int lane = threadIdx.x & 31;
        for (int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < B; b += (gridDim.x * blockDim.x) >> 5) {
            const int r1 = a1[b], r2 = quirk ? r1 : a2[b];
            float* o = ev + (size_t)b * E_NV * dp;
            for (int j = lane; j < d; j += 32) {
                o[E_L * dp + j] = ld_nc(A + (size_t)r1 * d + j);
                o[E_R * dp + j] = ld_nc(A + (size_t)r2 * d + j);
            }
        }
        return;
    }
    const size_t total = (size_t)nbc * 8 * NK;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int krow = (int)(idx % NK);
        const int bq = (int)((idx / NK) % 8);
        const int bc = (int)(idx / ((size_t)8 * NK));
        float x[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int b = bc * TC_NC + 4 * bq + u;
            x[u] = (b < B && krow < K) ? q[(size_t)b * K + krow] : 0.f;
        }
        float4 hi, lo;
        split4(x, hi, lo);
        float4* base = out + (size_t)bc * 2 * 8 * NK;
        base[(size_t)bq * NK + krow] = hi;
        base[(size_t)(8 + bq) * NK + krow] = lo;
    }
}

// ------------------------------------------------------------------------------------------------------------
// forward contraction (also used for the backward recompute with L := a, R := c)
// TMEM map: accumulator stages [0,384) (3 x 128 columns), P operand (FP16 pairs, two relations per column) hi at
//           [384, 384 + KH/2), lo at [384 + KH/2, 384 + KH)
// Work unit = one 128-row chunk of Cf = two 64-row half chunks; epilogue group g (4 warps) consumes half g of EVERY chunk
// (accumulator columns [64 g, 64 g + 64)), so for DP = 128 group g always holds the column half j in [64 g, 64 g + 64).
// ------------------------------------------------------------------------------------------------------------
// Every per-thread global access of the row-owning warps is COALESCED: a thread owns example row b, so the inputs come
// from transposed copies [column][example] (lane = example -> consecutive addresses) and the outputs are written the same
// way; k_tc_combine transposes / sums them back into the row-major per-example vectors.  (Reading ev[b][...] directly
// costs one L1 wavefront per lane, ~66 cycles per warp instruction: measured as 2/3 of the kernel's time.)
struct TcArgs {
    const float4* bop;      // B operand chunks
    const uint8_t* pimg;    // P operand images, one B-operand stage per example tile (k_tc_prep_qt)
    const float* LT;        // [dp][B]  left vectors transposed  (L forward, a for the recompute pass)
    const float* RT;        // [dp][B]  right vectors transposed (R forward, c for the recompute pass)
    float* spT;             // [2][dp][B]        c1, c2 (the accumulator rows of the C1 / C2 half chunks), transposed
    float* vT;              // [2][dp][B]        v partial per epilogue group
    float* wT;              // [slot][2][dp][B]  w partial per (segment slot, group)
    const uint32_t* scal;   // device scalars (TcScal): |max| of the dense tensors -> operand scale
    int B, K, d, dp;
    int KH;                 // relations padded to a multiple of 16 (one kind::f16 MMA reduces over 16)
    int n_bil_half;         // half chunks holding bilinear rows
    int n_sp_half;          // half chunks holding C1/C2 rows (forward only; 0 for the recompute pass)
    int nbs;                // B-operand shared-memory stages
    TcSched sch;            // units = 128-row chunks, tiles = example tiles
    const int4* segs;       // sch's per-CTA table (TcSegIter)
};

template <int DP>
__global__ void __launch_bounds__(TC_FWD_THREADS, 1) k_tc_bilinear(TcArgs p) {
    pdl_enter();
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    TC_TRACE_INIT();
    TC_TRACE_BASE(p.n_sp_half > 0);
    const uint32_t KQ8 = (uint32_t)p.KH / 8u;               // 16-byte planes (8 relations each) per hi / lo half of a chunk
    const uint32_t B_BYTES = 2u * KQ8 * TC_N * 16u;
    const uint32_t KC = (uint32_t)p.KH / 2u;                // TMEM columns of one P plane (two fp16 per column)
    const int nbs = p.nbs;
    uint8_t* smB = smem_raw;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + (size_t)nbs * B_BYTES);
    uint64_t* a_full = bars;                                // 8 epilogue-warp arrivals per segment: P operand is in TMEM
    uint64_t* b_full = bars + 1;                            // [4]
    uint64_t* b_empty = b_full + 4;                         // [4]
    uint64_t* t_full = b_empty + 4;                         // [TC_TSTAGES]
    uint64_t* t_empty = t_full + TC_TSTAGES;                // [TC_TSTAGES] 8 epilogue-warp arrivals
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + TC_TSTAGES);
    if (threadIdx.x == 0) { TC_TRACE(tc_tb_ + 0); TC_TRACE_NS(tc_tb_ + 14); TC_TRACE_SEGS(p.sch, tc_tb_ + 57, tc_tb_ + 62); }

    if (threadIdx.x == 0) {
        mbar_init(a_full, 8);
        for (int s = 0; s < nbs; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
        for (int s = 0; s < TC_TSTAGES; ++s) { mbar_init(&t_full[s], 1); mbar_init(&t_empty[s], 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == TC_FWD_WORKERS + 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) TC_TRACE(tc_tb_ + 1);

    if (warp >= TC_FWD_WORKERS) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;" ::: "memory");
    }
    if (warp == TC_FWD_WORKERS + 1) {
        // ===== producer: per segment the P image of its tile, then its chunks; one bulk copy per ring stage =====
        if (lane == 0) {
            TcSegIter si(p.segs, p.sch.upt, blockIdx.x);
            TcSeg sg;
            int it = 0;
            auto fill = [&](const uint8_t* src) {
                const int s = it % nbs;
                const uint32_t ph = (it / nbs) & 1;
                mbar_wait(&b_empty[s], ph ^ 1);
                if (TC_KNOCK(1) && it >= nbs) { mbar_arrive(&b_full[s]); ++it; return; }
                mbar_expect_tx(&b_full[s], B_BYTES);
                bulk_g2s_pieces(smB + (size_t)s * B_BYTES, src, B_BYTES, &b_full[s]);
                ++it;
            };
            while (si.next(sg)) {
                fill(p.pimg + (size_t)sg.tile * B_BYTES);
                for (int c = sg.u0; c < sg.u1; ++c) fill(reinterpret_cast<const uint8_t*>(p.bop) + (size_t)c * B_BYTES);
            }
        }
    } else if (warp == TC_FWD_WORKERS) {
        // ===== MMA issuer: ONE elected thread runs the whole loop; the k-loop is fully unrolled so that every descriptor is
        // the chunk's base plus a compile-time offset (a rolled loop carried the descriptors through vector registers: a
        // register <-> uniform-register round trip per MMA, 129 issue cycles per MMA instead of 64 - measured).  The barrier
        // waits of chunk c+1 are taken in the middle of chunk c's MMA sequence, while the tensor pipe has queued work. =====
        if (elect_one()) {
            const uint32_t idesc = make_idesc_f16(TC_M, TC_N);
            const uint32_t a_hi = tmem_base + TC_FWD_ACOL, a_lo = a_hi + KC;
            const int ksteps = p.KH / 16;                   // 1 .. 7
            const int kmid = ksteps / 2;
            TcSegIter si(p.segs, p.sch.upt, blockIdx.x);
            TcSeg sg;
            int it = 0, seg = 0;
            // ring positions kept incrementally (no division by the runtime stage count in the loop): operand stage s with
            // phase bit sp, accumulator stage ts with phase bit tp
            int s = 0, ts = 0;
            uint32_t sp = 0, tp = 0;
            bool ready = false;                             // the barriers of chunk `it` have been acquired already
            while (si.next(sg)) {
                mbar_wait(a_full, seg & 1);                 // this segment's P rows are in TMEM
                tc_fence_after();
                if (seg == 1) TC_TRACE(tc_tb_ + 59);
                mbar_arrive(&b_empty[s]);                   // ... so the epilogue warps are done with its P image's stage
                if (++s == nbs) { s = 0; sp ^= 1; }
                for (int c = sg.u0; c < sg.u1; ++c, ++it) {
                    if (!ready) {
                        mbar_wait(&t_empty[ts], tp ^ 1);
                        mbar_wait(&b_full[s], sp);
                        tc_fence_after();
                    }
                    ready = false;
                    if (it == 4) TC_TRACE(tc_tb_ + 6);
                    if (it == 12) TC_TRACE(tc_tb_ + 10);
                    const uint32_t b_hi = smem_u32(smB + (size_t)s * B_BYTES);
                    const uint64_t h0 = make_desc(b_hi, TC_N * 16u, 128u);
                    const uint64_t l0 = make_desc(b_hi + KQ8 * TC_N * 16u, TC_N * 16u, 128u);
                    const uint32_t d0 = tmem_base + (uint32_t)(ts * TC_N);
                    const bool has_next = c + 1 < sg.u1;
                    int s1 = s + 1, ts1 = ts + 1;               // position of the next chunk
                    uint32_t sp1 = sp, tp1 = tp;
                    if (s1 == nbs) { s1 = 0; sp1 ^= 1; }
                    if (ts1 == TC_TSTAGES) { ts1 = 0; tp1 ^= 1; }
#pragma unroll
                    for (int ks = 0; ks < 7; ++ks) {
                        if (ks < ksteps && !TC_KNOCK(2)) {
                            if (has_next && ks == kmid) {
                                mbar_wait(&t_empty[ts1], tp1 ^ 1);
                                mbar_wait(&b_full[s1], sp1);
                                tc_fence_after();
                                ready = true;
                            }
                            const uint64_t hk = desc_advance(h0, (uint32_t)ks * 2u * TC_N * 16u);
                            const uint64_t lk = desc_advance(l0, (uint32_t)ks * 2u * TC_N * 16u);
                            tc_mma_f16_ts(d0, a_hi + 8u * ks, hk, idesc, ks > 0 ? 1u : 0u);      // hi * hi
                            tc_mma_f16_ts(d0, a_hi + 8u * ks, lk, idesc, 1u);                    // hi * lo
                            tc_mma_f16_ts(d0, a_lo + 8u * ks, hk, idesc, 1u);                    // lo * hi
                        }
                    }
                    tc_commit(&b_empty[s]);      // the stage is reusable once these MMAs have read it
                    tc_commit(&t_full[ts]);      // accumulators complete
                    if (it == 4) TC_TRACE(tc_tb_ + 7);
                    if (it == 12) TC_TRACE(tc_tb_ + 11);
                    if (seg == 1 && c == sg.u0) TC_TRACE(tc_tb_ + 60);
                    s = s1; sp = sp1; ts = ts1; tp = tp1;
                }
                ++seg;
            }
            TC_TRACE(tc_tb_ + 3);
        }
        __syncwarp();
    } else if (warp < TC_FWD_WORKERS) {
        // ===== row-owning warps: P operand -> TMEM, then epilogue =====
        asm volatile("setmaxnreg.inc.sync.aligned.u32 224;" ::: "memory");
        const int ew = warp, g = ew >> 2, q4 = ew & 3;
        const int row = q4 * 32 + lane;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q4 * 32) << 16);
        constexpr int RW = (DP >= 64) ? 64 : 32;      // columns of R / w held per thread
        const int jbase = (DP == 128) ? 64 * g : 0;
        const float inv = 1.f / (TC_QSCALE * pow2_scale(p.scal[TS_AMAX_C]));      // undoes the operand scales (a power of two)
        TcSegIter si(p.segs, p.sch.upt, blockIdx.x);
        TcSeg sg;
        int it = 0, seg = 0;
        while (si.next(sg)) {
            const int b = sg.tile * TC_M + row;
            const bool ok = b < p.B;
            if (ew == 0 && lane == 0 && seg == 1) TC_TRACE(tc_tb_ + 58);
            // R (c) rows first: their loads are in flight while the P operand is copied
            float Rr[RW], Wr[RW];
            const float* rp = p.RT + (ok ? b : 0);
            // re-read per segment (opaque to the compiler): otherwise the 64 clamped offsets are hoisted out of the segment
            // loop and spilled across it
            int jlast;
            asm volatile("mov.b32 %0, %1;" : "=r"(jlast) : "r"(p.dp - 1));
#pragma unroll
            for (int c = 0; c < RW; ++c) Rr[c] = ldg_stream(rp + (size_t)min(jbase + c, jlast) * p.B);
            if (ew == 0 && lane == 0 && it == 0) TC_TRACE(tc_tb_ + 12);
            {
                // the segment's P operand (q rows x 2^12 as FP16 hi / lo planes, two relations per column: k_tc_prep_qt's
                // image of the tile, streamed into the operand ring ahead of the segment's chunks) -> TMEM.  Group g copies
                // columns [28 g, 28 g + 28) of each plane.  Segments after the first: this warp has seen t_full of the
                // previous segment's last chunk, so every MMA that read the old rows is done.
                const int r = it + seg;                        // ring stages filled before this one: chunks and P images
                mbar_wait(&b_full[r % nbs], (r / nbs) & 1);
                if (ew == 0 && lane == 0 && it == 0) TC_TRACE(tc_tb_ + 13);
                const uint4* img = reinterpret_cast<const uint4*>(smB + (size_t)(r % nbs) * B_BYTES) + row;
                const uint32_t a_hi_col = lane_base + TC_FWD_ACOL + 28u * g, a_lo_col = a_hi_col + KC;
#pragma unroll
                for (int c4 = 0; c4 < 7; ++c4) {
                    const uint32_t kq = 7u * g + c4;
                    if (kq < KQ8) {
                        const uint4 h = img[kq * TC_M], l = img[(KQ8 + kq) * TC_M];
                        const uint32_t hi[4] = {h.x, h.y, h.z, h.w}, lo[4] = {l.x, l.y, l.z, l.w};
                        tc_st4u(a_hi_col + 4u * c4, hi);
                        tc_st4u(a_lo_col + 4u * c4, lo);
                    }
                }
                tc_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(a_full);
                if (ew == 0 && lane == 0 && it == 0) TC_TRACE(tc_tb_ + 2);
                if (ew == 0 && lane == 0 && seg == 1) TC_TRACE(tc_tb_ + 63);
            }
#pragma unroll
            for (int c = 0; c < RW; ++c) {
                if (!(ok && jbase + c < p.dp)) Rr[c] = 0.f;
                Wr[c] = 0.f;
            }
            if (ew == 0 && lane == 0 && it == 0 && Rr[0] != -1.f) TC_TRACE(tc_tb_ + 8);
            if (ew == 0 && lane == 0 && seg == 1 && Rr[0] != -1.f) TC_TRACE(tc_tb_ + 61);
            for (int c = sg.u0; c < sg.u1; ++c, ++it) {
                const int ts = it % TC_TSTAGES;
                const uint32_t tph = (it / TC_TSTAGES) & 1;
                const int hc = 2 * c + g;                      // this group's half chunk
                const bool bil = hc < p.n_bil_half;
                const bool sp = !bil && hc < p.n_bil_half + p.n_sp_half;
                // L values this half chunk needs (issued before the wait so the loads overlap it)
                float L0 = 0.f, L1 = 0.f;
                int i0 = 0;
                if (bil) {
                    i0 = (DP == 128) ? (hc >> 1) : (DP == 64 ? hc : 2 * hc);
                    if (ok && i0 < p.d) L0 = p.LT[(size_t)i0 * p.B + b];
                    if (DP == 32 && ok && i0 + 1 < p.d) L1 = p.LT[(size_t)(i0 + 1) * p.B + b];
                }
                const bool etr = ew == 0 && lane == 0 && it == 8;
                if (etr) TC_TRACE(tc_tb_ + 53);
                mbar_wait(&t_full[ts], tph);
                tc_fence_after();
                if (etr) TC_TRACE(tc_tb_ + 54);
                if (!bil && !sp) {                             // padding half chunk: nothing to read
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&t_empty[ts]);
                    continue;
                }
                const int sc = hc - p.n_bil_half;
                float vsum = 0.f;
                // the 64 accumulator columns are consumed in two halves of 32 to bound register pressure
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    float t[32];
                    tc_ld32(lane_base + (uint32_t)(ts * TC_N + TC_H * g + 32 * hf), t);
                    if (hf == 1) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&t_empty[ts]);     // this group is done with the accumulator stage
                        if (etr) TC_TRACE(tc_tb_ + 55);
                    }
                    if (TC_KNOCK(4)) continue;
                    if (bil) {
                        if (DP >= 64) {
                            float v4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                            for (int x = 0; x < 32; ++x) {
                                v4[x & 3] = fmaf(t[x], Rr[(32 * hf + x) % RW], v4[x & 3]);
                                Wr[(32 * hf + x) % RW] = fmaf(t[x], L0, Wr[(32 * hf + x) % RW]);
                            }
                            vsum += (v4[0] + v4[1]) + (v4[2] + v4[3]);
                        } else {
                            const float Lh = hf == 0 ? L0 : L1;
                            float v4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                            for (int x = 0; x < 32; ++x) {
                                v4[x & 3] = fmaf(t[x], Rr[x % RW], v4[x & 3]);
                                Wr[x % RW] = fmaf(t[x], Lh, Wr[x % RW]);
                            }
                            if (ok && i0 + hf < p.d) p.vT[((size_t)g * p.dp + i0 + hf) * p.B + b] = inv * ((v4[0] + v4[1]) + (v4[2] + v4[3]));
                        }
                    } else if (ok) {
                        // selectional-preference rows: the accumulator row IS c1 / c2 (x the operand scales)
                        int which, jb;
                        if (DP == 128) { which = sc >> 1; jb = 64 * (sc & 1) + 32 * hf; }
                        else if (DP == 64) { which = sc; jb = 32 * hf; }
                        else { which = hf; jb = 0; }
                        float* o = p.spT + (size_t)which * p.dp * p.B + b;
#pragma unroll
                        for (int x = 0; x < 32; ++x)
                            if (jb + x < p.d) o[(size_t)(jb + x) * p.B] = inv * t[x];
                    }
                }
                if (DP >= 64 && bil && ok && i0 < p.d) p.vT[((size_t)g * p.dp + i0) * p.B + b] = inv * vsum;
                if (etr) TC_TRACE(tc_tb_ + 56);
            }
            if (ok) {
                float* wo = p.wT + ((size_t)sg.slot * 2 + g) * p.dp * p.B + b;
#pragma unroll
                for (int c = 0; c < RW; ++c) {
                    const int j = jbase + c;
                    if (j < p.dp) wo[(size_t)j * p.B] = inv * Wr[c];
                }
            }
            if (ew == 0 && lane == 0 && it <= (sg.u1 - sg.u0)) TC_TRACE(tc_tb_ + 9);     // first segment done
            ++seg;
        }
        if (ew == 0 && lane == 0) TC_TRACE(tc_tb_ + 4);
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) { TC_TRACE(tc_tb_ + 5); TC_TRACE_NS(tc_tb_ + 15); }
    if (warp == TC_FWD_WORKERS + 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------------------
// backward kernels: generated A operand in TMEM, 64 reduction rows per pipeline stage.
// TMEM map: accumulator [0,128) (NK <= 128 columns used); A stage s: hi at [128 + 128 s, +64), lo at [128 + 128 s + 64, +64);
//           dq: 3 A stages ([128, 512)); dC: 2 A stages ([128, 384)) and a second accumulator at [384, 512)
// generated operand  G[b,n]:  bilinear row n=(i,j): a_bi R_bj + L_bi Y2_bj ;  C1 row j: a_bj + G2_b L_bj ;  C2 row j: c_bj + G1_b R_bj
// Each of the 16 generator warps publishes 16 columns of a stage per hand-off (one mbarrier arrival per warp and stage).
// ------------------------------------------------------------------------------------------------------------
constexpr uint32_t TC_BWD_ACOL = 128;
constexpr int TC_DQ_ASTAGES = 3;
constexpr int TC_DC_ASTAGES = 2;
// Second accumulator of the dC contraction at [384, 512).  tcgen05.mma adds into the fp32 accumulator with truncation, so
// a long chain of MMAs into ONE accumulator drifts towards zero by ~2e-8 of the sum per MMA (measured at the target shape,
// profiles/r01_accum_chain.md: 1536 MMAs -> 3.4e-5 of ||dC||_inf, 180 MMAs -> 3.2e-6).  The reduction over examples is
// therefore dealt over two accumulators (even / odd stages, summed with a rounded fp32 add in the epilogue) and the
// schedule (tc_init) gives no segment more than TC_DC_MAX_STAGES stages of 24 MMAs per accumulator.
constexpr uint32_t TC_BWD_ACC2 = 384;
constexpr int TC_DC_MAX_STAGES = 16;   // stages (of 64 examples, 24 MMAs each) per accumulator: 384 MMAs
constexpr int TC_DQ_MAX_STAGES = 64;   // dq: stages (of 64 reduction rows) per segment: 1536 MMAs; random-sign terms drift less

// tiled transposes: job z copies src[b * stride + c] (b < B, c < cols) to dst[c * B + b], zero rows for cols <= c < cols_out,
// and folds |max| of the job's values into *amax (bits of a non-negative float; nullptr: skip).  They give the contraction
// kernels their [column][example] views (lane = example reads are coalesced) and the scales of the FP16 operands.
// img_rows != 0: the destination is a stack of STAGE IMAGES [b / 64][img_rows][TC_IMG_LD], the job's columns c in its first
// rows (64 examples per row, padded to 68 floats so that 16-byte shared-memory reads of consecutive rows are
// conflict-free): one contiguous block per stage that the dC kernel fetches with bulk copies.
// src2 != nullptr: the job copies src + coef[b * SC_N] * src2 instead (both rounded, as the one-tile dC kernel's generator
// rounds them): the selectional-preference rows a + G2 L, c + G1 R of the dC operand
constexpr int TC_IMG_LD = 68;
struct TrJob { const float* src; size_t stride; int cols, cols_out; float* dst; uint32_t* amax; int img_rows; const float* src2; const float* coef; };
struct TrJobs { TrJob j[6]; int B; };
__global__ void __launch_bounds__(256) k_tc_transpose(TrJobs jobs) {
    pdl_enter();
    __shared__ float tile[32][33];
    __shared__ uint32_t red[8];
    const TrJob jb = jobs.j[blockIdx.z];
    const int b0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    if (c0 >= jb.cols_out) return;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 8 rows of 32
    uint32_t m = 0;
    for (int r = ty; r < 32; r += 8) {
        const int b = b0 + r, c = c0 + tx;
        float v = 0.f;
        if (b < jobs.B && c < jb.cols) {
            v = jb.src[(size_t)b * jb.stride + c];
            if (jb.src2 != nullptr) v = __fadd_rn(v, __fmul_rn(jb.coef[(size_t)b * SC_N], jb.src2[(size_t)b * jb.stride + c]));
        }
        tile[r][tx] = v;
        m = max(m, __float_as_uint(fabsf(v)));
    }
    if (jb.amax != nullptr) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(kFull, m, o));
        if (tx == 0) red[ty] = m;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int c = c0 + r, b = b0 + tx;
        if (c < jb.cols_out && b < jobs.B) {
            if (jb.img_rows) jb.dst[((size_t)(b >> 6) * jb.img_rows + c) * TC_IMG_LD + (b & 63)] = tile[tx][r];
            else jb.dst[(size_t)c * jobs.B + b] = tile[tx][r];
        }
    }
    if (jb.amax != nullptr && threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) m = max(m, red[w]);
        atomicMax(jb.amax, m);
    }
}

// v, w of a contraction pass: transposed partial buffers -> row-major per-example vectors ev[b][slotV | slotW][j]
//   vT [2][dp][B]        DP=128: both epilogue groups hold a half-row partial; DP=64: group j%2; DP=32: group (j/2)%2
//   wT [slot][2][dp][B]  sum over the slots of the example's tile (DP=128: only group j/64 holds column j; else both groups)
//   spT [2][dp][B]       c1, c2 -> ev[b][E_C1 | E_C2][j] (forward pass only; nullptr otherwise)
// zero_amax: the forward pass's combine also clears the |max| words the NEXT transposes (a, c, Y2, the SP images) accumulate into
__global__ void __launch_bounds__(256) k_tc_combine(const float* __restrict__ vT, const float* __restrict__ wT, const float* __restrict__ spT,
                                                    float* __restrict__ ev, int B, int d, int dp, int DP, TcSched sch, int slotV, int slotW,
                                                    uint32_t* __restrict__ zero_amax) {
    pdl_enter();
    __shared__ float tv[32][33], tw[32][33], t1[32][33], t2[32][33];
    if (zero_amax != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < 4) zero_amax[TS_AMAX_A + threadIdx.x] = 0u;
    const int b0 = blockIdx.x * 32, j0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int ns = tcs_nslots(sch, b0 >> 7);                    // the 32 examples of a block share a 128-example tile
    const size_t plane = (size_t)dp * B;
    constexpr int MAXP = 16;                                    // partial planes summed per element (slots x groups)
    for (int r = ty; r < 32; r += 8) {
        const int j = j0 + r, b = b0 + tx;
        float v = 0.f, w = 0.f, c1 = 0.f, c2 = 0.f;
        if (j < d && b < B) {
            const size_t idx = (size_t)j * B + b;
            // every load of the element is issued before the first add (one memory latency, not one per slot)
            float v0, v1 = 0.f;
            if (DP == 128) { v0 = vT[idx]; v1 = vT[plane + idx]; }
            else if (DP == 64) v0 = vT[(size_t)(j & 1) * plane + idx];
            else v0 = vT[(size_t)((j >> 1) & 1) * plane + idx];
            const int np = DP == 128 ? ns : 2 * ns;                     // planes of wT that hold column j
            const int first = DP == 128 ? (j >> 6) : 0, step = DP == 128 ? 2 : 1;
            // unconditional loads from clamped plane indices (volatile asm: issued back to back, one latency); planes beyond np
            // re-read the last valid one and are dropped by the select.  (As conditional loads they compiled into a
            // load - add chain through one register.)
            float wv[MAXP];
#pragma unroll
            for (int s = 0; s < MAXP; ++s) wv[s] = ldg_stream(wT + (size_t)(first + step * min(s, np - 1)) * plane + idx);
            for (int s = MAXP; s < np; ++s) w += wT[(size_t)(first + step * s) * plane + idx];      // (more than 16 planes: tiny tiles only)
            if (spT != nullptr) { c1 = spT[idx]; c2 = spT[plane + idx]; }
            v = v0 + v1;
#pragma unroll
            for (int s = 0; s < MAXP; ++s) w += s < np ? wv[s] : 0.f;
        }
        tv[r][tx] = v;
        tw[r][tx] = w;
        t1[r][tx] = c1;
        t2[r][tx] = c2;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int b = b0 + r, j = j0 + tx;
        if (b < B && j < d) {
            float* e = ev + (size_t)b * E_NV * dp;
            e[slotV * dp + j] = tv[tx][r];
            e[slotW * dp + j] = tw[tx][r];
            if (spT != nullptr) { e[E_C1 * dp + j] = t1[tx][r]; e[E_C2 * dp + j] = t2[tx][r]; }
        }
    }
}

// shared skeleton pieces of the two backward kernels ------------------------------------------------------------
struct BwdBars {
    uint64_t* a_full; uint64_t* a_empty; uint64_t* b_full; uint64_t* b_empty; uint64_t* acc_full; uint64_t* acc_empty; uint32_t* tmem_slot;
};

__device__ __forceinline__ BwdBars bwd_setup(uint8_t* smem_raw, uint32_t ST_BYTES, int warp, uint32_t& tmem_base, uint32_t drain_warps) {
    BwdBars br;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + TC_BSTAGES * ST_BYTES);
    br.a_full = bars;                 // [4] 16 generator-warp arrivals
    br.a_empty = bars + 4;            // [4] tcgen05.commit
    br.b_full = bars + 8;             // [4] bulk-copy tx
    br.b_empty = bars + 12;           // [4] tcgen05.commit
    br.acc_full = bars + 16;          // tcgen05.commit behind a segment's last MMA
    br.acc_empty = bars + 17;         // drain-warp arrivals: the accumulators may be overwritten by the next segment
    br.tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);
    if (threadIdx.x == 0) {
        for (int s = 0; s < 4; ++s) { mbar_init(&br.a_full[s], 16); mbar_init(&br.a_empty[s], 1); }
        for (int s = 0; s < 4; ++s) { mbar_init(&br.b_full[s], 1); mbar_init(&br.b_empty[s], 1); }
        mbar_init(br.acc_full, 1);
        mbar_init(br.acc_empty, drain_warps);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == TC_BWD_WORKERS + 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(br.tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    tmem_base = *br.tmem_slot;
    return br;
}

// producer of one segment: stage `st0 + lt` of the operand = two consecutive 32-row chunks, one bulk copy
__device__ __forceinline__ void bwd_produce(const BwdBars& br, uint8_t* smB, const uint8_t* src, uint32_t ST_BYTES, int st0, int nst, int it0) {
    for (int lt = 0; lt < nst; ++lt) {
        const int git = it0 + lt, s = git % TC_BSTAGES;
        mbar_wait(&br.b_empty[s], ((git / TC_BSTAGES) & 1) ^ 1);
        if (TC_KNOCK(1) && git >= TC_BSTAGES) { mbar_arrive(&br.b_full[s]); continue; }
        mbar_expect_tx(&br.b_full[s], ST_BYTES);
        bulk_g2s_pieces(smB + (size_t)s * ST_BYTES, src + (size_t)(st0 + lt) * ST_BYTES, ST_BYTES, &br.b_full[s]);
    }
}

// MMAs of one segment: 24 per stage (2 chunks x 4 k-steps x {hi.hi, hi.lo, lo.hi}); stage lt accumulates into accumulator
// lt % nacc, whose first MMA overwrites; the commit behind the last stage signals acc_full
template <int NAS>
__device__ __forceinline__ void bwd_mma_segment(const BwdBars& br, uint8_t* smB, uint32_t ST_BYTES, int NK, uint32_t tmem_base, int nst,
                                                int it0, int nacc) {
    TC_TRACE_INIT();
    const uint32_t idesc = make_idesc_tf32(TC_M, NK);
    const uint32_t CH_BYTES = ST_BYTES / 2;
    for (int lt = 0; lt < nst; ++lt) {
        const int git = it0 + lt, s = git % TC_BSTAGES, as = git % NAS;
        mbar_wait(&br.a_full[as], (git / NAS) & 1);
        mbar_wait(&br.b_full[s], (git / TC_BSTAGES) & 1);
        tc_fence_after();
        if ((threadIdx.x & 31) == 0 && git == 8) TC_TRACE(38);
        if ((threadIdx.x & 31) == 0 && git == 24) TC_TRACE(43);
        if (elect_one()) {
            const uint32_t a_hi = tmem_base + TC_BWD_ACOL + 128u * as, a_lo = a_hi + 64u;
            const uint32_t acc = tmem_base + ((nacc == 2 && (lt & 1)) ? TC_BWD_ACC2 : 0u);
            const uint32_t b_base = smem_u32(smB + (size_t)s * ST_BYTES);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                uint64_t dbh = make_desc(b_base + h * CH_BYTES, (uint32_t)NK * 16u, 128u);
                uint64_t dbl = make_desc(b_base + h * CH_BYTES + 8u * (uint32_t)NK * 16u, (uint32_t)NK * 16u, 128u);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    const uint32_t col = 32u * h + 8u * ks;
                    tc_mma_tf32_ts(acc, a_hi + col, dbh, idesc, (lt >= nacc || h > 0 || ks > 0) ? 1u : 0u);
                    tc_mma_tf32_ts(acc, a_hi + col, dbl, idesc, 1u);
                    tc_mma_tf32_ts(acc, a_lo + col, dbh, idesc, 1u);
                    dbh = desc_advance(dbh, 2u * (uint32_t)NK * 16u);
                    dbl = desc_advance(dbl, 2u * (uint32_t)NK * 16u);
                }
            }
            tc_commit(&br.a_empty[as]);
            tc_commit(&br.b_empty[s]);
            if (lt == nst - 1) tc_commit(br.acc_full);
        }
        __syncwarp();
        if ((threadIdx.x & 31) == 0 && git == 8) TC_TRACE(39);
        if ((threadIdx.x & 31) == 0 && git == 24) TC_TRACE(44);
    }
}

// 8 generated values -> hi / lo planes of A stage `as`, columns col8 .. col8 + 7 (the caller waits for the stores)
__device__ __forceinline__ void bwd_store8(uint32_t lane_base, int as, int col8, const float (&g)[8]) {
    float hi[8], lo[8];
    split8(g, hi, lo);
    const uint32_t col = lane_base + TC_BWD_ACOL + 128u * as + (uint32_t)col8;
    tc_st8(col, hi);
    tc_st8(col + 64u, lo);
}
// the warp's columns of stage `as` are in TMEM: one arrival
__device__ __forceinline__ void bwd_publish(const BwdBars& br, int as, int lane) {
    tc_wait_st();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&br.a_full[as]);
}

struct TcDqArgs {
    const uint4* bop2;      // Cf^T stages [st][hi/lo][oct 0..15][NK] x 16 B (FP16 pairs, scaled by s_C)
    const float* sc;
    const float* aT; const float* LT; const float* RT; const float* cT; const float* Y2T;   // [dp][B] transposed a, L, R, c, Y2
    float* dqT;             // [slot][NK][B]  dq partial per segment slot, transposed (coalesced stores)
    const uint32_t* scal;   // device scalars (TcScal): |max| of the dense tensors and of L, R, a, c, Y2
    float g_bound;          // S / Z: upper bound of G1_b, G2_b (sums of S terms in (0, 1/Z))
    int B, d, dp, K, NK;
    int n_bil_rows;         // reduction rows holding bilinear rows (a multiple of 128)
    TcSched sch;            // units = stages of 128 reduction rows, tiles = example tiles
    const int4* segs;       // sch's per-CTA table (TcSegIter)
};

// MMAs of one dq segment: 24 kind::f16 MMAs per stage (8 k-steps of 16 reduction rows x {hi.hi, hi.lo, lo.hi}); issued by ONE
// elected thread, which takes the barrier waits of stage lt+1 in the middle of stage lt's MMAs (the pipe keeps queued work)
__device__ __forceinline__ void dq_mma_segment(const BwdBars& br, uint8_t* smB, uint32_t ST_BYTES, int NK, uint32_t tmem_base, int nst,
                                               int it0) {
    TC_TRACE_INIT();
    constexpr int NAS = TC_DQ_ASTAGES;
    const uint32_t idesc = make_idesc_f16(TC_M, NK);
    bool ready = false;
    for (int lt = 0; lt < nst; ++lt) {
        const int git = it0 + lt, s = git % TC_BSTAGES, as = git % NAS;
        if (!ready) {
            mbar_wait(&br.a_full[as], (git / NAS) & 1);
            mbar_wait(&br.b_full[s], (git / TC_BSTAGES) & 1);
            tc_fence_after();
        }
        ready = false;
        if (git == 8) TC_TRACE(22);
        if (git == 24) TC_TRACE(27);
        const uint32_t a_hi = tmem_base + TC_BWD_ACOL + 128u * as, a_lo = a_hi + 64u;
        const uint32_t b_base = smem_u32(smB + (size_t)s * ST_BYTES);
        uint64_t dbh = make_desc(b_base, (uint32_t)NK * 16u, 128u);
        uint64_t dbl = make_desc(b_base + 16u * (uint32_t)NK * 16u, (uint32_t)NK * 16u, 128u);
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) {
            if (TC_KNOCK(2)) continue;
            if (ks == 4 && lt + 1 < nst) {
                const int g1 = git + 1;
                mbar_wait(&br.a_full[g1 % NAS], (g1 / NAS) & 1);
                mbar_wait(&br.b_full[g1 % TC_BSTAGES], (g1 / TC_BSTAGES) & 1);
                tc_fence_after();
                ready = true;
            }
            tc_mma_f16_ts(tmem_base, a_hi + 8u * ks, dbh, idesc, (lt > 0 || ks > 0) ? 1u : 0u);
            tc_mma_f16_ts(tmem_base, a_hi + 8u * ks, dbl, idesc, 1u);
            tc_mma_f16_ts(tmem_base, a_lo + 8u * ks, dbh, idesc, 1u);
            dbh = desc_advance(dbh, 2u * (uint32_t)NK * 16u);
            dbl = desc_advance(dbl, 2u * (uint32_t)NK * 16u);
        }
        tc_commit(&br.a_empty[as]);
        tc_commit(&br.b_empty[s]);
        if (lt == nst - 1) tc_commit(br.acc_full);
        if (git == 8) TC_TRACE(23);
        if (git == 24) TC_TRACE(28);
    }
}

// 16 generated (scaled) values -> FP16 hi / lo pairs of A stage `as`, packed columns col8 .. col8 + 7
__device__ __forceinline__ void dq_store16(uint32_t lane_base, int as, int col8, const float (&g)[16]) {
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) split_h2(g[2 * u], g[2 * u + 1], hi[u], lo[u]);
    const uint32_t col = lane_base + TC_BWD_ACOL + 128u * as + (uint32_t)col8;
    tc_st8u(col, hi);
    tc_st8u(col + 64u, lo);
}

// dq: rows = examples, 128 reduction rows per stage.  Generator thread = (row b, column group cg: reduction rows 32 cg .. +31
// of the stage = 16 packed TMEM columns); the R / Y2 values it needs for every bilinear stage are cached in registers
// (X, Y), a_bi / L_bi come coalesced from the transposed copies, one stage ahead of their use.  Bilinear stage st holds
// 128 / DP rows i: the thread's row is i = (128 / DP) st + (32 cg) / DP, its columns j = (32 cg) % DP + 0..31.
template <int DP>
__global__ void __launch_bounds__(TC_BWD_THREADS, 1) k_tc_dq(TcDqArgs p) {
    pdl_enter();
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    TC_TRACE_INIT();
    constexpr int NAS = TC_DQ_ASTAGES;
    constexpr int RPS = 128 / DP;                            // bilinear rows i per stage
    const uint32_t ST_BYTES = 2u * 16u * (uint32_t)p.NK * 16u;
    uint8_t* smB = smem_raw;
    uint32_t tmem_base;
    if (threadIdx.x == 0) { TC_TRACE(16); TC_TRACE_NS(30); TC_TRACE_SEGS(p.sch, 96, 103); }
    const BwdBars br = bwd_setup(smem_raw, ST_BYTES, warp, tmem_base, TC_BWD_WORKERS);
    if (threadIdx.x == 0) TC_TRACE(17);

    if (warp >= TC_BWD_WORKERS) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 32;" ::: "memory");
    }
    if (warp == TC_BWD_WORKERS + 1) {
        if (lane == 0) {
            TcSegIter si(p.segs, p.sch.upt, blockIdx.x);
            TcSeg sg;
            int it = 0;
            while (si.next(sg)) {
                bwd_produce(br, smB, reinterpret_cast<const uint8_t*>(p.bop2), ST_BYTES, sg.u0, sg.u1 - sg.u0, it);
                it += sg.u1 - sg.u0;
            }
        }
    } else if (warp == TC_BWD_WORKERS) {
        if (elect_one()) {
            TcSegIter si(p.segs, p.sch.upt, blockIdx.x);
            TcSeg sg;
            int it = 0, seg = 0;
            while (si.next(sg)) {
                if (seg > 0) {                                   // the previous segment's accumulator has been drained
                    mbar_wait(br.acc_empty, (seg - 1) & 1);
                    tc_fence_after();
                    if (seg == 1) TC_TRACE(99);
                }
                dq_mma_segment(br, smB, ST_BYTES, p.NK, tmem_base, sg.u1 - sg.u0, it);
                it += sg.u1 - sg.u0;
                ++seg;
            }
            TC_TRACE(19);
        }
        __syncwarp();
    } else if (warp < TC_BWD_WORKERS) {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 112;" ::: "memory");
        const int gw = warp, q4 = gw & 3, cg = gw >> 2;              // lane quarter, column group
        const int row = q4 * 32 + lane;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q4 * 32) << 16);
        const int rsel = (32 * cg) / DP, j0 = (32 * cg) % DP;        // which of the stage's rows, first column
        const int n_bil_st = p.n_bil_rows / TC_M;
        // operand scale of the generated values: a power of two from a bound of |G| (triangle inequality over the |max| of
        // the factors; G1_b, G2_b <= S / Z) and the scale of the dense operand, undone in the epilogue
        float sG, inv;
        {
            const float aL = __uint_as_float(p.scal[TS_AMAX_L]), aR = __uint_as_float(p.scal[TS_AMAX_R]);
            const float aA = __uint_as_float(p.scal[TS_AMAX_A]), aC = __uint_as_float(p.scal[TS_AMAX_CV]);
            const float aY = __uint_as_float(p.scal[TS_AMAX_Y2]);
            const float bound = fmaxf(fmaf(aA, aR, aL * aY), fmaxf(fmaf(p.g_bound, aL, aA), fmaf(p.g_bound, aR, aC)));
            sG = pow2_scale(__float_as_uint(bound));
            inv = 1.f / (sG * pow2_scale(p.scal[TS_AMAX_C]));
        }
        TcSegIter si(p.segs, p.sch.upt, blockIdx.x);
        TcSeg sg;
        int it = 0, seg = 0;
        while (si.next(sg)) {
            const int b = sg.tile * TC_M + row;
            const bool ok = b < p.B;
            const float* scb = p.sc + (size_t)(ok ? b : 0) * SC_N;
            [[maybe_unused]] const bool tr0 = gw == 0 && lane == 0;
            if (tr0 && seg == 1) TC_TRACE(97);
            // register cache of the thread's 32 columns of R and Y2 (coalesced loads from the transposed copies)
            float X[32], Y[32];
            {
                const float* rp = p.RT + (ok ? b : 0);
                const float* yp = p.Y2T + (ok ? b : 0);
                const int jlast = p.dp - 1;
#pragma unroll
                for (int u = 0; u < 32; ++u) {
                    X[u] = ldg_stream(rp + (size_t)min(j0 + u, jlast) * p.B);
                    Y[u] = ldg_stream(yp + (size_t)min(j0 + u, jlast) * p.B);
                }
#pragma unroll
                for (int u = 0; u < 32; ++u)
                    if (!(ok && j0 + u < p.dp)) { X[u] = 0.f; Y[u] = 0.f; }
            }
            if (gw == 0 && lane == 0 && it == 0 && X[0] != -1.f) TC_TRACE(29);
            if (tr0 && seg == 1 && X[0] != -1.f) TC_TRACE(98);
            const int st0 = sg.u0, st1 = sg.u1, nst = st1 - st0;
            const int nbil = max(0, min(st1, n_bil_st) - st0);
            float ai_n = 0.f, li_n = 0.f;
            {
                const int i = RPS * st0 + rsel;
                if (nbil > 0 && ok && i < p.dp) {
                    ai_n = p.aT[(size_t)i * p.B + b];
                    li_n = p.LT[(size_t)i * p.B + b];
                }
            }
            int lt = 0;
            for (; lt < nbil; ++lt) {
                const int git = it + lt, as = git % NAS;
                const float ai = ai_n * sG, li = li_n * sG;
                const int i_next = RPS * (st0 + lt + 1) + rsel;
                const bool more = ok && i_next < p.dp && lt + 1 < nbil;
                ai_n = more ? p.aT[(size_t)i_next * p.B + b] : 0.f;
                li_n = more ? p.LT[(size_t)i_next * p.B + b] : 0.f;
                const bool tr = gw == 0 && lane == 0 && git == 8;
                if (tr) TC_TRACE(24);
                mbar_wait(&br.a_empty[as], ((git / NAS) & 1) ^ 1);
                tc_fence_after();
                if (tr) TC_TRACE(25);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (TC_KNOCK(4)) continue;
                    float g[16];
#pragma unroll
                    for (int u = 0; u < 16; ++u) g[u] = fmaf(ai, X[16 * h + u], li * Y[16 * h + u]);
                    dq_store16(lane_base, as, 16 * cg + 8 * h, g);
                }
                bwd_publish(br, as, lane);
                if (tr) TC_TRACE(26);
                if (gw == 0 && lane == 0 && git == 0) TC_TRACE(18);
                if (tr0 && seg == 1 && lt == 0) TC_TRACE(104);
            }
            // selectional-preference rows (at most two stages per tile): coalesced loads from the transposed copies
            for (; lt < nst; ++lt) {
                const int git = it + lt, as = git % NAS;
                const int m = (st0 + lt) * TC_M - p.n_bil_rows + 32 * cg;
                const int which = m / DP, jj = m - which * DP;
                const float* sx = which == 0 ? p.aT : p.cT;
                const float* sy = which == 0 ? p.LT : p.RT;
                const float s2 = (ok && which < 2) ? sG * (which == 0 ? scb[SC_G2] : scb[SC_G1]) : 0.f;
                if (tr0 && lt == nbil) TC_TRACE(100);
                mbar_wait(&br.a_empty[as], ((git / NAS) & 1) ^ 1);
                tc_fence_after();
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    float g[16];
#pragma unroll
                    for (int u = 0; u < 16; ++u) {
                        const int j = jj + 16 * h + u;
                        const bool in = ok && which < 2 && j < p.dp;
                        g[u] = in ? fmaf(s2, sy[(size_t)j * p.B + b], sG * sx[(size_t)j * p.B + b]) : 0.f;
                    }
                    dq_store16(lane_base, as, 16 * cg + 8 * h, g);
                }
                bwd_publish(br, as, lane);
                if (tr0 && lt == nst - 1) TC_TRACE(101);
            }
            it += nst;
            {
                // ===== epilogue: accumulator row -> dq partial of this segment's slot.  All 16 warps drain: warp (q4, cg)
                // takes the 32-column chunks 32 cg, 32 cg + 128, ... of its lane quarter (NK <= 112: one chunk each), so the
                // next segment's MMAs - and the CTA's exit - wait for a quarter of the tcgen05.ld / store sequence =====
                mbar_wait(br.acc_full, seg & 1);
                tc_fence_after();
                if (tr0 && seg == 0) TC_TRACE(102);
                float* o = p.dqT + (size_t)sg.slot * p.NK * p.B + (ok ? b : 0);
                for (int c0 = 32 * cg; c0 < p.NK; c0 += 128) {
                    float t[32];
                    tc_ld32(lane_base + (uint32_t)c0, t);
                    if (ok) {
#pragma unroll
                        for (int x = 0; x < 32; ++x)
                            if (c0 + x < p.NK) o[(size_t)(c0 + x) * p.B] = inv * t[x];
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(br.acc_empty);
            }
            ++seg;
        }
        if (gw == 0 && lane == 0) TC_TRACE(20);
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) { TC_TRACE(21); TC_TRACE_NS(31); }
    if (warp == TC_BWD_WORKERS + 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// dC: rows = operand rows n (128-row tiles), reduction over examples in stages of 64, TF32 pairs.  The whole-dC fallback of
// the two-tile kernel below: it runs only where that one cannot (B % 4 != 0, or its stages do not fit in shared memory).
struct TcDcArgs {
    const float4* pop3;     // q^T chunks [bc][hi/lo][8][NK]
    const float* ev; const float* sc; const float* aT; const float* LT;
    float* out;             // gC_part [slot][units*d*K]
    int B, d, dp, K, NK, DP;
    int n_bil_rows, n_rows_total, hasM;
    int nacc;               // TMEM accumulators the example stages are dealt over (1 or 2)
    int share;              // most stages one CTA handles (sizes the per-example scalar staging)
    size_t split_stride;    // units*d*K
    TcSched sch;            // units = stages of 64 examples, tiles = 128-row tiles of the operand rows
    const int4* segs;       // sch's per-CTA table (TcSegIter)
};

__global__ void __launch_bounds__(TC_BWD_THREADS, 1) k_tc_dc(TcDcArgs p) {
    pdl_enter();
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    TC_TRACE_INIT();
    constexpr int NAS = TC_DC_ASTAGES;
    const uint32_t ST_BYTES = 2u * 2u * 8u * (uint32_t)p.NK * 16u;
    uint8_t* smB = smem_raw;
    if (threadIdx.x == 0) { TC_TRACE(32); TC_TRACE_NS(46); }
    // Per-example scalars of the generated operand, staged once in shared memory for every segment of the CTA.  A 32-row
    // quarter of a tile is one bilinear row i (P1 = a_bi, P2 = L_bi) or one selectional-preference table (P1 = 1,
    // P2 = G2_b | G1_b); a tile holds TC_M / DP such sources.  Coalesced reads of the transposed copies aT / LT.
    const int nsrc = TC_M / p.DP;
    const int nbc = p.share * TC_SR;
    float* sP1 = reinterpret_cast<float*>(smem_raw + TC_BSTAGES * ST_BYTES + 256);
    float* sP2 = sP1 + (size_t)nsrc * nbc;
    {
        TcSegIter si(p.segs, p.sch.upt, blockIdx.x);
        TcSeg sg;
        int off = 0;                                        // example offset of the segment inside the staging area
        while (si.next(sg)) {
            const int ne = (sg.u1 - sg.u0) * TC_SR;
            for (int idx = threadIdx.x; idx < nsrc * ne; idx += blockDim.x) {
                const int src = idx / ne, bl = idx - src * ne;
                const int b = sg.u0 * TC_SR + bl;
                const int n0 = sg.tile * TC_M + src * p.DP;
                float v1 = 0.f, v2 = 0.f;
                if (b < p.B) {
                    if (n0 < p.n_bil_rows) {
                        const int i = n0 / p.DP;
                        if (i < p.d) { v1 = p.aT[(size_t)i * p.B + b]; v2 = p.LT[(size_t)i * p.B + b]; }
                    } else if (n0 < p.n_rows_total && (n0 - p.n_bil_rows) / p.DP < 2) {
                        v1 = 1.f;
                        v2 = p.sc[(size_t)b * SC_N + ((n0 - p.n_bil_rows) / p.DP == 0 ? SC_G2 : SC_G1)];
                    }
                }
                sP1[(size_t)src * nbc + off + bl] = v1;
                sP2[(size_t)src * nbc + off + bl] = v2;
            }
            off += ne;
        }
    }
    uint32_t tmem_base;
    const BwdBars br = bwd_setup(smem_raw, ST_BYTES, warp, tmem_base, 4);  // __syncthreads inside: staging visible
    if (threadIdx.x == 0) TC_TRACE(33);

    if (warp >= TC_BWD_WORKERS) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 32;" ::: "memory");
    }
    if (warp == TC_BWD_WORKERS + 1) {
        if (lane == 0) {
            TcSegIter si(p.segs, p.sch.upt, blockIdx.x);
            TcSeg sg;
            int it = 0;
            while (si.next(sg)) {
                bwd_produce(br, smB, reinterpret_cast<const uint8_t*>(p.pop3), ST_BYTES, sg.u0, sg.u1 - sg.u0, it);
                it += sg.u1 - sg.u0;
            }
        }
    } else if (warp == TC_BWD_WORKERS) {
        TcSegIter si(p.segs, p.sch.upt, blockIdx.x);
        TcSeg sg;
        int it = 0, seg = 0;
        while (si.next(sg)) {
            if (seg > 0) {                                   // the previous segment's accumulators have been drained
                mbar_wait(br.acc_empty, (seg - 1) & 1);
                tc_fence_after();
            }
            bwd_mma_segment<NAS>(br, smB, ST_BYTES, p.NK, tmem_base, sg.u1 - sg.u0, it, p.nacc);
            it += sg.u1 - sg.u0;
            ++seg;
        }
        if (lane == 0) TC_TRACE(35);
    } else if (warp < TC_BWD_WORKERS) {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 112;" ::: "memory");
        const int gw = warp, q4 = gw & 3, cg = gw >> 2;         // lane quarter; examples 16 cg .. 16 cg + 15 of a stage
        const int row = q4 * 32 + lane;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q4 * 32) << 16);
        const size_t estride = (size_t)E_NV * p.dp;
        const int src = q4 / (p.DP >> 5);
        TcSegIter si(p.segs, p.sch.upt, blockIdx.x);
        TcSeg sg;
        int it = 0, seg = 0, off = 0;
        while (si.next(sg)) {
            const int n = sg.tile * TC_M + row;
            // decode the row once: g(b) = P1(b) * X(b) + P2(b) * Y(b)
            int type = -1, i = 0, j = 0;          // -1: padding row (zero)
            if (n < p.n_bil_rows) {
                i = n / p.DP; j = n - i * p.DP;
                if (i < p.d && j < p.d) type = 0;
            } else if (n < p.n_rows_total) {
                const int m = n - p.n_bil_rows;
                const int which = m / p.DP;
                j = m - which * p.DP;
                if (j < p.d && which < 2) type = 1 + which;
            }
            int oX = 0, oY = 0;
            if (type == 0) { oX = E_R * p.dp + j; oY = E_Y2 * p.dp + j; }
            else if (type == 1) { oX = E_A * p.dp + j; oY = E_L * p.dp + j; }
            else if (type == 2) { oX = E_CV * p.dp + j; oY = E_R * p.dp + j; }
            const float* s1 = sP1 + (size_t)src * nbc + off + 16 * cg;
            const float* s2 = sP2 + (size_t)src * nbc + off + 16 * cg;
            const int nst = sg.u1 - sg.u0, nh = 2 * nst;
            const int e0 = sg.u0 * TC_SR + 16 * cg;              // first example of this thread in the segment's first stage
            // Half-stage software pipeline: the 16 per-lane loads of half hh+1 are issued before half hh is generated
            // (register double buffer), so the generator loop does not pay a memory latency per hand-off.
            auto load = [&](int hh, float (&x)[8], float (&y)[8]) {
                const int b0 = e0 + (hh >> 1) * TC_SR + 8 * (hh & 1);
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const float* evb = p.ev + (size_t)min(b0 + u, p.B - 1) * estride;
                    x[u] = evb[oX];
                    y[u] = evb[oY];
                }
            };
            auto process = [&](int hh, const float (&x)[8], const float (&y)[8]) {
                const int lt = hh >> 1, git = it + lt, as = git % NAS, half = hh & 1;
                const int b0 = e0 + lt * TC_SR + 8 * half;
                const float* q1 = s1 + lt * TC_SR + 8 * half;
                const float* q2 = s2 + lt * TC_SR + 8 * half;
                const float4 pa = *reinterpret_cast<const float4*>(q1), pb = *reinterpret_cast<const float4*>(q1 + 4);
                const float4 qa = *reinterpret_cast<const float4*>(q2), qb = *reinterpret_cast<const float4*>(q2 + 4);
                const float p1[8] = {pa.x, pa.y, pa.z, pa.w, pb.x, pb.y, pb.z, pb.w};
                const float p2[8] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
                float g[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) g[u] = (type >= 0 && b0 + u < p.B) ? fmaf(p1[u], x[u], p2[u] * y[u]) : 0.f;
                const bool tr = gw == 0 && lane == 0 && git == 8;
                if (half == 0) {
                    if (tr) TC_TRACE(40);
                    mbar_wait(&br.a_empty[as], ((git / NAS) & 1) ^ 1);
                    tc_fence_after();
                    if (tr) TC_TRACE(41);
                }
                bwd_store8(lane_base, as, 16 * cg + 8 * half, g);
                if (half == 1) {
                    bwd_publish(br, as, lane);
                    if (tr) TC_TRACE(42);
                }
            };
            float xa[8], ya[8], xb[8], yb[8];
            load(0, xa, ya);
            for (int hh = 0; hh < nh; hh += 2) {          // nh is even
                load(hh + 1, xb, yb);
                process(hh, xa, ya);
                if (hh + 2 < nh) load(hh + 2, xa, ya);
                process(hh + 1, xb, yb);
            }
            it += nst;
            off += nst * TC_SR;
            if (gw < 4) {
                mbar_wait(br.acc_full, seg & 1);
                tc_fence_after();
                // destination inside the slot's block: units are [bilinear rows i][C1][C2], each [d][K]
                size_t o_off = 0;
                if (type == 0) o_off = ((size_t)i * p.d + j) * p.K;
                else if (type > 0) o_off = ((size_t)((p.hasM ? p.d : 0) + (type - 1)) * p.d + j) * p.K;
                float* o = p.out + (size_t)sg.slot * p.split_stride + o_off;
                for (int c0 = 0; c0 < p.NK; c0 += 32) {
                    float t[32];
                    tc_ld32(lane_base + (uint32_t)c0, t);
                    if (p.nacc == 2 && nst > 1) {            // odd stages went to the second accumulator
                        float t2[32];
                        tc_ld32(lane_base + TC_BWD_ACC2 + (uint32_t)c0, t2);
#pragma unroll
                        for (int x = 0; x < 32; ++x) t[x] += t2[x];
                    }
                    if (type >= 0) store_row32(o + c0, t, p.K - c0, (p.K & 3) == 0);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(br.acc_empty);
            }
            ++seg;
        }
        if (gw == 0 && lane == 0) TC_TRACE(36);
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) { TC_TRACE(37); TC_TRACE_NS(47); }
    if (warp == TC_BWD_WORKERS + 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------------------
// dC, FP16 pairs, TWO 128-row tiles per CTA (rows n of tiles 2 tp and 2 tp + 1: the same columns j,
// different rows i): every R_bj / Y2_bj the generators read serves both tiles, and nothing in the loop is a per-thread
// global load - the one-tile kernel above spent its time on lane-strided L2 reads (47 % of the MMA floor, in-kernel trace).
//   per stage of 64 examples: bulk copies bring the stage images of R and Y2 ([j][64 examples], rows padded to 68 floats),
//   the per-example scalars a_bi, L_bi of the tiles' rows i (64 floats each, straight from the transposed copies) and the
//   q^T operand stage into shared memory; generator thread = (tile row n_l = lane + 32 q4, example group cg): 16 examples
//   per stage, both tiles; TMEM: accumulators [0,128) (tile A) and [128,256) (tile B), A stage s: tile t at
//   [256 + 128 s + 64 t, +64) = 32 packed hi + 32 packed lo columns.  One accumulator per tile: a segment never exceeds
//   TC_DC2_MAX_STAGES stages = 384 MMAs per accumulator (the chain bound of profiles/r01_accum_chain.md).
// The last pair of the schedule (n_bil_pairs) is the selectional-preference pair: its stage image holds the generated rows
// themselves, C1 rows a + G2 L then C2 rows c + G1 R ([2 DP][TC_IMG_LD], built by the transposes after scoring), so its
// generators only scale them; DP = 128: tile A = C1, tile B = C2; DP <= 64: both in tile A.
// Needs B % 4 == 0 (16-byte aligned slices of the transposed copies); other batches use k_tc_dc.
// ------------------------------------------------------------------------------------------------------------
constexpr int TC_DC2_BSTAGES = 3;      // q^T operand stages (28 KB each at K = 100)
constexpr int TC_DC2_XSTAGES = 2;      // image stages (R, Y2: 34 KB each at d = 128, + scalars)
constexpr int TC_DC2_MAX_STAGES = 32;
constexpr uint32_t TC_DC2_ACOL = 256;

struct TcDc2Args {
    const uint4* pop4;      // q^T stages [st][hi/lo][oct 0..7][NK] x 16 B
    const float* Rimg; const float* Yimg;     // stage images [st][j < DP][TC_IMG_LD]
    const float* SPimg;                       // selectional-preference stage images [st][C1 j < DP | C2 j < DP][TC_IMG_LD]
    const float* aT; const float* LT;         // [dp][B] (+ 64 floats of slack)
    float* out;             // gC_part [slot][units*d*K]
    const uint32_t* scal; float g_bound;
    int B, d, dp, K, NK, DP;
    int n_bil_tiles, n_bil_pairs;
    size_t split_stride;
    TcSched sch;            // units = stages of 64 examples, tiles = PAIRS of 128-row tiles (then the SP pair, if any)
    const int4* segs;       // sch's per-CTA table (TcSegIter)
};

__global__ void __launch_bounds__(TC_BWD_THREADS, 1) k_tc_dc2(TcDc2Args p) {
    pdl_enter();
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    TC_TRACE_INIT();
    const int DP = p.DP, nsrc = TC_M / DP;
    const uint32_t STB = 2u * 8u * (uint32_t)p.NK * 16u;                 // q^T operand stage
    const uint32_t IMG = (uint32_t)DP * TC_IMG_LD * 4u;                  // one stage image
    const uint32_t PAREA = 2u * (uint32_t)nsrc * 2u * 256u;              // [tile][source][a | L][64 examples]
    const uint32_t XST = 2u * IMG + PAREA;
    uint8_t* smB = smem_raw;
    uint8_t* smX = smem_raw + TC_DC2_BSTAGES * STB;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smX + TC_DC2_XSTAGES * XST);
    uint64_t* a_full = bars;            // [2] 16 generator-warp arrivals
    uint64_t* a_empty = bars + 2;       // [2] tcgen05.commit
    uint64_t* b_full = bars + 4;        // [3] bulk-copy tx
    uint64_t* b_empty = bars + 7;       // [3] tcgen05.commit
    uint64_t* x_full = bars + 10;       // [2] bulk-copy tx
    uint64_t* x_empty = bars + 12;      // [2] 16 generator-warp arrivals (their reads of the stage are done)
    uint64_t* acc_full = bars + 14;
    uint64_t* acc_empty = bars + 15;    // 16 drain-warp arrivals
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
    if (threadIdx.x == 0) { TC_TRACE(32); TC_TRACE_NS(46); }
#ifdef RAE_TRACE
    if (threadIdx.x == 0) {      // segment count, and whether the CTA's range holds stages of the SP pair
        TcSegIter si_(p.segs, p.sch.upt, blockIdx.x);
        TcSeg sg_;
        int n_ = 0, sp_ = 0;
        while (si_.next(sg_)) { ++n_; sp_ |= sg_.tile == p.n_bil_pairs; }
        TC_TRACE_VAL(80, n_);
        TC_TRACE_VAL(81, sp_);
    }
#endif
    if (threadIdx.x == 0) {
        for (int i = 0; i < 2; ++i) { mbar_init(&a_full[i], 16); mbar_init(&a_empty[i], 1); mbar_init(&x_full[i], 1); mbar_init(&x_empty[i], 16); }
        for (int i = 0; i < 3; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
        mbar_init(acc_full, 1);
        mbar_init(acc_empty, TC_BWD_WORKERS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == TC_BWD_WORKERS + 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) TC_TRACE(33);

    if (warp >= TC_BWD_WORKERS) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 32;" ::: "memory");
    }
    if (warp == TC_BWD_WORKERS + 1) {
        // ===== producer of the q^T operand ring =====
        if (lane == 0) {
            TcSegIter si(p.segs, p.sch.upt, blockIdx.x);
            TcSeg sg;
            int it = 0;
            while (si.next(sg)) {
                for (int st = sg.u0; st < sg.u1; ++st, ++it) {
                    const int s = it % TC_DC2_BSTAGES;
                    mbar_wait(&b_empty[s], ((it / TC_DC2_BSTAGES) & 1) ^ 1);
                    mbar_expect_tx(&b_full[s], STB);
                    bulk_g2s(smB + (size_t)s * STB, reinterpret_cast<const uint8_t*>(p.pop4) + (size_t)st * STB, STB, &b_full[s]);
                }
            }
        }
    } else if (warp == TC_BWD_WORKERS + 3) {
        // ===== producer of the image ring: R image, Y2 image, and the 64-example slices of a_i / L_i of the tiles' rows;
        // for the SP pair its image alone (the same 2 IMG bytes) =====
        if (lane == 0) {
            TcSegIter si(p.segs, p.sch.upt, blockIdx.x);
            TcSeg sg;
            int it = 0;
            while (si.next(sg)) {
                const bool sp = sg.tile == p.n_bil_pairs;
                const int i0 = sp ? p.dp : (2 * sg.tile * TC_M) / DP;   // first row i of tile A; tile B starts nsrc rows later
                for (int st = sg.u0; st < sg.u1; ++st, ++it) {
                    const int xs = it % TC_DC2_XSTAGES;
                    mbar_wait(&x_empty[xs], ((it / TC_DC2_XSTAGES) & 1) ^ 1);
                    uint32_t bytes = 2u * IMG;
                    for (int ts = 0; ts < 2 * nsrc; ++ts)
                        if (i0 + ts < p.dp) bytes += 512u;
                    mbar_expect_tx(&x_full[xs], bytes);
                    uint8_t* dst = smX + (size_t)xs * XST;
                    const uint8_t* srcX = sp ? reinterpret_cast<const uint8_t*>(p.SPimg) + (size_t)st * 2 * IMG
                                             : reinterpret_cast<const uint8_t*>(p.Rimg) + (size_t)st * IMG;
                    const uint8_t* srcY = sp ? srcX + IMG : reinterpret_cast<const uint8_t*>(p.Yimg) + (size_t)st * IMG;
                    bulk_g2s(dst, srcX, IMG, &x_full[xs]);
                    bulk_g2s(dst + IMG, srcY, IMG, &x_full[xs]);
                    for (int ts = 0; ts < 2 * nsrc; ++ts) {
                        const int i = i0 + ts;                  // (tile, source) -> row i
                        if (i < p.dp) {
                            bulk_g2s(dst + 2 * IMG + (size_t)ts * 512, p.aT + (size_t)i * p.B + (size_t)st * TC_SR, 256u, &x_full[xs]);
                            bulk_g2s(dst + 2 * IMG + (size_t)ts * 512 + 256, p.LT + (size_t)i * p.B + (size_t)st * TC_SR, 256u, &x_full[xs]);
                        }
                    }
                }
            }
        }
    } else if (warp == TC_BWD_WORKERS) {
        // ===== MMA issuer: one elected thread, fully unrolled (see k_tc_bilinear) =====
        if (elect_one()) {
            const uint32_t idesc = make_idesc_f16(TC_M, p.NK);
            TcSegIter si(p.segs, p.sch.upt, blockIdx.x);
            TcSeg sg;
            int it = 0, seg = 0;
            while (si.next(sg)) {
                const bool hasB = sg.tile == p.n_bil_pairs ? 2 * DP > TC_M : 2 * sg.tile + 1 < p.n_bil_tiles;
                const int nst = sg.u1 - sg.u0;
                if (seg > 0) {                                   // the previous segment's accumulators have been drained
                    mbar_wait(acc_empty, (seg - 1) & 1);
                    tc_fence_after();
                }
                bool ready = false;
                for (int lt = 0; lt < nst; ++lt) {
                    const int git = it + lt, s = git % TC_DC2_BSTAGES, as = git & 1;
                    if (!ready) {
                        mbar_wait(&a_full[as], (git >> 1) & 1);
                        mbar_wait(&b_full[s], (git / TC_DC2_BSTAGES) & 1);
                        tc_fence_after();
                    }
                    ready = false;
                    if (git == 8) TC_TRACE(38);
                    if (git == 24) TC_TRACE(43);
                    const uint32_t b_base = smem_u32(smB + (size_t)s * STB);
                    const uint64_t h0 = make_desc(b_base, (uint32_t)p.NK * 16u, 128u);
                    const uint64_t l0 = make_desc(b_base + 8u * (uint32_t)p.NK * 16u, (uint32_t)p.NK * 16u, 128u);
                    const uint32_t a0 = tmem_base + TC_DC2_ACOL + 128u * as;
#pragma unroll
                    for (int t = 0; t < 2; ++t) {
                        if (t == 1) {
                            if (lt + 1 < nst) {                  // the next stage's barriers, while this stage's MMAs are queued
                                const int g1 = git + 1;
                                mbar_wait(&a_full[g1 & 1], (g1 >> 1) & 1);
                                mbar_wait(&b_full[g1 % TC_DC2_BSTAGES], (g1 / TC_DC2_BSTAGES) & 1);
                                tc_fence_after();
                                ready = true;
                            }
                            if (!hasB) break;
                        }
                        const uint32_t acc = tmem_base + 128u * t, at = a0 + 64u * t;
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) {
                            if (TC_KNOCK(2)) continue;
                            const uint64_t hk = desc_advance(h0, (uint32_t)ks * 2u * (uint32_t)p.NK * 16u);
                            const uint64_t lk = desc_advance(l0, (uint32_t)ks * 2u * (uint32_t)p.NK * 16u);
                            tc_mma_f16_ts(acc, at + 8u * ks, hk, idesc, (lt > 0 || ks > 0) ? 1u : 0u);
                            tc_mma_f16_ts(acc, at + 8u * ks, lk, idesc, 1u);
                            tc_mma_f16_ts(acc, at + 32u + 8u * ks, hk, idesc, 1u);
                        }
                    }
                    tc_commit(&a_empty[as]);
                    tc_commit(&b_empty[s]);
                    if (lt == nst - 1) tc_commit(acc_full);
                    if (git == 8) TC_TRACE(39);
                    if (git == 24) TC_TRACE(44);
                }
                it += nst;
                ++seg;
            }
            TC_TRACE(35);
        }
        __syncwarp();
    } else if (warp < TC_BWD_WORKERS) {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 112;" ::: "memory");
        const int gw = warp, q4 = gw & 3, cg = gw >> 2;         // lane quarter; examples 16 cg .. 16 cg + 15 of a stage
        const int nl = q4 * 32 + lane;                          // row of the tile
        const int j = nl % DP, srcl = nl / DP;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q4 * 32) << 16);
        // operand scales (powers of two, undone in the epilogue): bilinear pairs from a bound of |a R + L Y2|, the SP pair
        // from the |max| of its image
        float sGb, invb, sGs, invs;
        {
            const float aL = __uint_as_float(p.scal[TS_AMAX_L]), aR = __uint_as_float(p.scal[TS_AMAX_R]);
            const float aA = __uint_as_float(p.scal[TS_AMAX_A]), aY = __uint_as_float(p.scal[TS_AMAX_Y2]);
            sGb = pow2_scale(__float_as_uint(fmaf(aA, aR, aL * aY)));
            invb = 1.f / (sGb * TC_QSCALE);
            sGs = pow2_scale(p.scal[TS_AMAX_SP]);
            invs = 1.f / (sGs * TC_QSCALE);
        }
        TcSegIter si(p.segs, p.sch.upt, blockIdx.x);
        TcSeg sg;
        int it = 0, seg = 0;
        while (si.next(sg)) {
            // SP pair: image row nl + 128 t is C1 row j (nl < DP) or C2 row j (DP <= nl + 128 t < 2 DP), i.e. rows d and d + 1 of
            // the slot block's [units][d][K] (the tensor path always has the bilinear units); tile A reads its C2 rows from
            // the second image half, where the bilinear pairs keep Y2
            const bool sp = sg.tile == p.n_bil_pairs;
            const bool hasB = sp ? 2 * DP > TC_M : 2 * sg.tile + 1 < p.n_bil_tiles;
            const int iA = sp ? p.d + srcl : (2 * sg.tile * TC_M) / DP + srcl, iB = iA + nsrc;
            const bool vA = (sp ? srcl < 2 : iA < p.d) && j < p.d, vB = hasB && (sp || iB < p.d) && j < p.d;
            const float sG = sp ? sGs : sGb, inv = sp ? invs : invb;
            const int xrow = (sp && srcl == 1) ? nl : j;
            const int nst = sg.u1 - sg.u0;
            for (int lt = 0; lt < nst; ++lt) {
                const int git = it + lt, xs = git & 1, as = git & 1;
                const uint8_t* stg = smX + (size_t)xs * XST;
                const float* Xr = reinterpret_cast<const float*>(stg) + (size_t)xrow * TC_IMG_LD + 16 * cg;
                const float* Yr = reinterpret_cast<const float*>(stg + IMG) + (size_t)j * TC_IMG_LD + 16 * cg;
                const float* Pa = reinterpret_cast<const float*>(stg + 2 * IMG) + (size_t)srcl * 128 + 16 * cg;     // tile A: [a | L]
                const float* Pb = Pa + (size_t)nsrc * 128;                                                             // tile B
                const bool tr = gw == 0 && lane == 0 && git == 8;
                if (tr) TC_TRACE(40);
                mbar_wait(&x_full[xs], (git >> 1) & 1);
                if (tr) TC_TRACE(41);
                const int b0 = (sg.u0 + lt) * TC_SR + 16 * cg;
                const bool full = b0 + 16 <= p.B;
                float x[16], y[16];
#pragma unroll
                for (int v4 = 0; v4 < 4; ++v4) {
                    const float4 xv = *reinterpret_cast<const float4*>(Xr + 4 * v4), yv = *reinterpret_cast<const float4*>(Yr + 4 * v4);
                    x[4 * v4] = xv.x * sG; x[4 * v4 + 1] = xv.y * sG; x[4 * v4 + 2] = xv.z * sG; x[4 * v4 + 3] = xv.w * sG;
                    y[4 * v4] = yv.x * sG; y[4 * v4 + 1] = yv.y * sG; y[4 * v4 + 2] = yv.z * sG; y[4 * v4 + 3] = yv.w * sG;
                }
                float gA[16], gB[16];
                if (sp) {                                        // the image rows are the operand (zero beyond B)
#pragma unroll
                    for (int e = 0; e < 16; ++e) {
                        gA[e] = (vA && !TC_KNOCK(4)) ? x[e] : 0.f;
                        gB[e] = (vB && !TC_KNOCK(4)) ? y[e] : 0.f;
                    }
                } else {
#pragma unroll
                    for (int v4 = 0; v4 < 4; ++v4) {
                        const float4 a1 = *reinterpret_cast<const float4*>(Pa + 4 * v4), l1 = *reinterpret_cast<const float4*>(Pa + 64 + 4 * v4);
                        const float4 a2 = *reinterpret_cast<const float4*>(Pb + 4 * v4), l2 = *reinterpret_cast<const float4*>(Pb + 64 + 4 * v4);
                        const float pa[4] = {a1.x, a1.y, a1.z, a1.w}, pl[4] = {l1.x, l1.y, l1.z, l1.w};
                        const float qa[4] = {a2.x, a2.y, a2.z, a2.w}, ql[4] = {l2.x, l2.y, l2.z, l2.w};
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int e = 4 * v4 + u;
                            const bool in = full || b0 + e < p.B;
                            gA[e] = (vA && in && !TC_KNOCK(4)) ? fmaf(pa[u], x[e], pl[u] * y[e]) : 0.f;
                            gB[e] = (vB && in && !TC_KNOCK(4)) ? fmaf(qa[u], x[e], ql[u] * y[e]) : 0.f;
                        }
                    }
                }
                // this warp's reads of the image stage are done (the values above depend on every one of them)
                __syncwarp();
                if (lane == 0) mbar_arrive(&x_empty[xs]);
                mbar_wait(&a_empty[as], ((git >> 1) & 1) ^ 1);
                tc_fence_after();
                {
                    uint32_t hi[8], lo[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) split_h2(gA[2 * u], gA[2 * u + 1], hi[u], lo[u]);
                    const uint32_t col = lane_base + TC_DC2_ACOL + 128u * as + 8u * cg;
                    tc_st8u(col, hi);
                    tc_st8u(col + 32u, lo);
                    if (hasB) {
#pragma unroll
                        for (int u = 0; u < 8; ++u) split_h2(gB[2 * u], gB[2 * u + 1], hi[u], lo[u]);
                        tc_st8u(col + 64u, hi);
                        tc_st8u(col + 96u, lo);
                    }
                }
                tc_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&a_full[as]);
                if (tr) TC_TRACE(42);
            }
            it += nst;
            {
                // ===== epilogue: both tiles' accumulator rows -> the segment's slot of the partial gradient, drained by all
                // 16 warps (warp (q4, cg): the 32-column chunks 32 cg, 32 cg + 128, ... of its lane quarter, as in k_tc_dq) =====
                mbar_wait(acc_full, seg & 1);
                tc_fence_after();
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    const int i = t == 0 ? iA : iB;
                    const bool valid = t == 0 ? vA : vB;
                    if (t == 1 && !hasB) break;
                    float* o = p.out + (size_t)sg.slot * p.split_stride + ((size_t)i * p.d + j) * p.K;
                    for (int c0 = 32 * cg; c0 < p.NK; c0 += 128) {
                        float tt[32];
                        tc_ld32(lane_base + 128u * t + (uint32_t)c0, tt);
#pragma unroll
                        for (int xx = 0; xx < 32; ++xx) tt[xx] *= inv;
                        if (valid) store_row32(o + c0, tt, p.K - c0, (p.K & 3) == 0);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(acc_empty);
            }
            ++seg;
        }
        if (gw == 0 && lane == 0) TC_TRACE(36);
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) { TC_TRACE(37); TC_TRACE_NS(47); }
    if (warp == TC_BWD_WORKERS + 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// per-example finishing of the backward: SP terms of dL/dR, dq (sum of the tile's slot partials) += entropy term, softmax
// backward.  One CTA of 32 warps per 32 examples: the transposed dq partials dqT[slot][k][b] are read coalesced (lane =
// example) into a shared tile, then one warp per example works on its row.
__global__ void __launch_bounds__(1024) k_tc_bwd_finish(float* __restrict__ ev, const float* __restrict__ sc, const float* __restrict__ q,
                                                       const float* __restrict__ logq, const float* __restrict__ dqT, float* __restrict__ dz,
                                                       float* __restrict__ dzsum_part, int B, int K, int NK, TcSched sch_dq, int d, int dp,
                                                       int hasSP, float ent_coef) {
    pdl_enter();
    extern __shared__ float fin_smem[];
    const int KS = K | 1;                  // odd row stride: conflict-free transposed writes
    float* sdq = fin_smem;                 // [32][KS]
    float* dzs = fin_smem + 32 * KS;       // [32][K]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b0 = blockIdx.x * 32;
    // Every loop below is "4 strided elements per lane" (K, d <= 128): the loads of all four are issued before the first use
    // (volatile asm, clamped addresses, results dropped by selects) - the kernel runs one 1024-thread CTA per SM, so a chain of
    // dependent round trips is paid in full (18.7 us for 21 MB before, ncu long-scoreboard).
    {
        const int ns = tcs_nslots(sch_dq, b0 >> 7);
        const int b = b0 + lane, bb = min(b, B - 1);
        float t[4][4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int sl = 0; sl < 4; ++sl)
                t[u][sl] = ldg_stream(dqT + ((size_t)min(sl, ns - 1) * NK + min(warp + 32 * u, K - 1)) * B + bb);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int k = warp + 32 * u;
            if (k >= K) continue;
            float v = 0.f;
#pragma unroll
            for (int sl = 0; sl < 4; ++sl) v += sl < ns ? t[u][sl] : 0.f;
            for (int sl = 4; sl < ns; ++sl) v += dqT[((size_t)sl * NK + k) * B + bb];
            sdq[lane * KS + k] = b < B ? v : 0.f;
        }
    }
    __syncthreads();
    {
        const int e = warp;
        const int b = b0 + e;
        if (b < B) {
            float* evb = ev + (size_t)b * E_NV * dp;
            float lq[4], qq[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int kk = min(lane + 32 * u, K - 1);
                lq[u] = ldg_stream(logq + (size_t)b * K + kk);
                qq[u] = ldg_stream(q + (size_t)b * K + kk);
            }
            if (hasSP) {
                // d cost / d L = M c + SP term, d cost / d R = M^T a + SP term: k_tc_combine left M c and M^T a in E_GA1 / E_GA2
                const float gp = sc[(size_t)b * SC_N + SC_GP], g1 = sc[(size_t)b * SC_N + SC_G1], g2 = sc[(size_t)b * SC_N + SC_G2];
                float x1[4], x2[4], y1[4], y2[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int jj = min(lane + 32 * u, d - 1);
                    x1[u] = ldg_ordered(evb + E_GA1 * dp + jj); y1[u] = ldg_ordered(evb + E_C1 * dp + jj);
                    x2[u] = ldg_ordered(evb + E_GA2 * dp + jj); y2[u] = ldg_ordered(evb + E_C2 * dp + jj);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int j = lane + 32 * u;
                    if (j < d) {
                        evb[E_GA1 * dp + j] = fmaf(gp + g2, y1[u], x1[u]);
                        evb[E_GA2 * dp + j] = fmaf(gp + g1, y2[u], x2[u]);
                    }
                }
            }
            float dot = 0.f, vv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int k = lane + 32 * u;
                vv[u] = 0.f;
                if (k < K) {
                    vv[u] = fmaf(ent_coef, lq[u] + 1.f, sdq[e * KS + k]);
                    dot = fmaf(qq[u], vv[u], dot);
                }
            }
            dot = warp_sum(dot);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int k = lane + 32 * u;
                if (k < K) {
                    const float v = qq[u] * (vv[u] - dot);
                    dzs[e * K + k] = v;
                    dz[(size_t)b * K + k] = v;
                }
            }
        } else {
            for (int k = lane; k < K; k += 32) dzs[e * K + k] = 0.f;
        }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
        double s = 0.0;            // cancelling sum: see k_dense_finalize
#pragma unroll 8
        for (int w = 0; w < 32; ++w) s += (double)dzs[w * K + k];
        dzsum_part[(size_t)blockIdx.x * K + k] = (float)s;
    }
}

int tc_dp(int d) { return d <= 32 ? 32 : d <= 64 ? 64 : 128; }

#ifdef RAE_TRACE
}  // namespace
extern "C" int rae_debug_set_trace(unsigned long long* dev_buf) {
    return (int)cudaMemcpyToSymbol(g_tc_trace, &dev_buf, sizeof(dev_buf));
}
extern "C" int rae_debug_set_knock(int bits) { return (int)cudaMemcpyToSymbol(g_tc_knock, &bits, sizeof(bits)); }
namespace {
#endif

// cost weights of a schedule (TcSched): tail units, body / tail unit weight, tile-start weight
struct TcCost { int ntail = 0, wb = 1, wt = 1, h = 0; };

int sched_max_share(TcSched s) {
    int m = 0;
    for (int x = 0; x < s.G; ++x) m = std::max(m, tcs_start(s, x + 1) - tcs_start(s, x));
    return m;
}
bool sched_nonempty(TcSched s) {
    for (int x = 0; x < s.G; ++x)
        if (tcs_start(s, x + 1) == tcs_start(s, x)) return false;
    return true;
}

// balanced schedule of T = ntile * upt units: one CTA per SM, or whole waves of CTAs when a CTA's share would exceed
// `max_share` units (accuracy bound on the MMA chain of one accumulator / capacity of a staging area).  A CTA's share
// of the virtual time must hold a unit: where a tile's first unit (h + wb) or a tail unit (wt) is longer than the share
// (a few units per CTA, as at d = 30), both are capped at it.
TcSched make_sched(int ntile, int upt, int num_sms, int max_share, TcCost c = TcCost{}) {
    TcSched s{0, upt, ntile, std::min(c.ntail, upt), c.wb, c.wt, c.h};
    const long long T = (long long)ntile * upt;
    long long G = std::min<long long>(T, num_sms);
    if (max_share > 0 && (T + G - 1) / G > max_share) {
        const long long waves = (T + (long long)num_sms * max_share - 1) / ((long long)num_sms * max_share);
        G = std::min<long long>(T, waves * num_sms);
    }
    s.G = (int)std::max<long long>(G, 1);
    // terminates: each step lowers h or wt or adds a wave; with uniform weights every CTA is non-empty (G <= T) and
    // the wave count above bounds the share
    for (;;) {
        if (!sched_nonempty(s)) {
            const int share = (int)((long long)tcs_tile_len(s) * s.ntile / s.G);
            int wt = std::max(s.wb, std::min(s.wt, share));
            int h = std::max(0, std::min(s.h, share - s.wb));
            if (wt == s.wt && h == s.h) { wt = std::max(s.wb, wt - 1); h = std::max(0, h - 1); }   // rounding: step down
            s.wt = wt; s.h = h;
        } else if (max_share > 0 && s.G < T && sched_max_share(s) > max_share) {
            s.G = (int)std::min<long long>(T, (long long)s.G + num_sms);
        } else {
            return s;
        }
    }
}
int sched_max_slots(TcSched s) {
    int m = 1;
    for (int t = 0; t < s.ntile; ++t) m = std::max(m, tcs_nslots(s, t));
    return m;
}

}  // namespace

// L = A[a1], R = A[a2] (A[a1] with the model-C quirk) -> ev
namespace {
__global__ void __launch_bounds__(256) k_tc_gather_lr(const float* __restrict__ A, const int32_t* __restrict__ a1,
                                                      const int32_t* __restrict__ a2, int B, int d, int dp, int quirk,
                                                      float* __restrict__ ev) {
    const int lane = threadIdx.x & 31;
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= B) return;
    const int r1 = a1[b], r2 = quirk ? r1 : a2[b];
    float* o = ev + (size_t)b * E_NV * dp;
    for (int j = lane; j < d; j += 32) {
        o[E_L * dp + j] = ld_nc(A + (size_t)r1 * d + j);
        o[E_R * dp + j] = ld_nc(A + (size_t)r2 * d + j);
    }
}
}  // namespace

// shapes the tensor path handles: 16 < d <= 128 (padded to 32/64/128 columns per row) and K <= 104 (P operand resident
// in TMEM next to the accumulators)
int tc_supported(const rae_engine* h) {
    if (!h->hasM) return 0;
    if (h->d <= 16 || h->d > 128) return 0;
    if (h->K > 104) return 0;
    if (h->B > (1 << 24)) return 0;     // the schedules' virtual time (TcSched) is an int: ntile * L < 2^17 * 2^11
    return 1;
}

namespace {
// Cost weights of the forward, recompute and dq schedules, in eighths of a body unit, fitted to the in-kernel trace at
// K = 100 with selectional preferences on one B200 (profiles/r04_weighted_schedule.md, profiles/fit_sched_cost.py: CTA
// life, less the body units at the pass's steady cadence, by least squares over the tail units and the extra segments of
// each CTA).  DP = 128: the trace of the weighted schedule at T (profiles/r04_cta_life_weighted_T.csv), where CTAs of
// 15-32 units and one or two segments pin h and wt down better than the uniform split did.  DP = 32: the trace of the
// uniform split at cfg2 (profiles/r04_cta_life_before_cfg2.csv); make_sched caps these there anyway (two units per CTA).
// DP = 64: the mean of the two.  Other K and shapes without selectional preferences take the same weights unmeasured.
TcCost tc_cost(int DP, int pass, int ntail) {
    const int di = DP == 128 ? 0 : DP == 64 ? 1 : 2;
    static const int H[3][3] = {{64, 48, 33}, {52, 40, 29}, {76, 77, 78}};       // [pass][DP 128, 64, 32] tile start
    static const int WT[3][3] = {{30, 57, 84}, {8, 8, 8}, {41, 32, 22}};         // [pass][DP 128, 64, 32] tail unit
    TcCost c;
    c.ntail = ntail; c.wb = 8; c.wt = WT[pass][di]; c.h = H[pass][di];
    return c;
}

// geometry of the contraction operands and the forward (pass 0), recompute (1) and dq (2) schedules of a shape: host
// arithmetic only
void tc_plan(TcState& t, int B, int K, int d, bool hasSP, int num_sms) {
    const int DP = tc_dp(d);
    t.DP = DP;
    t.KH = (K + 15) & ~15;
    // bilinear rows i padded so that the operand rows fill whole 128-row stages (DP = 64: pairs of rows, DP = 32: fours)
    const int rps = 128 / DP;
    const int di = (d + rps - 1) / rps * rps;
    t.n_bil_rows = di * DP;
    t.n_bil_half = t.n_bil_rows / TC_H;
    t.n_sp_half = hasSP ? (2 * DP) / TC_H : 0;
    t.n_rows_total = (t.n_bil_rows + (hasSP ? 2 * DP : 0) + TC_M - 1) / TC_M * TC_M;
    t.n_chunks_fwd = (t.n_bil_half + t.n_sp_half + 1) / 2;
    t.n_chunks_rec = t.n_bil_half / 2;
    t.ntile = (B + TC_M - 1) / TC_M;
    // the chunks / stages that hold C1 / C2 rows close every tile of the forward and dq passes
    const int n_st = t.n_rows_total / TC_M;
    t.sch_fwd = make_sched(t.ntile, t.n_chunks_fwd, num_sms, 0, tc_cost(DP, 0, t.n_chunks_fwd - t.n_chunks_rec));
    t.sch_rec = make_sched(t.ntile, t.n_chunks_rec, num_sms, 0, tc_cost(DP, 1, 0));
    t.slots_vw = std::max(sched_max_slots(t.sch_fwd), sched_max_slots(t.sch_rec));
    // backward operands: NK = relations padded to a multiple of 16.  dq reduces over stages of 128 operand rows (FP16
    // pairs), dC over stages of 64 examples (TF32 pairs): both 2 * 2 * 8 * NK * 16 bytes per stage
    t.NK = (K + 15) & ~15;
    // accuracy bound of the dq reduction: the measured-safe chain is 1560 MMAs into one accumulator (4.5e-6 of
    // ||dW||_inf at the target shape); a segment never exceeds TC_DQ_MAX_STAGES stages = 1536 MMAs
    t.sch_dq = make_sched(t.ntile, n_st, num_sms, TC_DQ_MAX_STAGES, tc_cost(DP, 2, n_st - t.n_bil_rows / TC_M));
    t.slots_dq = sched_max_slots(t.sch_dq);
}

// the dC plan of a shape (after tc_plan; host arithmetic only).  The two-tile FP16 kernel takes every 128-row tile of the
// operand rows - the bilinear tiles in pairs, then the C1 / C2 tiles as one more pair - when B % 4 == 0 and its stages fit
// in shared memory; otherwise the one-tile kernel takes them all.  Uniform weights: a stage of the SP pair issues as many
// MMAs as a bilinear pair's, except at DP <= 64 (half as many, one pair among 4 - 65).  -> tile_slots: the partial slots
// of every tile (k_dense_finalize).  Returns 0, 1 when the backward operand stages do not fit in shared memory, 2 when the
// one-tile kernel's staging area does not.
int tc_plan_dc(TcState& t, int B, bool hasSP, int num_sms, int max_smem_optin, std::vector<int32_t>& tile_slots) {
    const int DP = t.DP;
    t.smem_dq = (size_t)TC_BSTAGES * (2 * 2 * 8 * t.NK * 16) + 256;
    if (t.smem_dq > (size_t)max_smem_optin) return 1;
    t.n_ntiles = t.n_rows_total / TC_M;
    t.n_bst = (B + TC_SR - 1) / TC_SR;
    // one-tile kernel: accuracy bound (see TC_DC_MAX_STAGES) and the capacity of the per-example scalar staging area
    t.dc_nacc = 2;
    const size_t per_stage = (size_t)(TC_M / DP) * 2 * TC_SR * sizeof(float);
    const int cap = (int)(((size_t)max_smem_optin - t.smem_dq) / per_stage);
    if (cap < 1) return 2;
    // the two-tile kernel needs 16-byte aligned slices of the transposed copies
    const int n_bil_tiles = t.n_bil_rows / TC_M, n_bil_pairs = (n_bil_tiles + 1) / 2;
    t.dc2 = (B % 4 == 0) && n_bil_tiles > 0;
    t.smem_dc2 = (size_t)TC_DC2_BSTAGES * (2 * 8 * t.NK * 16) + (size_t)TC_DC2_XSTAGES * (2 * (size_t)DP * TC_IMG_LD * 4 + 2 * (TC_M / DP) * 2 * 256) + 256;
    if (t.smem_dc2 > (size_t)max_smem_optin) t.dc2 = false;
    t.dc_tiles = t.dc2 ? 0 : t.n_ntiles;
    t.dc_share = 0;
    tile_slots.assign((size_t)t.n_ntiles, 1);
    if (t.dc2) {
        t.sch_dc2 = make_sched(n_bil_pairs + (hasSP ? 1 : 0), t.n_bst, num_sms, TC_DC2_MAX_STAGES);
        t.slots_dc = sched_max_slots(t.sch_dc2);
        for (int nt = 0; nt < t.n_ntiles; ++nt) tile_slots[nt] = tcs_nslots(t.sch_dc2, nt < n_bil_tiles ? nt / 2 : n_bil_pairs);
    } else {
        t.sch_dc = make_sched(t.dc_tiles, t.n_bst, num_sms, std::min(t.dc_nacc * TC_DC_MAX_STAGES, cap));
        t.dc_share = sched_max_share(t.sch_dc);
        t.slots_dc = sched_max_slots(t.sch_dc);
        for (int nt = 0; nt < t.n_ntiles; ++nt) tile_slots[nt] = tcs_nslots(t.sch_dc, nt);
    }
    t.smem_dc = t.smem_dq + (size_t)t.dc_share * per_stage;
    return 0;
}
}  // namespace

// The schedule tc_plan builds for one pass (0 forward, 1 recompute, 2 dq), for the tests: its seven fields
// (G, upt, ntile, ntail, wb, wt, h) -> sched[7], the first unit of every CTA and the end -> starts[G + 1] (when
// max_starts >= G + 1) and the partial slots of every tile -> nslots[ntile] (when max_tiles >= ntile).  Returns G, or -1
// for a shape the tensor path does not take.  Host only: needs no device.
extern "C" int rae_debug_tc_schedule(int B, int K, int d, int hasSP, int num_sms, int pass, int32_t* sched, int64_t* starts,
                                     int max_starts, int32_t* nslots, int max_tiles) {
    if (B < 1 || K < 1 || K > 104 || d <= 16 || d > 128 || num_sms < 1 || pass < 0 || pass > 2) return -1;
    TcState t;
    tc_plan(t, B, K, d, hasSP != 0, num_sms);
    const TcSched s = pass == 0 ? t.sch_fwd : pass == 1 ? t.sch_rec : t.sch_dq;
    const int f[7] = {s.G, s.upt, s.ntile, s.ntail, s.wb, s.wt, s.h};
    if (sched != nullptr) std::copy(f, f + 7, sched);
    if (starts != nullptr && max_starts >= s.G + 1)
        for (int x = 0; x <= s.G; ++x) starts[x] = tcs_start(s, x);
    if (nslots != nullptr && max_tiles >= s.ntile)
        for (int tl = 0; tl < s.ntile; ++tl) nslots[tl] = tcs_nslots(s, tl);
    return s.G;
}

// make_sched itself, for the tests: the schedule of ntile tiles of upt units with the given weights (wb = 0: the default
// uniform weights) -> sched[7] as above and starts[G + 1] (when max_starts >= G + 1).  Returns G.  Host only.
extern "C" int rae_debug_tc_make_sched(int ntile, int upt, int num_sms, int max_share, int ntail, int wb, int wt, int h,
                                       int32_t* sched, int64_t* starts, int max_starts) {
    if (ntile < 1 || upt < 1 || num_sms < 1 || max_share < 0 || wb < 0 || (wb > 0 && (wt < wb || h < 0 || ntail < 0))) return -1;
    TcCost c;
    if (wb > 0) { c.ntail = ntail; c.wb = wb; c.wt = wt; c.h = h; }
    const TcSched s = make_sched(ntile, upt, num_sms, max_share, c);
    const int f[7] = {s.G, s.upt, s.ntile, s.ntail, s.wb, s.wt, s.h};
    if (sched != nullptr) std::copy(f, f + 7, sched);
    if (starts != nullptr && max_starts >= s.G + 1)
        for (int x = 0; x <= s.G; ++x) starts[x] = tcs_start(s, x);
    return s.G;
}

// The dC plan tc_init builds, for the tests: info[4] = {two-tile kernel runs, bilinear 128-row tiles, all row tiles,
// slots_dc}, the fields of the launched kernel's schedule -> sched[7] (as above), the first unit of every CTA and the end
// -> starts[G + 1] (when max_starts >= G + 1) and the partial slots of every row tile -> tile_slots[n_ntiles] (when
// max_tiles >= n_ntiles).  Returns G, or -1 for a shape the tensor path does not take or whose dC stages do not fit in
// max_smem_optin bytes.  Host only: needs no device.
extern "C" int rae_debug_tc_dc_plan(int B, int K, int d, int hasSP, int num_sms, int max_smem_optin, int32_t* info, int32_t* sched,
                                    int64_t* starts, int max_starts, int32_t* tile_slots, int max_tiles) {
    if (B < 1 || K < 1 || K > 104 || d <= 16 || d > 128 || num_sms < 1) return -1;
    TcState t;
    std::vector<int32_t> ts;
    tc_plan(t, B, K, d, hasSP != 0, num_sms);
    if (tc_plan_dc(t, B, hasSP != 0, num_sms, max_smem_optin, ts) != 0) return -1;
    const TcSched s = t.dc2 ? t.sch_dc2 : t.sch_dc;
    const int in[4] = {t.dc2 ? 1 : 0, t.n_bil_rows / TC_M, t.n_ntiles, t.slots_dc};
    if (info != nullptr) std::copy(in, in + 4, info);
    const int f[7] = {s.G, s.upt, s.ntile, s.ntail, s.wb, s.wt, s.h};
    if (sched != nullptr) std::copy(f, f + 7, sched);
    if (starts != nullptr && max_starts >= s.G + 1)
        for (int x = 0; x <= s.G; ++x) starts[x] = tcs_start(s, x);
    if (tile_slots != nullptr && max_tiles >= t.n_ntiles) std::copy(ts.begin(), ts.end(), tile_slots);
    return s.G;
}

int tc_init(rae_engine* h) {
    TcState& t = h->tc;
    tc_plan(t, h->B, h->K, h->d, h->hasSP, h->num_sms);
    const int DP = t.DP;
    // forward: as many 128-row operand stages as fit (4 at K = 100: 57 KB each)
    const size_t b_bytes = (size_t)2 * (t.KH / 8) * TC_N * 16;
    t.fwd_stages = (int)std::min<size_t>(4, ((size_t)h->max_smem_optin - 256) / b_bytes);
    if (t.fwd_stages < 2) return fail(h, RAE_EINVAL, "tensor path: K=%d needs %zu bytes per operand stage, two do not fit", h->K, b_bytes);
    t.smem = (size_t)t.fwd_stages * b_bytes + 256;
    const int n_st = t.n_rows_total / TC_M;
    const size_t st_bytes = (size_t)2 * 2 * 8 * t.NK * 16;
    std::vector<int32_t> ts;
    const int rc = tc_plan_dc(t, h->B, h->hasSP, h->num_sms, h->max_smem_optin, ts);
    if (rc == 1) return fail(h, RAE_EINVAL, "tensor path: backward operand stages do not fit in shared memory");
    if (rc == 2) return fail(h, RAE_EINVAL, "tensor path: no shared memory left for the dC staging area");
    const bool sp_img = t.dc2 && h->hasSP;
    const size_t sp_img_bytes = (size_t)t.n_bst * 2 * DP * TC_IMG_LD * sizeof(float);
    cudaError_t e;
    const size_t vec = (size_t)h->dp * h->B * sizeof(float);
    if ((e = cudaMalloc((void**)&t.bop, (size_t)t.n_chunks_fwd * b_bytes)) != cudaSuccess ||
        (e = cudaMalloc((void**)&t.pimg, (size_t)t.ntile * b_bytes)) != cudaSuccess ||
        (e = cudaMalloc((void**)&t.vT, 2 * vec)) != cudaSuccess ||
        (e = cudaMalloc((void**)&t.wT, 2 * t.slots_vw * vec)) != cudaSuccess ||
        (e = cudaMalloc((void**)&t.spT, 2 * vec)) != cudaSuccess ||
        (e = cudaMalloc((void**)&t.bop2, (size_t)n_st * st_bytes)) != cudaSuccess ||
        (e = cudaMalloc((void**)&t.dqT, (size_t)t.slots_dq * h->B * t.NK * sizeof(float))) != cudaSuccess ||
        (e = cudaMalloc((void**)&t.pop3, (size_t)t.n_bst * st_bytes)) != cudaSuccess ||
        (e = cudaMalloc((void**)&t.aT, vec + 256)) != cudaSuccess || (e = cudaMalloc((void**)&t.LT, vec + 256)) != cudaSuccess ||
        (e = cudaMemset(t.aT, 0, vec + 256)) != cudaSuccess || (e = cudaMemset(t.LT, 0, vec + 256)) != cudaSuccess ||
        (e = cudaMalloc((void**)&t.pop4, (size_t)t.n_bst * 2 * 8 * t.NK * 16)) != cudaSuccess ||
        (e = cudaMalloc((void**)&t.Rimg, (size_t)t.n_bst * DP * TC_IMG_LD * sizeof(float))) != cudaSuccess ||
        (e = cudaMalloc((void**)&t.Yimg, (size_t)t.n_bst * DP * TC_IMG_LD * sizeof(float))) != cudaSuccess ||
        (e = cudaMemset(t.Rimg, 0, (size_t)t.n_bst * DP * TC_IMG_LD * sizeof(float))) != cudaSuccess ||
        (e = cudaMemset(t.Yimg, 0, (size_t)t.n_bst * DP * TC_IMG_LD * sizeof(float))) != cudaSuccess ||
        (sp_img && (e = cudaMalloc((void**)&t.SPimg, sp_img_bytes)) != cudaSuccess) ||
        (sp_img && (e = cudaMemset(t.SPimg, 0, sp_img_bytes)) != cudaSuccess) ||
        (e = cudaMalloc((void**)&t.RT, vec)) != cudaSuccess || (e = cudaMalloc((void**)&t.cT, vec)) != cudaSuccess ||
        (e = cudaMalloc((void**)&t.Y2T, vec)) != cudaSuccess ||
        (e = cudaMalloc((void**)&t.scal, TS_N * sizeof(uint32_t))) != cudaSuccess ||
        (e = cudaMemset(t.scal, 0, TS_N * sizeof(uint32_t))) != cudaSuccess)
        return fail(h, RAE_ENOMEM, "tensor-path workspace: %s", cudaGetErrorString(e));
    if ((e = cudaMalloc((void**)&t.tile_slots, ts.size() * sizeof(int32_t))) != cudaSuccess ||
        (e = cudaMemcpy(t.tile_slots, ts.data(), ts.size() * sizeof(int32_t), cudaMemcpyHostToDevice)) != cudaSuccess)
        return fail(h, RAE_ENOMEM, "tensor-path workspace: %s", cudaGetErrorString(e));
    {
        // per-CTA tables of the five schedules (TcSegIter): first unit, end unit, slot of the first segment
        std::vector<int4> tab;
        auto add = [&](const TcSched& sc) {
            const int off = (int)tab.size();
            for (int x = 0; x < sc.G; ++x) {
                const int u0 = tcs_start(sc, x);
                tab.push_back(make_int4(u0, tcs_start(sc, x + 1), x - tcs_first(sc, u0 / sc.upt), 0));
            }
            return off;
        };
        t.segs_fwd = add(t.sch_fwd); t.segs_rec = add(t.sch_rec); t.segs_dq = add(t.sch_dq);
        if (t.dc2) t.segs_dc2 = add(t.sch_dc2);
        if (t.dc_tiles > 0) t.segs_dc = add(t.sch_dc);
        if ((e = cudaMalloc((void**)&t.segs, tab.size() * sizeof(int4))) != cudaSuccess ||
            (e = cudaMemcpy(t.segs, tab.data(), tab.size() * sizeof(int4), cudaMemcpyHostToDevice)) != cudaSuccess)
            return fail(h, RAE_ENOMEM, "tensor-path workspace: %s", cudaGetErrorString(e));
    }
#define RAE_TC_ATTR(KERN, BYTES)                                                                                     \
    if ((e = cudaFuncSetAttribute(KERN, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(BYTES))) != cudaSuccess) \
        return fail(h, RAE_ECUDA, "cudaFuncSetAttribute(" #KERN "): %s", cudaGetErrorString(e));
    RAE_TC_ATTR(k_tc_bilinear<32>, t.smem) RAE_TC_ATTR(k_tc_bilinear<64>, t.smem) RAE_TC_ATTR(k_tc_bilinear<128>, t.smem)
    RAE_TC_ATTR(k_tc_dq<32>, t.smem_dq) RAE_TC_ATTR(k_tc_dq<64>, t.smem_dq) RAE_TC_ATTR(k_tc_dq<128>, t.smem_dq)
    RAE_TC_ATTR(k_tc_dc, t.smem_dc)
    if (t.dc2) { RAE_TC_ATTR(k_tc_dc2, t.smem_dc2) }
#undef RAE_TC_ATTR
    t.ready = true;
    return RAE_OK;
}

void tc_free(rae_engine* h) {
    TcState& t = h->tc;
    cudaFree(t.bop); cudaFree(t.pimg); cudaFree(t.vT); cudaFree(t.wT); cudaFree(t.spT); cudaFree(t.bop2); cudaFree(t.dqT); cudaFree(t.pop3); cudaFree(t.scal); cudaFree(t.pop4); cudaFree(t.Rimg); cudaFree(t.Yimg); cudaFree(t.SPimg); cudaFree(t.tile_slots); cudaFree(t.segs);
    cudaFree(t.aT); cudaFree(t.LT); cudaFree(t.RT); cudaFree(t.cT); cudaFree(t.Y2T);
    t = TcState{};
}

// pre-split / pre-arrange the dense operands (call whenever C, C1, C2 changed, i.e. once per step): |max| -> scale -> FP16 pairs
int tc_prepare_c(rae_engine* h, cudaStream_t st) {
    TcState& t = h->tc;
    RAE_CUDA(h, cudaMemsetAsync(t.scal + TS_AMAX_C, 0, sizeof(uint32_t), st));
    const size_t dd = h->hasM ? (size_t)h->d * h->d * h->K : 0, dk = h->hasSP ? (size_t)h->d * h->K : 0;
    launch_pdl(k_tc_absmax, dim3(h->num_sms * 8), dim3(256), 0, st, h->P[RAE_P_C], dd, h->P[RAE_P_C1], dk, h->P[RAE_P_C2], dk, t.scal + TS_AMAX_C);
    const size_t total = (size_t)t.n_chunks_fwd * TC_N * (t.KH / 8);
    const int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)h->num_sms * 8);
    launch_pdl(k_tc_prep_c, dim3(blocks, 2), dim3(256), 0, st, h->P[RAE_P_C], h->P[RAE_P_C1], h->P[RAE_P_C2], h->d, h->K, t.KH / 8, t.DP, t.n_bil_rows,
                                                 t.n_chunks_fwd * TC_N, reinterpret_cast<uint4*>(t.bop), t.NK, t.n_rows_total,
                                                 reinterpret_cast<uint4*>(t.bop2), t.scal);
    h->launches += 2;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

namespace {
// img_slot >= 0: that slot is ALSO written as the stack of stage images the two-tile dC kernel fetches; sp_img: so are the
// selectional-preference rows a + G2 L, c + G1 R of its SP pair (after scoring: a, c and G1, G2 are final)
int tc_transpose_slots(rae_engine* h, int n, const int* slots, float* const* dst, const int* amax_word, int img_slot,
                       float* img_dst, bool sp_img, cudaStream_t st) {
    TcState& t = h->tc;
    TrJobs jobs{};
    jobs.B = h->B;
    int nj = 0, maxc = 0;
    for (int i = 0; i < n; ++i) {
        jobs.j[nj++] = TrJob{h->ev + (size_t)slots[i] * h->dp, (size_t)E_NV * h->dp, h->d, h->dp, dst[i], t.scal + amax_word[i], 0, nullptr, nullptr};
        maxc = std::max(maxc, h->dp);
    }
    if (img_slot >= 0 && t.dc2) {
        jobs.j[nj++] = TrJob{h->ev + (size_t)img_slot * h->dp, (size_t)E_NV * h->dp, h->d, t.DP, img_dst, nullptr, t.DP, nullptr, nullptr};
        maxc = std::max(maxc, t.DP);
    }
    if (sp_img && t.dc2 && h->hasSP) {
        const size_t es = (size_t)E_NV * h->dp;
        jobs.j[nj++] = TrJob{h->ev + (size_t)E_A * h->dp, es, h->d, t.DP, t.SPimg, t.scal + TS_AMAX_SP, 2 * t.DP, h->ev + (size_t)E_L * h->dp, h->sc + SC_G2};
        jobs.j[nj++] = TrJob{h->ev + (size_t)E_CV * h->dp, es, h->d, t.DP, t.SPimg + (size_t)t.DP * TC_IMG_LD, t.scal + TS_AMAX_SP, 2 * t.DP,
                             h->ev + (size_t)E_R * h->dp, h->sc + SC_G1};
        maxc = std::max(maxc, t.DP);
    }
    launch_pdl(k_tc_transpose, dim3((h->B + 31) / 32, (maxc + 31) / 32, nj), dim3(256), 0, st, jobs);
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}
}  // namespace

// q-dependent operands of the dC and forward / recompute contractions (after the encoder) + L / R gather, then the
// transposed views LT, RT
int tc_prepare_p(rae_engine* h, const int32_t* a1, const int32_t* a2, cudaStream_t st) {
    TcState& t = h->tc;
    const int nbc = 2 * t.n_bst;
    const size_t total3 = (size_t)nbc * 8 * t.NK;
    const int blocks3 = (int)std::min<size_t>((total3 + 255) / 256, (size_t)h->num_sms * 8);
    launch_pdl(k_tc_prep_qt, dim3(blocks3, t.dc2 ? 4 : 3), dim3(256), 0, st, h->q, h->B, h->K, t.NK, nbc, t.pop3, h->P[RAE_P_A], a1, a2, h->d, h->dp,
                                                              h->quirk ? 1 : 0, h->ev, t.scal, reinterpret_cast<uint4*>(t.pop4), t.pimg);
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    const int slots[2] = {E_L, E_R};
    float* const dst[2] = {t.LT, t.RT};
    const int words[2] = {TS_AMAX_L, TS_AMAX_R};
    return tc_transpose_slots(h, 2, slots, dst, words, E_R, t.Rimg, false, st);
}

// the q-dependent operand alone (only the dC contraction at the end of the step needs it: prepared off the critical path)
int tc_prepare_qt(rae_engine* h, cudaStream_t st) {
    TcState& t = h->tc;
    const int nbc = 2 * t.n_bst;
    const size_t total3 = (size_t)nbc * 8 * t.NK;
    const int blocks3 = (int)std::min<size_t>((total3 + 255) / 256, (size_t)h->num_sms * 8);
    launch_pdl(k_tc_prep_qt, dim3(blocks3, 1), dim3(256), 0, st, h->q, h->B, h->K, t.NK, nbc, t.pop3, h->P[RAE_P_A], nullptr, nullptr, h->d, h->dp,
                                                   h->quirk ? 1 : 0, h->ev, t.scal, nullptr, nullptr);
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

// one contraction pass over the transposed views (LT_in, RT_in): v = M R [+ SP rows to E_C1/E_C2 when with_sp], w = M^T L,
// combined into ev[b][slotV | slotW]
int tc_contract(rae_engine* h, const float* LT_in, const float* RT_in, int slotV, int slotW, bool with_sp, cudaStream_t st) {
    TcState& t = h->tc;
    TcArgs p{};
    p.bop = t.bop; p.pimg = reinterpret_cast<const uint8_t*>(t.pimg); p.LT = LT_in; p.RT = RT_in; p.spT = t.spT; p.vT = t.vT; p.wT = t.wT; p.scal = t.scal;
    p.B = h->B; p.K = h->K; p.d = h->d; p.dp = h->dp; p.KH = t.KH;
    p.n_bil_half = t.n_bil_half; p.n_sp_half = with_sp ? t.n_sp_half : 0;
    p.nbs = t.fwd_stages;
    p.sch = with_sp ? t.sch_fwd : t.sch_rec;
    p.segs = t.segs + (with_sp ? t.segs_fwd : t.segs_rec);
    if (t.DP == 32) launch_pdl(k_tc_bilinear<32>, dim3(p.sch.G), dim3(TC_FWD_THREADS), t.smem, st, p);
    else if (t.DP == 64) launch_pdl(k_tc_bilinear<64>, dim3(p.sch.G), dim3(TC_FWD_THREADS), t.smem, st, p);
    else launch_pdl(k_tc_bilinear<128>, dim3(p.sch.G), dim3(TC_FWD_THREADS), t.smem, st, p);
    RAE_CUDA(h, cudaGetLastError());
    launch_pdl(k_tc_combine, dim3((h->B + 31) / 32, (h->d + 31) / 32), dim3(256), 0, st, t.vT, t.wT, (with_sp && h->hasSP) ? t.spT : nullptr, h->ev, h->B, h->d,
                                                                          h->dp, t.DP, p.sch, slotV, slotW, with_sp ? t.scal : nullptr);
    h->launches += 2;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

int tc_forward(rae_engine* h, cudaStream_t st) { return tc_contract(h, h->tc.LT, h->tc.RT, E_V1, E_V2, true, st); }

// backward on the tensor path, three parts (separately timed phases): (1) the transposed views of a, c, Y2 and M c, M^T a
// through the forward kernel with L := a, R := c; (2) dq contraction; (3) per-example finish: dL, dR, entropy term,
// softmax backward -> dz
int tc_backward_recompute(rae_engine* h, cudaStream_t st) {
    TcState& t = h->tc;
    const int slots[3] = {E_A, E_CV, E_Y2};
    float* const dst[3] = {t.aT, t.cT, t.Y2T};
    const int words[3] = {TS_AMAX_A, TS_AMAX_CV, TS_AMAX_Y2};
    int rc = tc_transpose_slots(h, 3, slots, dst, words, E_Y2, t.Yimg, true, st);
    if (rc) return rc;
    return tc_contract(h, t.aT, t.cT, E_GA1, E_GA2, false, st);
}

int tc_backward_dq(rae_engine* h, cudaStream_t st) {
    TcState& t = h->tc;
    TcDqArgs p{};
    p.bop2 = reinterpret_cast<const uint4*>(t.bop2); p.sc = h->sc; p.aT = t.aT; p.LT = t.LT; p.RT = t.RT; p.cT = t.cT; p.Y2T = t.Y2T;
    p.dqT = t.dqT; p.scal = t.scal; p.g_bound = (float)((double)h->S / h->Z);
    p.B = h->B; p.d = h->d; p.dp = h->dp; p.K = h->K; p.NK = t.NK;
    p.n_bil_rows = t.n_bil_rows;
    p.sch = t.sch_dq;
    p.segs = t.segs + t.segs_dq;
    if (t.DP == 32) launch_pdl(k_tc_dq<32>, dim3(p.sch.G), dim3(TC_BWD_THREADS), t.smem_dq, st, p);
    else if (t.DP == 64) launch_pdl(k_tc_dq<64>, dim3(p.sch.G), dim3(TC_BWD_THREADS), t.smem_dq, st, p);
    else launch_pdl(k_tc_dq<128>, dim3(p.sch.G), dim3(TC_BWD_THREADS), t.smem_dq, st, p);
    h->launches += 1;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

int tc_backward_finish(rae_engine* h, cudaStream_t st) {
    TcState& t = h->tc;
    const int blocks = (h->B + 31) / 32;
    if (blocks > h->n_dz_part) return fail(h, RAE_EINVAL, "internal: dzsum_part too small");
    h->dz_part_used = blocks;
    const size_t smem = sizeof(float) * 32 * ((size_t)(h->K | 1) + h->K);
    launch_pdl(k_tc_bwd_finish, dim3(blocks), dim3(1024), smem, st, h->ev, h->sc, h->q, h->logq, t.dqT, h->dz, h->dzsum_part, h->B, h->K, t.NK, t.sch_dq,
                                               h->d, h->dp, h->hasSP ? 1 : 0, (float)(2.0 * h->cfg.alpha / h->Z));
    h->launches += 1;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

// dC, dC1, dC2 partials on the tensor path (k_dense_finalize sums the slots of every row tile / tile pair): every row tile
// through the two-tile FP16 kernel, or (B % 4 != 0, or its stages do not fit) through the one-tile kernel
int tc_grad_dense(rae_engine* h, cudaStream_t st) {
    TcState& t = h->tc;
    if (t.dc2) {
        TcDc2Args p{};
        p.pop4 = reinterpret_cast<const uint4*>(t.pop4); p.Rimg = t.Rimg; p.Yimg = t.Yimg; p.SPimg = t.SPimg; p.aT = t.aT; p.LT = t.LT; p.out = h->gC_part;
        p.scal = t.scal; p.g_bound = (float)((double)h->S / h->Z);
        p.B = h->B; p.d = h->d; p.dp = h->dp; p.K = h->K; p.NK = t.NK; p.DP = t.DP;
        p.n_bil_tiles = t.n_bil_rows / TC_M;
        p.n_bil_pairs = (p.n_bil_tiles + 1) / 2;
        p.split_stride = (size_t)h->off_gWb;
        p.sch = t.sch_dc2;
        p.segs = t.segs + t.segs_dc2;
        launch_pdl(k_tc_dc2, dim3(p.sch.G), dim3(TC_BWD_THREADS), t.smem_dc2, st, p);
        h->launches++;
        RAE_CUDA(h, cudaGetLastError());
    } else {
        TcDcArgs p{};
        p.pop3 = t.pop3; p.ev = h->ev; p.sc = h->sc; p.aT = t.aT; p.LT = t.LT; p.out = h->gC_part;
        p.B = h->B; p.d = h->d; p.dp = h->dp; p.K = h->K; p.NK = t.NK; p.DP = t.DP;
        p.n_bil_rows = t.n_bil_rows; p.n_rows_total = t.n_rows_total; p.hasM = h->hasM ? 1 : 0;
        p.nacc = t.dc_nacc;
        p.share = t.dc_share;
        p.split_stride = (size_t)h->off_gWb;
        p.sch = t.sch_dc;
        p.segs = t.segs + t.segs_dc;
        launch_pdl(k_tc_dc, dim3(p.sch.G), dim3(TC_BWD_THREADS), t.smem_dc, st, p);
        h->launches++;
        RAE_CUDA(h, cudaGetLastError());
    }
    return RAE_OK;
}

int tc_gather_lr(rae_engine* h, const int32_t* a1, const int32_t* a2, cudaStream_t st) {
    const int blocks = (h->B * 32 + 255) / 256;
    k_tc_gather_lr<<<blocks, 256, 0, st>>>(h->P[RAE_P_A], a1, a2, h->B, h->d, h->dp, h->quirk ? 1 : 0, h->ev);
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

namespace {
// ------------------------------------------------------------------------------------------------------------
// argument ranking (rae_rank_arguments): every held-out example's true argument against all N entities, per slot
//   s1(x) = A[x].(v + c1) + Ab[x],  s2(x) = A[x].(w + c2) + Ab[x]      (+ terms that do not depend on x)
//   rank = 1 + #{x != true : s(x) > s(true)}
// The scores form the GEMM D[query, x] = U[query] . A[x] with fp32 accuracy through the FP16 pair split of the forward
// contraction (hi.hi + hi.lo + lo.hi, power-of-two operand scales): the queries are the A operand, resident in TMEM,
// 128 per tile; the candidates stream through shared memory in 128-row chunks, each ONE bulk copy of a pre-split image
// that also carries the chunk's 128 biases (-inf for the padding rows beyond N).  The epilogue compares every
// accumulator against the query's fp32 threshold t = U . A[true] + Ab[true] and counts in a register: no score is
// stored.  Chain length per accumulator: 3 ceil(d / 16) <= 48 MMAs.
// ------------------------------------------------------------------------------------------------------------
constexpr int RK_WORKERS = 8;          // epilogue warps 0..7 (group g = warp / 4 takes accumulator columns [64 g, 64 g + 64))
constexpr int RK_THREADS = 384;        // 8 epilogue + MMA issuer + producer + TMEM allocator + idle
constexpr uint32_t RK_ACOL = 256;      // TMEM: accumulator stages [0, 256) (2 x 128 columns), query operand hi / lo from 256
constexpr int RK_MAX_STAGES = 4;
constexpr int RK_PASS_ROWS = 131072;   // examples per ranking launch (query image: 2 x 131072 x DH x 4 bytes)

// bytes of one candidate chunk image: [hi/lo][kq < DH/8][row < 128] x 16 B, then float Ab[128]
__host__ __device__ constexpr size_t rank_chunk_bytes(int DH) { return (size_t)512 * DH + 512; }

// A -> candidate chunk images, scaled by pow2_scale(|max A|) (*amax, from k_tc_absmax).  Thread = (chunk, kq, row): it
// reads 8 consecutive columns of one row of A and writes its 16-byte hi and lo units (consecutive threads: consecutive rows)
__global__ void __launch_bounds__(256) k_rank_prep_a(const float* __restrict__ A, const float* __restrict__ Ab, int64_t N, int d,
                                                     int DH, int NC, const uint32_t* __restrict__ amax, uint8_t* __restrict__ img) {
    pdl_enter();
    const float sA = pow2_scale(*amax);
    const int KQ8 = DH / 8;
    const size_t total = (size_t)NC * KQ8 * 128;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(idx & 127);
        const int kq = (int)((idx >> 7) % KQ8);
        const int64_t c = (int64_t)(idx / ((size_t)128 * KQ8));
        const int64_t n = c * 128 + r;
        const float* src = A + (size_t)n * d;
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = 8 * kq + 2 * u;
            const float x0 = (n < N && j < d) ? src[j] * sA : 0.f;
            const float x1 = (n < N && j + 1 < d) ? src[j + 1] * sA : 0.f;
            split_h2(x0, x1, hi[u], lo[u]);
        }
        uint8_t* base = img + (size_t)c * rank_chunk_bytes(DH);
        uint4* u4 = reinterpret_cast<uint4*>(base);
        u4[(size_t)kq * 128 + r] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        u4[(size_t)(KQ8 + kq) * 128 + r] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        if (kq == 0) reinterpret_cast<float*>(base + (size_t)512 * DH)[r] = n < N ? Ab[n] : -INFINITY;
    }
}

// the rows of a partial last chunk, padded to B with empty rows and entity 0 (their ranks are not stored)
__global__ void __launch_bounds__(256) k_rank_pad(const int32_t* __restrict__ indptr, const int32_t* __restrict__ a1,
                                                  const int32_t* __restrict__ a2, int m, int B, int32_t* __restrict__ ip_out,
                                                  int32_t* __restrict__ a1_out, int32_t* __restrict__ a2_out) {
    pdl_enter();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= B; i += gridDim.x * blockDim.x) {
        ip_out[i] = indptr[min(i, m)];
        if (i < B) { a1_out[i] = i < m ? a1[i] : 0; a2_out[i] = i < m ? a2[i] : 0; }
    }
}

// query vectors of one forward chunk (ev after the contraction: v, w, c1, c2) -> the ranking kernel's operand image.
// One warp per (example i < m, slot s); query index s * Rpad + off + i.  Per query: its own power-of-two scale
// (pow2_scale(|max U|)), the unscale factor 1 / (s_U s_A), the fp32 threshold U . A[true] + Ab[true] and the true id.
// Image: [query tile][word w < DH][row < 128] uint32, words w < DH/2 the hi FP16 pairs (columns 2w, 2w + 1), then lo.
struct RankQArgs {
    const float* ev; const float* A; const float* Ab; const int32_t* a1; const int32_t* a2; const uint32_t* amaxA;
    uint32_t* qimg; float* qinv; float* qthr; int32_t* qtrue;
    int m, off, Rpad, d, dp, DH, hasM, hasSP;
};
__global__ void __launch_bounds__(256) k_rank_queries(RankQArgs p) {
    pdl_enter();
    const int lane = threadIdx.x & 31;
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (gw >= 2 * p.m) return;
    const int s = gw & 1, i = gw >> 1;
    const float* evb = p.ev + (size_t)i * E_NV * p.dp;
    const float* vs = evb + (s == 0 ? E_V1 : E_V2) * p.dp;
    const float* cs = evb + (s == 0 ? E_C1 : E_C2) * p.dp;
    auto u_at = [&](int j) -> float {
        if (j >= p.d) return 0.f;
        float x = p.hasM ? vs[j] : 0.f;
        if (p.hasSP) x += cs[j];
        return x;
    };
    const int tru = s == 0 ? p.a1[i] : p.a2[i];
    const float* Ar = p.A + (size_t)tru * p.d;
    float dot = 0.f, amax = 0.f;
    for (int j = lane; j < p.d; j += 32) {
        const float x = u_at(j);
        dot = fmaf(x, Ar[j], dot);
        amax = fmaxf(amax, fabsf(x));
    }
    dot = warp_sum(dot);
    amax = warp_max(amax);
    const float sU = pow2_scale(__float_as_uint(amax));
    const int q = s * p.Rpad + p.off + i;
    if (lane == 0) {
        p.qthr[q] = dot + p.Ab[tru];
        p.qinv[q] = 1.f / (sU * pow2_scale(*p.amaxA));
        p.qtrue[q] = tru;
    }
    uint32_t* img = p.qimg + (size_t)(q >> 7) * p.DH * 128 + (q & 127);
    const int half = p.DH / 2;
    for (int c = lane; c < half; c += 32) {
        uint32_t hi, lo;
        split_h2(u_at(2 * c) * sU, u_at(2 * c + 1) * sU, hi, lo);
        img[(size_t)c * 128] = hi;
        img[(size_t)(half + c) * 128] = lo;
    }
}

struct RankArgs {
    const uint8_t* aimg;        // candidate chunk images (k_rank_prep_a)
    const uint32_t* qimg; const float* qinv; const float* qthr; const int32_t* qtrue;   // k_rank_queries
    int32_t* out1; int32_t* out2;   // ranks of the pass's first example, zeroed; counts are added with integer atomics
    int NC, DH, nbs;
    int Rpad, nr;               // queries of slot s at [s Rpad, s Rpad + nr)
    int n_tiles, splits;        // work item = (query tile, candidate range); item = tile * splits + split
    float* ps; int32_t* pi;     // TopK: partial lists, [item][group][KT][128 rows] scores / ids
};

// Epilogue policies of the ranking GEMM.  step() sees 32 consecutive candidate columns [col0, col0 + 32) of one query
// row: t the raw accumulators, a the biases; the score is fmaf(t, inv, a).  finish() runs once per work item.
struct RankCount {               // rank: count the candidates above the true argument's threshold (no score is stored)
    int cnt = 0;
    __device__ __forceinline__ void step(const float (&t)[32], const float (&a)[32], float inv, float thr, int tru, int col0) {
        const int tcol = tru - col0;   // the true entity's column in these 32, if any
        if (__any_sync(kFull, (unsigned)tcol < 32u)) {
#pragma unroll
            for (int x = 0; x < 32; ++x) cnt += (fmaf(t[x], inv, a[x]) > thr && x != tcol) ? 1 : 0;
        } else {
#pragma unroll
            for (int x = 0; x < 32; ++x) cnt += fmaf(t[x], inv, a[x]) > thr ? 1 : 0;
        }
    }
    __device__ __forceinline__ void finish(const RankArgs& p, bool valid, int slot, int r, int g, int, int split, int) {
        if (valid) atomicAdd((slot ? p.out2 : p.out1) + r, cnt + ((g == 0 && split == 0) ? 1 : 0));
    }
};

// predict: keep the KT best (score, id) of the row's candidates, score descending then id ascending, sorted in registers.
// A thread sees its ids in ascending order, so the strict > keeps the lower id on equal scores.  The -inf padding rows
// never enter (k <= N real candidates exist, the merge drops the -inf / INT_MAX fillers).
template <int KT>
struct RankTopK {
    float s[KT];
    int id[KT];
    __device__ __forceinline__ RankTopK() {
#pragma unroll
        for (int j = 0; j < KT; ++j) { s[j] = -INFINITY; id[j] = 0x7fffffff; }
    }
    __device__ __forceinline__ void step(const float (&t)[32], const float (&a)[32], float inv, float, int, int col0) {
#pragma unroll
        for (int x = 0; x < 32; ++x) {
            const float v = fmaf(t[x], inv, a[x]);
            if (v > s[KT - 1]) {
#pragma unroll
                for (int j = KT - 1; j > 0; --j) {
                    const bool up = v > s[j - 1];
                    const bool here = !up && v > s[j];
                    s[j] = up ? s[j - 1] : (here ? v : s[j]);
                    id[j] = up ? id[j - 1] : (here ? col0 + x : id[j]);
                }
                if (v > s[0]) { s[0] = v; id[0] = col0 + x; }
            }
        }
    }
    __device__ __forceinline__ void finish(const RankArgs& p, bool, int, int, int g, int item, int, int row) {
        const size_t base = ((size_t)item * 2 + g) * KT * 128 + row;
#pragma unroll
        for (int j = 0; j < KT; ++j) { p.ps[base + (size_t)j * 128] = s[j]; p.pi[base + (size_t)j * 128] = id[j]; }
    }
};

// Persistent: CTA x takes items x, x + G, ...  When the query tiles outnumber the SMs every CTA sweeps ALL candidate
// chunks in the same order at the same rate, so the CTAs resident together read each chunk from L2 (A is read from HBM
// about once per wave instead of once per query tile).  With fewer tiles than SMs the candidates are split into ranges.
template <class Epi>
__device__ __forceinline__ void tc_rank_body(const RankArgs& p) {
    pdl_enter();
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t CB = (uint32_t)rank_chunk_bytes(p.DH);
    const uint32_t KQ8 = (uint32_t)p.DH / 8u;
    const uint32_t HALF = (uint32_t)p.DH / 2u;         // TMEM columns of one query plane (two fp16 per column)
    const int nbs = p.nbs;
    uint8_t* smB = smem_raw;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + (size_t)nbs * CB);
    uint64_t* a_full = bars;                           // 8 epilogue-warp arrivals per item: query operand is in TMEM
    uint64_t* b_full = bars + 1;                       // [RK_MAX_STAGES]
    uint64_t* b_empty = b_full + RK_MAX_STAGES;        // [RK_MAX_STAGES] MMA commit + 8 epilogue warps (they read the biases)
    uint64_t* t_full = b_empty + RK_MAX_STAGES;        // [2]
    uint64_t* t_empty = t_full + 2;                    // [2] 8 epilogue-warp arrivals
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 2);
    if (threadIdx.x == 0) {
        mbar_init(a_full, RK_WORKERS);
        for (int s = 0; s < nbs; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1 + RK_WORKERS); }
        for (int s = 0; s < 2; ++s) { mbar_init(&t_full[s], 1); mbar_init(&t_empty[s], RK_WORKERS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == RK_WORKERS + 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int n_items = p.n_tiles * p.splits;
    auto range = [&](int item, int& c0, int& c1) {
        const int split = item % p.splits;
        c0 = (int)((long long)split * p.NC / p.splits);
        c1 = (int)((long long)(split + 1) * p.NC / p.splits);
    };

    if (warp == RK_WORKERS + 1) {
        // ===== producer: one bulk copy per candidate chunk =====
        if (lane == 0) {
            int it = 0;
            for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
                int c0, c1;
                range(item, c0, c1);
                for (int c = c0; c < c1; ++c, ++it) {
                    const int s = it % nbs;
                    mbar_wait(&b_empty[s], ((it / nbs) & 1) ^ 1);
                    mbar_expect_tx(&b_full[s], CB);
                    bulk_g2s_pieces(smB + (size_t)s * CB, p.aimg + (size_t)c * CB, CB, &b_full[s]);
                }
            }
        }
    } else if (warp == RK_WORKERS) {
        // ===== MMA issuer (one elected thread); k-loop unrolled so every descriptor is the stage base + a constant =====
        if (elect_one()) {
            const uint32_t idesc = make_idesc_f16(TC_M, 128);
            const uint32_t a_hi = tmem_base + RK_ACOL, a_lo = a_hi + HALF;
            const int ksteps = p.DH / 16;              // 1 .. 16
            int it = 0, k = 0;
            for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++k) {
                int c0, c1;
                range(item, c0, c1);
                mbar_wait(a_full, k & 1);
                tc_fence_after();
                for (int c = c0; c < c1; ++c, ++it) {
                    const int s = it % nbs, ts = it & 1;
                    mbar_wait(&t_empty[ts], ((it >> 1) & 1) ^ 1);
                    mbar_wait(&b_full[s], (it / nbs) & 1);
                    tc_fence_after();
                    const uint32_t b_hi = smem_u32(smB + (size_t)s * CB);
                    const uint64_t h0 = make_desc(b_hi, 128u * 16u, 128u);
                    const uint64_t l0 = make_desc(b_hi + KQ8 * 128u * 16u, 128u * 16u, 128u);
                    const uint32_t d0 = tmem_base + (uint32_t)(ts * 128);
#pragma unroll
                    for (int ks = 0; ks < 16; ++ks) {
                        if (ks < ksteps) {
                            const uint64_t hk = desc_advance(h0, (uint32_t)ks * 2u * 128u * 16u);
                            const uint64_t lk = desc_advance(l0, (uint32_t)ks * 2u * 128u * 16u);
                            tc_mma_f16_ts(d0, a_hi + 8u * ks, hk, idesc, ks > 0 ? 1u : 0u);   // hi * hi
                            tc_mma_f16_ts(d0, a_hi + 8u * ks, lk, idesc, 1u);                 // hi * lo
                            tc_mma_f16_ts(d0, a_lo + 8u * ks, hk, idesc, 1u);                 // lo * hi
                        }
                    }
                    tc_commit(&b_empty[s]);
                    tc_commit(&t_full[ts]);
                }
            }
        }
        __syncwarp();
    } else if (warp < RK_WORKERS) {
        // ===== query operand -> TMEM, then the counting epilogue =====
        const int g = warp >> 2, q4 = warp & 3;
        const int row = q4 * 32 + lane;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q4 * 32) << 16);
        int it = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
            const int tile = item / p.splits, split = item % p.splits;
            int c0, c1;
            range(item, c0, c1);
            {
                // group g writes plane g (hi, lo) of its 32 rows.  After the first item this warp has seen t_full of the
                // previous item's last chunk: every MMA that read the old operand is done.
                const uint32_t* src = p.qimg + ((size_t)tile * p.DH + g * HALF) * 128 + row;
                for (uint32_t w0 = 0; w0 < HALF; w0 += 32) {
                    uint32_t w[4][8];
#pragma unroll
                    for (int u = 0; u < 4; ++u)
#pragma unroll
                        for (int e = 0; e < 8; ++e) w[u][e] = (w0 + 8 * u < HALF) ? __ldg(src + (size_t)(w0 + 8 * u + e) * 128) : 0u;
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (w0 + 8 * u < HALF) tc_st8u(lane_base + RK_ACOL + g * HALF + w0 + 8 * u, w[u]);
                }
                tc_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(a_full);
            }
            const int qi = tile * 128 + row;
            const int slot = qi >= p.Rpad ? 1 : 0, r = qi - slot * p.Rpad;
            const bool valid = r < p.nr;
            const float thr = valid ? p.qthr[qi] : INFINITY;     // padding rows count nothing
            const float inv = valid ? p.qinv[qi] : 0.f;
            const int tru = valid ? p.qtrue[qi] : -1;
            Epi epi;
            for (int c = c0; c < c1; ++c, ++it) {
                const int s = it % nbs, ts = it & 1;
                mbar_wait(&t_full[ts], (it >> 1) & 1);
                mbar_wait(&b_full[s], (it / nbs) & 1);         // the biases: this phase cannot complete again before our b_empty arrival
                tc_fence_after();
                const float* ab = reinterpret_cast<const float*>(smB + (size_t)s * CB + (size_t)512 * p.DH) + 64 * g;
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    float t[32];
                    tc_ld32(lane_base + (uint32_t)(ts * 128 + 64 * g + 32 * hf), t);
                    if (hf == 1) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&t_empty[ts]);
                    }
                    float a[32];
#pragma unroll
                    for (int x = 0; x < 32; x += 4) {
                        const float4 v = *reinterpret_cast<const float4*>(ab + 32 * hf + x);
                        a[x] = v.x; a[x + 1] = v.y; a[x + 2] = v.z; a[x + 3] = v.w;
                    }
                    epi.step(t, a, inv, thr, tru, c * 128 + 64 * g + 32 * hf);
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&b_empty[s]);
            }
            epi.finish(p, valid, slot, r, g, item, split, row);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == RK_WORKERS + 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

__global__ void __launch_bounds__(RK_THREADS, 1) k_tc_rank(RankArgs p) { tc_rank_body<RankCount>(p); }

template <int KT>
__global__ void __launch_bounds__(RK_THREADS, 1) k_tc_predict(RankArgs p) { tc_rank_body<RankTopK<KT>>(p); }

// the 2 * splits partial lists of a query -> its first k entries under (score descending, id ascending).  One warp per
// query: each lane keeps the best KT of the entries lane, lane + 32, ..., then k rounds of a butterfly arg-best over the
// lanes' heads, the owning lane popping its head.  Ids are unique, so the result does not depend on how the candidates
// were split; no floating-point arithmetic is done.
struct PredictMergeArgs {
    const float* ps; const int32_t* pi;
    int32_t* ids1; float* sc1; int32_t* ids2; float* sc2;   // [nr, k] of the pass's first example
    int nr, Rpad, splits, k;
};
__device__ __forceinline__ bool pred_before(float v, int x, float w, int y) { return v > w || (v == w && x < y); }

template <int KT>
__global__ void __launch_bounds__(256) k_predict_merge(PredictMergeArgs p) {
    pdl_enter();
    const int lane = threadIdx.x & 31;
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (gw >= 2 * p.nr) return;
    const int slot = gw >= p.nr ? 1 : 0, r = gw - slot * p.nr;
    const int qi = slot * p.Rpad + r, tile = qi >> 7, row = qi & 127;
    float s[KT];
    int id[KT];
#pragma unroll
    for (int j = 0; j < KT; ++j) { s[j] = -INFINITY; id[j] = 0x7fffffff; }
    const int n = 2 * p.splits * KT;
    const size_t base = (size_t)tile * p.splits * 2 * KT * 128 + row;   // lists (split, group) of the tile's items
    for (int e = lane; e < n; e += 32) {
        const float v = p.ps[base + (size_t)e * 128];
        const int x = p.pi[base + (size_t)e * 128];
        if (pred_before(v, x, s[KT - 1], id[KT - 1])) {
#pragma unroll
            for (int j = KT - 1; j > 0; --j) {
                const bool up = pred_before(v, x, s[j - 1], id[j - 1]);
                const bool here = !up && pred_before(v, x, s[j], id[j]);
                s[j] = up ? s[j - 1] : (here ? v : s[j]);
                id[j] = up ? id[j - 1] : (here ? x : id[j]);
            }
            if (pred_before(v, x, s[0], id[0])) { s[0] = v; id[0] = x; }
        }
    }
    int32_t* ids = (slot ? p.ids2 : p.ids1) + (size_t)r * p.k;
    float* sc = (slot ? p.sc2 : p.sc1) + (size_t)r * p.k;
    for (int j = 0; j < p.k; ++j) {
        float bv = s[0];
        int bi = id[0];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(kFull, bv, o);
            const int oi = __shfl_xor_sync(kFull, bi, o);
            if (pred_before(ov, oi, bv, bi)) { bv = ov; bi = oi; }
        }
        if (id[0] == bi) {
#pragma unroll
            for (int u = 0; u < KT - 1; ++u) { s[u] = s[u + 1]; id[u] = id[u + 1]; }
            s[KT - 1] = -INFINITY;
            id[KT - 1] = 0x7fffffff;
        }
        if (lane == 0) { ids[j] = bi; sc[j] = bv; }
    }
}

// what one call of the driver produces: kt = 0 counts ranks into rank1 / rank2; kt in {1, 2, 4, 8, 16} keeps the best
// kt candidates per query and writes the first k of them to ids / scores
struct RankOutputs {
    int32_t* rank1; int32_t* rank2;
    int kt, k;
    int32_t* ids1; float* sc1; int32_t* ids2; float* sc2;
};

template <int KT>
void predict_kernels(void (*&kern)(RankArgs), void (*&merge)(PredictMergeArgs)) { kern = k_tc_predict<KT>; merge = k_predict_merge<KT>; }

// A image, forward pass in chunks of B rows (the tail chunk padded), query packing, one tcgen05 launch per pass of up to
// RK_PASS_ROWS rows with the epilogue `o` selects (plus the merge of the partial lists for top-k)
int launch_rank_driver(rae_engine* h, const char* what, const int32_t* indptr, const int32_t* indices, const int32_t* a1,
                       const int32_t* a2, int64_t n_rows, const RankOutputs& o, cudaStream_t st) {
    if (n_rows == 0) return RAE_OK;
    const int B = h->B, d = h->d, DH = (d + 15) & ~15;
    const int64_t N = h->cfg.N;
    if (N > ((int64_t)1 << 31) - 256) return fail(h, RAE_EINVAL, "%s: N = %lld entities are too many", what, (long long)N);
    void (*kern)(RankArgs) = k_tc_rank;
    void (*merge)(PredictMergeArgs) = nullptr;
    switch (o.kt) {
        case 0: break;
        case 1: predict_kernels<1>(kern, merge); break;
        case 2: predict_kernels<2>(kern, merge); break;
        case 4: predict_kernels<4>(kern, merge); break;
        case 8: predict_kernels<8>(kern, merge); break;
        case 16: predict_kernels<16>(kern, merge); break;
        default: return fail(h, RAE_EINVAL, "%s: no top-%d epilogue", what, o.kt);
    }
    const int NC = (int)((N + 127) / 128);
    const size_t CB = rank_chunk_bytes(DH);
    const int nbs = (int)std::min<size_t>(RK_MAX_STAGES, ((size_t)h->max_smem_optin - 256) / CB);
    if (nbs < 1) return fail(h, RAE_EINVAL, "%s: d = %d needs %zu bytes per candidate stage", what, d, CB);
    // more than half the shared memory: one CTA per SM, so no CTA waits in tcgen05.alloc for another's 512 columns
    const size_t smem = std::max<size_t>((size_t)nbs * CB + 256, (size_t)h->max_smem_optin / 2 + 1024);
    const int64_t cpp = std::max<int64_t>(1, RK_PASS_ROWS / B);              // forward chunks of B rows per ranking pass
    const int64_t pass_rows = std::min<int64_t>(cpp, (n_rows + B - 1) / B) * B;
    const int64_t Rmax = (pass_rows + 127) / 128 * 128;
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t b_img = al((size_t)NC * CB), b_q = al((size_t)2 * Rmax * DH * 4), b_m = al((size_t)2 * Rmax * 4),
                 b_pad = al((size_t)(B + 1) * 4), b_a = al((size_t)B * 4);
    // top-k partial lists: one per (item, group); items <= max(query tiles, SMs) since splits <= num_sms / n_tiles
    const int64_t max_items = std::max<int64_t>(2 * Rmax / 128, h->num_sms);
    const size_t b_part = o.kt ? al((size_t)max_items * 2 * o.kt * 128 * 4) : 0;
    const size_t total = 256 + b_img + b_q + 3 * b_m + b_pad + 2 * b_a + 2 * b_part;
    uint8_t* ws = nullptr;
    cudaError_t e = cudaMallocAsync((void**)&ws, total, st);
    if (e != cudaSuccess) return fail(h, RAE_ENOMEM, "%s: %zu bytes of workspace: %s", what, total, cudaGetErrorString(e));
    uint32_t* amax = reinterpret_cast<uint32_t*>(ws);
    uint8_t* cur = ws + 256;
    auto take = [&](size_t b) { uint8_t* r = cur; cur += b; return r; };
    uint8_t* aimg = take(b_img);
    uint32_t* qimg = reinterpret_cast<uint32_t*>(take(b_q));
    float* qinv = reinterpret_cast<float*>(take(b_m));
    float* qthr = reinterpret_cast<float*>(take(b_m));
    int32_t* qtrue = reinterpret_cast<int32_t*>(take(b_m));
    int32_t* pad_ip = reinterpret_cast<int32_t*>(take(b_pad));
    int32_t* pad_a1 = reinterpret_cast<int32_t*>(take(b_a));
    int32_t* pad_a2 = reinterpret_cast<int32_t*>(take(b_a));
    float* ps = reinterpret_cast<float*>(take(b_part));
    int32_t* pi = reinterpret_cast<int32_t*>(take(b_part));
    auto body = [&]() -> int {
        int rc;
        if (!o.kt) {
            RAE_CUDA(h, cudaMemsetAsync(o.rank1, 0, sizeof(int32_t) * (size_t)n_rows, st));
            RAE_CUDA(h, cudaMemsetAsync(o.rank2, 0, sizeof(int32_t) * (size_t)n_rows, st));
        }
        RAE_CUDA(h, cudaMemsetAsync(amax, 0, sizeof(uint32_t), st));
        launch_pdl(k_tc_absmax, dim3(h->num_sms * 8), dim3(256), 0, st, (const float*)h->P[RAE_P_A], (size_t)N * d, (const float*)nullptr,
                   (size_t)0, (const float*)nullptr, (size_t)0, amax);
        {
            const size_t items = (size_t)NC * (DH / 8) * 128;
            const int blocks = (int)std::min<size_t>((items + 255) / 256, (size_t)h->num_sms * 16);
            launch_pdl(k_rank_prep_a, dim3(blocks), dim3(256), 0, st, (const float*)h->P[RAE_P_A], (const float*)h->P[RAE_P_AB], N, d, DH, NC,
                       (const uint32_t*)amax, aimg);
        }
        h->launches += 2;
        RAE_CUDA(h, cudaGetLastError());
        if (h->use_tc && (rc = tc_prepare_c(h, st))) return rc;
        RAE_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        for (int64_t row0 = 0; row0 < n_rows; row0 += pass_rows) {
            const int nr = (int)std::min<int64_t>(pass_rows, n_rows - row0);
            const int Rpad = (nr + 127) / 128 * 128;
            for (int off = 0; off < nr; off += B) {
                const int m = std::min(B, nr - off);
                const int64_t r = row0 + off;
                const int32_t* ip = indptr + r;
                const int32_t* x1 = a1 + r;
                const int32_t* x2 = a2 + r;
                if (m < B) {
                    launch_pdl(k_rank_pad, dim3((B + 256) / 256), dim3(256), 0, st, ip, x1, x2, m, B, pad_ip, pad_a1, pad_a2);
                    h->launches++;
                    RAE_CUDA(h, cudaGetLastError());
                    ip = pad_ip; x1 = pad_a1; x2 = pad_a2;
                }
                if ((rc = launch_encoder_forward(h, ip, indices, B, h->q, h->logq, nullptr, nullptr, st))) return rc;
                if (h->use_tc) {
                    if ((rc = tc_prepare_p(h, x1, x2, st))) return rc;
                    if ((rc = tc_forward(h, st))) return rc;
                } else if ((rc = launch_bilinear_forward_simt(h, x1, x2, st))) {
                    return rc;
                }
                RankQArgs q{};
                q.ev = h->ev; q.A = h->P[RAE_P_A]; q.Ab = h->P[RAE_P_AB]; q.a1 = x1; q.a2 = x2; q.amaxA = amax;
                q.qimg = qimg; q.qinv = qinv; q.qthr = qthr; q.qtrue = qtrue;
                q.m = m; q.off = off; q.Rpad = Rpad; q.d = d; q.dp = h->dp; q.DH = DH; q.hasM = h->hasM; q.hasSP = h->hasSP;
                launch_pdl(k_rank_queries, dim3((2 * m + 7) / 8), dim3(256), 0, st, q);
                h->launches++;
                RAE_CUDA(h, cudaGetLastError());
            }
            RankArgs p{};
            p.aimg = aimg; p.qimg = qimg; p.qinv = qinv; p.qthr = qthr; p.qtrue = qtrue;
            if (!o.kt) { p.out1 = o.rank1 + row0; p.out2 = o.rank2 + row0; }
            p.ps = ps; p.pi = pi;
            p.NC = NC; p.DH = DH; p.nbs = nbs; p.Rpad = Rpad; p.nr = nr;
            p.n_tiles = 2 * Rpad / 128;
            // fewer query tiles than SMs: split the candidates, at least 8 chunks per range
            p.splits = (int)std::max<int64_t>(1, std::min<int64_t>(h->num_sms / p.n_tiles, NC / 8));
            const int G = std::min(h->num_sms, p.n_tiles * p.splits);
            launch_pdl(kern, dim3(G), dim3(RK_THREADS), smem, st, p);
            h->launches++;
            RAE_CUDA(h, cudaGetLastError());
            if (merge) {
                PredictMergeArgs m{};
                m.ps = ps; m.pi = pi;
                const size_t at = (size_t)row0 * o.k;
                m.ids1 = o.ids1 + at; m.sc1 = o.sc1 + at; m.ids2 = o.ids2 + at; m.sc2 = o.sc2 + at;
                m.nr = nr; m.Rpad = Rpad; m.splits = p.splits; m.k = o.k;
                launch_pdl(merge, dim3((2 * nr + 7) / 8), dim3(256), 0, st, m);
                h->launches++;
                RAE_CUDA(h, cudaGetLastError());
            }
        }
        return RAE_OK;
    };
    const int rc = body();
    cudaFreeAsync(ws, st);
    return rc;
}
}  // namespace

int launch_rank_arguments(rae_engine* h, const int32_t* indptr, const int32_t* indices, const int32_t* a1, const int32_t* a2,
                          int64_t n_rows, int32_t* rank1, int32_t* rank2, cudaStream_t st) {
    RankOutputs o{};
    o.rank1 = rank1; o.rank2 = rank2;
    return launch_rank_driver(h, "rae_rank_arguments", indptr, indices, a1, a2, n_rows, o, st);
}

int launch_predict_arguments(rae_engine* h, const int32_t* indptr, const int32_t* indices, const int32_t* a1, const int32_t* a2,
                             int64_t n_rows, int k, int32_t* ids1, float* scores1, int32_t* ids2, float* scores2,
                             cudaStream_t st) {
    if (k < 1 || k > RAE_MAX_TOPK || k > h->cfg.N)
        return fail(h, RAE_EINVAL, "rae_predict_arguments: k = %d outside [1, min(N = %lld, %d)]", k, (long long)h->cfg.N,
                    RAE_MAX_TOPK);
    RankOutputs o{};
    o.kt = 1;
    while (o.kt < k) o.kt *= 2;              // the first k of a top-kt list are the top-k list
    o.k = k; o.ids1 = ids1; o.sc1 = scores1; o.ids2 = ids2; o.sc2 = scores2;
    return launch_rank_driver(h, "rae_predict_arguments", indptr, indices, a1, a2, n_rows, o, st);
}

}  // namespace rae
