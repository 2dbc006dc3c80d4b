// Peer-memory data path of the row-sharded multi-GPU step (one process per GPU, NVLink / NVSwitch, CUDA IPC).
//
// The reference is single-process (no counterpart).  What is exchanged follows from its optimiser: Theano sums duplicate
// rows before AdaGrad squares the gradient (AdvancedIncSubtensor1 + Optimizers.py:29-32), so the owner of a row must see
// the SUM of every rank's contribution before it applies the rule once.
//
//   k_fetch_rows : compact[i,:] = shard[id % world][id / world, :]      rows read straight from the owner's HBM over
//                                                                      NVLink (or locally), one warp per row, 16-byte lanes
//   k_pull_apply : owner-side: g = sum_{rank order} grad_rank[slot,:]   remote reads of the ranks' reduced gradient rows,
//                  then ONE optimiser read-modify-write per row        fixed order -> bitwise reproducible
//   k_shard_apply: owner-side, l1 / l2 != 0: every row of the W shard  the touched rows' sums as above (0 elsewhere),
//                  + adj*(l1 sgn w + 2 l2 w), then the rule             one pass over the shard, a pure HBM stream
//
// No atomics, no collective: the only synchronisation the sparse path needs is "all ranks have emitted" (given by the
// dense-gradient all-reduce that precedes the pull) and "all owners have applied" (the end-of-step barrier).
#include <string.h>

#include <algorithm>

#include "rae_common.cuh"
#include "rae_internal.h"

namespace rae {

namespace {

struct PeerPtrs {
    const float* p[RAE_MAX_PEERS];
};

// remote gradient rows were written by another GPU during this step: read them past L1 (ld.global.cv)
__device__ __forceinline__ float4 ld_cv4(const float4* p) { return __ldcv(p); }
__device__ __forceinline__ float ld_cv(const float* p) { return __ldcv(p); }

template <bool VEC>
__global__ void __launch_bounds__(256) k_fetch_rows(PeerPtrs tabs, int world, int width, const int32_t* __restrict__ ids, int n,
                                                    float* __restrict__ out) {
    pdl_enter();
    const int lane = threadIdx.x & 31;
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nw = (gridDim.x * blockDim.x) >> 5;
    constexpr int UN = 4;                       // rows in flight per warp
    for (int i0 = gw * UN; i0 < n; i0 += nw * UN) {
        const float* src[UN];
#pragma unroll
        for (int u = 0; u < UN; ++u) {
            const int i = min(i0 + u, n - 1);
            const int id = ids[i];
            const int owner = id % world;
            src[u] = tabs.p[owner] + (size_t)(id / world) * width;
        }
        if (VEC) {
            const int nq = width >> 2;
            for (int q0 = lane; q0 < nq; q0 += 32) {
                float4 v[UN];
#pragma unroll
                for (int u = 0; u < UN; ++u) v[u] = __ldg(reinterpret_cast<const float4*>(src[u]) + q0);
#pragma unroll
                for (int u = 0; u < UN; ++u)
                    if (i0 + u < n) reinterpret_cast<float4*>(out + (size_t)(i0 + u) * width)[q0] = v[u];
            }
        } else {
            for (int k = lane; k < width; k += 32) {
                float v[UN];
#pragma unroll
                for (int u = 0; u < UN; ++u) v[u] = __ldg(src[u] + k);
#pragma unroll
                for (int u = 0; u < UN; ++u)
                    if (i0 + u < n) out[(size_t)(i0 + u) * width + k] = v[u];
            }
        }
    }
}

// width == 1 (bias table): one thread per row
__global__ void __launch_bounds__(256) k_fetch_scalars(PeerPtrs tabs, int world, const int32_t* __restrict__ ids, int n,
                                                       float* __restrict__ out) {
    pdl_enter();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int id = ids[i];
        out[i] = __ldg(tabs.p[id % world] + id / world);
    }
}

template <bool VEC>
__global__ void __launch_bounds__(256) k_pull_apply(float* __restrict__ table, float* __restrict__ acc, int width,
                                                    const int32_t* __restrict__ rows_local, const int32_t* __restrict__ ent_off,
                                                    const int32_t* __restrict__ ent_src, const int32_t* __restrict__ ent_slot,
                                                    int n_rows, PeerPtrs grads, float lr, int adagrad, const int32_t* __restrict__ abort) {
    pdl_enter();
    if (*abort != 0) return;      // a peer barrier of this handle timed out: the peers' gradient rows may be stale
    const int lane = threadIdx.x & 31;
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nw = (gridDim.x * blockDim.x) >> 5;
    for (int i = gw; i < n_rows; i += nw) {
        const int e0 = ent_off[i], e1 = ent_off[i + 1];
        const size_t rowoff = (size_t)rows_local[i] * width;
        // lanes 0..(e1-e0) hold the entries (at most `world` <= 16 per row)
        int my_src = 0, my_slot = 0;
        if (e0 + lane < e1) { my_src = ent_src[e0 + lane]; my_slot = ent_slot[e0 + lane]; }
        const int ne = e1 - e0;
        if (VEC) {
            const int nq = width >> 2;
            for (int q0 = lane; q0 < ((nq + 31) & ~31); q0 += 32) {
                const bool in = q0 < nq;
                float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
                float4 w = g, a = g;
                if (in) {
                    w = reinterpret_cast<const float4*>(table + rowoff)[q0];
                    if (adagrad) a = reinterpret_cast<const float4*>(acc + rowoff)[q0];
                }
                // contributions are read 4 at a time (remote loads over NVLink: ~2 us each, so they must be in flight
                // together) and added in rank order: deterministic
                for (int e0 = 0; e0 < ne; e0 += 4) {
                    float4 x[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int s = __shfl_sync(kFull, my_src, (e0 + u) & 31), slot = __shfl_sync(kFull, my_slot, (e0 + u) & 31);
                        x[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (in && e0 + u < ne) x[u] = ld_cv4(reinterpret_cast<const float4*>(grads.p[s] + (size_t)slot * width) + q0);
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) { g.x += x[u].x; g.y += x[u].y; g.z += x[u].z; g.w += x[u].w; }
                }
                if (in) {
                    opt_step(w, a, g, lr, adagrad);
                    if (adagrad) reinterpret_cast<float4*>(acc + rowoff)[q0] = a;
                    reinterpret_cast<float4*>(table + rowoff)[q0] = w;
                }
            }
        } else {
            for (int k0 = 0; k0 < width; k0 += 32) {
                const int k = k0 + lane;
                const bool in = k < width;
                float g = 0.f, w = 0.f, a = 0.f;
                if (in) {
                    w = table[rowoff + k];
                    if (adagrad) a = acc[rowoff + k];
                }
                for (int e0 = 0; e0 < ne; e0 += 4) {
                    float x[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int s = __shfl_sync(kFull, my_src, (e0 + u) & 31), slot = __shfl_sync(kFull, my_slot, (e0 + u) & 31);
                        x[u] = (in && e0 + u < ne) ? ld_cv(grads.p[s] + (size_t)slot * width + k) : 0.f;
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) g += x[u];
                }
                if (in) {
                    opt_step(w, a, g, lr, adagrad);
                    if (adagrad) acc[rowoff + k] = a;
                    table[rowoff + k] = w;
                }
            }
        }
    }
}

// regulariser term of one element, added to its (cross-rank summed) data gradient: the expression of k_dense_apply
// (rae_update.cu), OieModel.py:54-62 with adj folded into r1 = adj*l1, r2 = adj*l2
__device__ __forceinline__ void add_reg(float& g, float w, float r1, float r2) {
    const float sgn = (w > 0.f) ? 1.f : ((w < 0.f) ? -1.f : 0.f);
    g += r1 * sgn + 2.f * r2 * w;
}
__device__ __forceinline__ void add_reg(float4& g, const float4& w, float r1, float r2) {
    add_reg(g.x, w.x, r1, r2); add_reg(g.y, w.y, r1, r2); add_reg(g.z, w.z, r1, r2); add_reg(g.w, w.w, r1, r2);
}

// Owner-side pass of a regularised W: EVERY row of the rank's shard, not only the rows the batch touched - the regulariser
// makes every element's gradient non-zero.  Per element, in the order of the single-GPU k_dense_apply: the data gradient
// (the sum over the row's contributions in rank order, as k_pull_apply, or 0 for a row no rank touched), then
// adj*(l1 sgn w + 2 l2 w), then the optimiser rule: one read-modify-write of w and acc.
// A CTA owns the contiguous rows [r0, r0 + rpc).  One binary search finds the first touched row of the range in rows_local
// (ascending); the touched rows of the range are then merged into a shared per-row table of entry ranges, so the element
// loop below needs no scratch in global memory.  The element loop is a flat stream over the range's rows * width elements
// (16-byte units when VEC), SU units per thread in flight.
constexpr int SHARD_MAX_RPC = 1024;
template <bool VEC>
__global__ void __launch_bounds__(256) k_shard_apply(float* __restrict__ table, float* __restrict__ acc, int width, int shard_rows,
                                                     int rpc, const int32_t* __restrict__ rows_local, const int32_t* __restrict__ ent_off,
                                                     const int32_t* __restrict__ ent_src, const int32_t* __restrict__ ent_slot,
                                                     int n_rows, PeerPtrs grads, float lr, int adagrad, float r1, float r2,
                                                     const int32_t* __restrict__ abort) {
    __shared__ int s_e0[SHARD_MAX_RPC], s_ne[SHARD_MAX_RPC];
    __shared__ const float* s_gp[RAE_MAX_PEERS];       // indexed by source rank: from shared, not a local copy of the argument
    pdl_enter();
    if (*abort != 0) return;      // a peer barrier of this handle timed out: the peers' gradient rows may be stale
    const int r0 = blockIdx.x * rpc;
    const int r1_ = min(r0 + rpc, shard_rows);
    if (r0 >= r1_) return;
    for (int j = threadIdx.x; j < r1_ - r0; j += blockDim.x) s_ne[j] = 0;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int r = 0; r < RAE_MAX_PEERS; ++r) s_gp[r] = grads.p[r];
    }
    // first touched row >= r0 (every thread finds the same index; rows_local is read through L1)
    int lo = 0, hi = n_rows;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(rows_local + mid) < r0) lo = mid + 1;
        else hi = mid;
    }
    __syncthreads();
    for (int t = lo + threadIdx.x; t < n_rows; t += blockDim.x) {
        const int r = __ldg(rows_local + t);
        if (r >= r1_) break;                  // ascending: every later entry is past the range too
        const int e0 = __ldg(ent_off + t);
        s_e0[r - r0] = e0;
        s_ne[r - r0] = __ldg(ent_off + t + 1) - e0;
    }
    __syncthreads();
    constexpr int SU = 4;
    const int upr = VEC ? width >> 2 : width;            // units per row
    const int n_units = (r1_ - r0) * upr;
    float* const tb = table + (size_t)r0 * width;
    float* const ac = adagrad ? acc + (size_t)r0 * width : nullptr;
    for (int u0 = threadIdx.x; u0 < n_units; u0 += SU * blockDim.x) {
        int row[SU], col[SU];
        bool in[SU];
        if (VEC) {
            float4 w[SU], a[SU], g[SU];
#pragma unroll
            for (int s = 0; s < SU; ++s) {
                const int u = u0 + s * blockDim.x;
                in[s] = u < n_units;
                row[s] = in[s] ? u / upr : 0;
                col[s] = u - row[s] * upr;
                g[s] = make_float4(0.f, 0.f, 0.f, 0.f);
                w[s] = g[s]; a[s] = g[s];
                if (in[s]) {
                    w[s] = reinterpret_cast<const float4*>(tb)[u];
                    if (adagrad) a[s] = reinterpret_cast<const float4*>(ac)[u];
                }
            }
            // the contributions of the touched rows, entry j of every unit in flight together, added in rank order
            int ne_max = 0;
#pragma unroll
            for (int s = 0; s < SU; ++s) ne_max = max(ne_max, in[s] ? s_ne[row[s]] : 0);
            for (int j = 0; j < ne_max; ++j) {
                float4 x[SU];
#pragma unroll
                for (int s = 0; s < SU; ++s) {
                    x[s] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (in[s] && j < s_ne[row[s]]) {
                        const int e = s_e0[row[s]] + j;
                        x[s] = ld_cv4(reinterpret_cast<const float4*>(s_gp[__ldg(ent_src + e)] + (size_t)__ldg(ent_slot + e) * width) + col[s]);
                    }
                }
#pragma unroll
                for (int s = 0; s < SU; ++s)
                    if (in[s] && j < s_ne[row[s]]) { g[s].x += x[s].x; g[s].y += x[s].y; g[s].z += x[s].z; g[s].w += x[s].w; }
            }
#pragma unroll
            for (int s = 0; s < SU; ++s) {
                if (!in[s]) continue;
                const int u = u0 + s * blockDim.x;
                add_reg(g[s], w[s], r1, r2);
                opt_step(w[s], a[s], g[s], lr, adagrad);
                if (adagrad) reinterpret_cast<float4*>(ac)[u] = a[s];
                reinterpret_cast<float4*>(tb)[u] = w[s];
            }
        } else {
            float w[SU], a[SU], g[SU];
#pragma unroll
            for (int s = 0; s < SU; ++s) {
                const int u = u0 + s * blockDim.x;
                in[s] = u < n_units;
                row[s] = in[s] ? u / upr : 0;
                col[s] = u - row[s] * upr;
                g[s] = 0.f; w[s] = 0.f; a[s] = 0.f;
                if (in[s]) {
                    w[s] = tb[u];
                    if (adagrad) a[s] = ac[u];
                }
            }
            int ne_max = 0;
#pragma unroll
            for (int s = 0; s < SU; ++s) ne_max = max(ne_max, in[s] ? s_ne[row[s]] : 0);
            for (int j = 0; j < ne_max; ++j) {
                float x[SU];
#pragma unroll
                for (int s = 0; s < SU; ++s) {
                    x[s] = 0.f;
                    if (in[s] && j < s_ne[row[s]]) {
                        const int e = s_e0[row[s]] + j;
                        x[s] = ld_cv(s_gp[__ldg(ent_src + e)] + (size_t)__ldg(ent_slot + e) * width + col[s]);
                    }
                }
#pragma unroll
                for (int s = 0; s < SU; ++s)
                    if (in[s] && j < s_ne[row[s]]) g[s] += x[s];
            }
#pragma unroll
            for (int s = 0; s < SU; ++s) {
                if (!in[s]) continue;
                const int u = u0 + s * blockDim.x;
                add_reg(g[s], w[s], r1, r2);
                opt_step(w[s], a[s], g[s], lr, adagrad);
                if (adagrad) ac[u] = a[s];
                tb[u] = w[s];
            }
        }
    }
}

// width == 1: one thread per row
__global__ void __launch_bounds__(256) k_pull_apply_scalars(float* __restrict__ table, float* __restrict__ acc,
                                                            const int32_t* __restrict__ rows_local,
                                                            const int32_t* __restrict__ ent_off, const int32_t* __restrict__ ent_src,
                                                            const int32_t* __restrict__ ent_slot, int n_rows, PeerPtrs grads,
                                                            float lr, int adagrad, const int32_t* __restrict__ abort) {
    pdl_enter();
    if (*abort != 0) return;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_rows; i += gridDim.x * blockDim.x) {
        float g = 0.f;
        const int e1 = ent_off[i + 1];
        for (int e0 = ent_off[i]; e0 < e1; e0 += 4) {
            float x[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) x[u] = (e0 + u < e1) ? ld_cv(grads.p[ent_src[e0 + u]] + ent_slot[e0 + u]) : 0.f;
#pragma unroll
            for (int u = 0; u < 4; ++u) g += x[u];
        }
        const int r = rows_local[i];
        float w = table[r], a = adagrad ? acc[r] : 0.f;
        opt_step(w, a, g, lr, adagrad);
        if (adagrad) acc[r] = a;
        table[r] = w;
    }
}

// ---- barrier over the ranks of the node -------------------------------------------------------------------------------
// One warp.  Lane r publishes `epoch` in rank r's flag word [my rank] (release, system scope: everything this GPU wrote
// before - emitted gradient rows, updated table rows - is visible to a peer that observes the flag) and then waits until
// rank r has published >= epoch in OUR word [r] (acquire).  Epochs only grow, so a rank that is already one barrier ahead
// still satisfies the wait.  The spin is bounded (~2 s).  A timeout is FATAL for the handle: the device status word makes
// every later owner-side kernel (pulls, peer dense update) return without touching the tables - the peers' buffers may not
// be emitted yet - and the page-locked copy makes the next rae_dist_* / rae_peer_* call on the host fail.
struct FlagPtrs {
    int32_t* p[RAE_MAX_PEERS];
};

__global__ void k_peer_barrier(FlagPtrs flags, int rank, int world, int epoch, int32_t* __restrict__ status,
                               volatile int32_t* __restrict__ status_host, int word0) {
    pdl_enter();
    const int r = threadIdx.x;
    __threadfence_system();
    if (r < world && *status == 0) {
        int32_t* dst = flags.p[r] + word0 + rank;
        asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(dst), "r"(epoch) : "memory");
        const int32_t* src = flags.p[rank] + word0 + r;
        const long long t0 = clock64();
        int32_t v;
        for (;;) {
            asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(src) : "memory");
            if (v >= epoch) break;
            if (clock64() - t0 > 4000000000LL) {
                *status = 1;
                *status_host = 1;
                break;
            }
        }
    }
    __syncwarp();
    __threadfence_system();
}

// global cost = sum of the ranks' local costs in rank order (the same double on every rank); each rank published its own
// in its flag buffer (words [RAE_MAX_PEERS, RAE_MAX_PEERS+2)) before the "every rank has emitted" barrier
__global__ void k_global_cost(FlagPtrs flags, int world, double* __restrict__ out_dev, double* __restrict__ out_mapped) {
    pdl_enter();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int r = 0; r < world; ++r) {
            const double* p = reinterpret_cast<const double*>(flags.p[r] + RAE_MAX_PEERS);
            double v;
            asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
            s += v;
        }
        if (out_dev) *out_dev = s;
        *out_mapped = s;
    }
}

// func['train'] hands the step its negatives although their routing was planned when the epoch's negatives were bound:
// they must be the planned ones.  ids[slot[s, j]] == given[s, j] for both arrays, else the (mapped, sticky) flag is set.
__global__ void __launch_bounds__(256) k_check_negatives(const int32_t* __restrict__ ids, int64_t n_ids, const int32_t* __restrict__ s1,
                                                         const int32_t* __restrict__ s2, int64_t slot_ld, const int32_t* __restrict__ g1,
                                                         const int32_t* __restrict__ g2, int S, int B, int32_t* __restrict__ err_mapped) {
    bool bad = false;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)S * B; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t s = i / B, j = i - s * B;
        const int32_t c1 = s1[s * slot_ld + j], c2 = s2[s * slot_ld + j];
        bad |= c1 < 0 || c1 >= n_ids || c2 < 0 || c2 >= n_ids;
        if (!bad) bad |= ids[c1] != g1[i] || ids[c2] != g2[i];
    }
    if (__any_sync(kFull, bad) && (threadIdx.x & 31) == 0) *err_mapped = 1;
}

// dense optimiser step with the ranks' flat dense gradients summed on the fly, in rank order (identical on every rank):
// replaces "all-reduce, then k_dense_apply" when the gradient is small enough to be read from every peer.  A regularised
// segment (C | C1 | C2 when ext_reg) adds adj*(l1 sgn w + 2 l2 w) to the sum before the rule, as k_dense_apply does.
struct DenseSeg { float* p; float* acc; size_t begin, end; float r1, r2; };      // [begin, end) of the flat gradient
struct DenseSegs { DenseSeg s[4]; int count; };

__global__ void __launch_bounds__(256) k_dense_apply_peers(DenseSegs segs, PeerPtrs grads, int world, size_t i_begin, size_t i_end,
                                                           float* __restrict__ sum_out, float lr, int adagrad, int vec,
                                                           const int32_t* __restrict__ abort) {
    pdl_enter();
    if (*abort != 0) return;
    if (vec) {
        // 16-byte path (every segment boundary, i_begin and the buffers are 16-byte aligned): 4 elements per thread, the
        // peers' loads of all of them in flight together
        for (size_t i = i_begin + 4 * ((size_t)blockIdx.x * blockDim.x + threadIdx.x); i < i_end; i += 4 * (size_t)gridDim.x * blockDim.x) {
            float4 x[RAE_MAX_PEERS];
#pragma unroll
            for (int r = 0; r < RAE_MAX_PEERS; ++r)
                x[r] = r < world ? ld_cv4(reinterpret_cast<const float4*>(grads.p[r] + i)) : make_float4(0.f, 0.f, 0.f, 0.f);
            float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int r = 0; r < RAE_MAX_PEERS; ++r) { g.x += x[r].x; g.y += x[r].y; g.z += x[r].z; g.w += x[r].w; }
            if (sum_out) *reinterpret_cast<float4*>(sum_out + i) = g;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (k < segs.count && i >= segs.s[k].begin && i < segs.s[k].end) {
                    const size_t j = i - segs.s[k].begin;
                    float4 w = *reinterpret_cast<const float4*>(segs.s[k].p + j), a = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (adagrad) a = *reinterpret_cast<const float4*>(segs.s[k].acc + j);
                    float4 gk = g;
                    if (segs.s[k].r1 != 0.f || segs.s[k].r2 != 0.f) add_reg(gk, w, segs.s[k].r1, segs.s[k].r2);
                    opt_step(w, a, gk, lr, adagrad);
                    if (adagrad) *reinterpret_cast<float4*>(segs.s[k].acc + j) = a;
                    *reinterpret_cast<float4*>(segs.s[k].p + j) = w;
                }
            }
        }
        return;
    }
    for (size_t i = i_begin + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < i_end; i += (size_t)gridDim.x * blockDim.x) {
        float x[RAE_MAX_PEERS];
#pragma unroll
        for (int r = 0; r < RAE_MAX_PEERS; ++r) x[r] = r < world ? ld_cv(grads.p[r] + i) : 0.f;
        float g = 0.f;
#pragma unroll
        for (int r = 0; r < RAE_MAX_PEERS; ++r) g += x[r];
        if (sum_out) sum_out[i] = g;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (k < segs.count && i >= segs.s[k].begin && i < segs.s[k].end) {
                const size_t j = i - segs.s[k].begin;
                float w = segs.s[k].p[j], a = adagrad ? segs.s[k].acc[j] : 0.f;
                float gk = g;
                if (segs.s[k].r1 != 0.f || segs.s[k].r2 != 0.f) add_reg(gk, w, segs.s[k].r1, segs.s[k].r2);
                opt_step(w, a, gk, lr, adagrad);
                if (adagrad) segs.s[k].acc[j] = a;
                segs.s[k].p[j] = w;
            }
        }
    }
}

int fill_peers(rae_engine* h, const void* const* ptrs, int world, PeerPtrs* out, const char* what) {
    if (world < 1 || world > RAE_MAX_PEERS) return fail(h, RAE_EINVAL, "%s: world %d out of range [1, %d]", what, world, RAE_MAX_PEERS);
    memset(out, 0, sizeof(*out));
    for (int r = 0; r < world; ++r) {
        if (!ptrs[r]) return fail(h, RAE_EINVAL, "%s: null table pointer for rank %d", what, r);
        out->p[r] = static_cast<const float*>(ptrs[r]);
    }
    return RAE_OK;
}

}  // namespace

int launch_fetch_rows(rae_engine* h, const void* const* tables, int world, int64_t width, const int32_t* ids, int64_t n,
                      float* out, cudaStream_t st) {
    if (n <= 0) return RAE_OK;
    PeerPtrs pp;
    int rc = fill_peers(h, tables, world, &pp, "rae_fetch_rows");
    if (rc) return rc;
    if (width == 1) {
        const int blocks = (int)std::min<int64_t>((n + 255) / 256, (int64_t)h->num_sms * 8);
        launch_pdl(k_fetch_scalars, dim3(blocks), dim3(256), 0, st, pp, world, ids, (int)n, out);
    } else {
        const int64_t warps = (n + 3) / 4;
        const int blocks = (int)std::min<int64_t>((warps + 7) / 8, (int64_t)h->num_sms * 8);
        if ((width & 3) == 0) launch_pdl(k_fetch_rows<true>, dim3(blocks), dim3(256), 0, st, pp, world, (int)width, ids, (int)n, out);
        else launch_pdl(k_fetch_rows<false>, dim3(blocks), dim3(256), 0, st, pp, world, (int)width, ids, (int)n, out);
    }
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

int launch_pull_apply(rae_engine* h, float* table, float* acc, int64_t width, const int32_t* rows_local, const int32_t* ent_off,
                      const int32_t* ent_src, const int32_t* ent_slot, int64_t n_rows, const void* const* grads, int world,
                      cudaStream_t st) {
    if (n_rows <= 0) return RAE_OK;
    PeerPtrs pp;
    int rc = fill_peers(h, grads, world, &pp, "rae_pull_apply");
    if (rc) return rc;
    const float lr = (float)h->cfg.lr;
    const int adagrad = h->adagrad ? 1 : 0;
    if (width == 1) {
        const int blocks = (int)std::min<int64_t>((n_rows + 255) / 256, (int64_t)h->num_sms * 8);
        launch_pdl(k_pull_apply_scalars, dim3(blocks), dim3(256), 0, st, table, acc, rows_local, ent_off, ent_src, ent_slot, (int)n_rows, pp, lr, adagrad, h->peer_err_dev);
    } else {
        const int blocks = (int)std::min<int64_t>((n_rows + 7) / 8, (int64_t)h->num_sms * 16);
        if ((width & 3) == 0)
            launch_pdl(k_pull_apply<true>, dim3(blocks), dim3(256), 0, st, table, acc, (int)width, rows_local, ent_off, ent_src, ent_slot, (int)n_rows, pp, lr, adagrad, h->peer_err_dev);
        else
            launch_pdl(k_pull_apply<false>, dim3(blocks), dim3(256), 0, st, table, acc, (int)width, rows_local, ent_off, ent_src, ent_slot, (int)n_rows, pp, lr, adagrad, h->peer_err_dev);
    }
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

int launch_shard_apply(rae_engine* h, float* table, float* acc, int64_t width, const int32_t* rows_local, const int32_t* ent_off,
                       const int32_t* ent_src, const int32_t* ent_slot, int64_t n_rows, const void* const* grads, int world,
                       int64_t shard_rows, cudaStream_t st) {
    if (shard_rows <= 0) return RAE_OK;
    if (shard_rows >= ((int64_t)1 << 31) || shard_rows * width >= ((int64_t)1 << 40))
        return fail(h, RAE_EINVAL, "rae_shard_apply: shard of %lld rows is too large", (long long)shard_rows);
    PeerPtrs pp;
    int rc = fill_peers(h, grads, world, &pp, "rae_shard_apply");
    if (rc) return rc;
    const float lr = (float)h->cfg.lr;
    const int adagrad = h->adagrad ? 1 : 0;
    const float r1 = (float)(h->cfg.adj * h->cfg.l1), r2 = (float)(h->cfg.adj * h->cfg.l2);     // as launch_dense_apply
    // about 16K elements per CTA: a few passes of the element loop, a grid of several waves
    const int rpc = (int)std::max<int64_t>(1, std::min<int64_t>(SHARD_MAX_RPC, 16384 / width));
    const int blocks = (int)((shard_rows + rpc - 1) / rpc);
    bool vec = (width & 3) == 0 && (((uintptr_t)table | (uintptr_t)acc) & 15) == 0;
    for (int r = 0; r < world; ++r)
        if ((uintptr_t)pp.p[r] & 15) vec = false;
    if (vec)
        launch_pdl(k_shard_apply<true>, dim3(blocks), dim3(256), 0, st, table, acc, (int)width, (int)shard_rows, rpc, rows_local, ent_off,
                   ent_src, ent_slot, (int)n_rows, pp, lr, adagrad, r1, r2, h->peer_err_dev);
    else
        launch_pdl(k_shard_apply<false>, dim3(blocks), dim3(256), 0, st, table, acc, (int)width, (int)shard_rows, rpc, rows_local, ent_off,
                   ent_src, ent_slot, (int)n_rows, pp, lr, adagrad, r1, r2, h->peer_err_dev);
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

// a peer barrier of this handle has timed out (seen through the page-locked status word): every later call fails
int peer_failed(rae_engine* h) {
    if (*(volatile int32_t*)h->peer_err_pinned == 0) return RAE_OK;
    return fail(h, RAE_ECUDA, "a peer barrier timed out: a rank of the node did not arrive within ~2 s; the sharded tables were left "
                              "untouched from that step on - the run cannot continue");
}

// kind 0: words [0, RAE_MAX_PEERS) of the flag buffers; kind 1: words [RAE_FLAG_WORDS / 2, + RAE_MAX_PEERS) - a second,
// independent barrier sequence for the side stream (the ranks must issue the barriers of one kind in the same order)
int launch_peer_barrier(rae_engine* h, const void* const* flag_bufs, int world, int rank, cudaStream_t st, int kind) {
    if (world < 1 || world > RAE_MAX_PEERS || rank < 0 || rank >= world) return fail(h, RAE_EINVAL, "rae_peer_barrier: bad world / rank");
    FlagPtrs fp;
    memset(&fp, 0, sizeof(fp));
    for (int r = 0; r < world; ++r) {
        if (!flag_bufs[r]) return fail(h, RAE_EINVAL, "rae_peer_barrier: null flag buffer for rank %d", r);
        fp.p[r] = static_cast<int32_t*>(const_cast<void*>(flag_bufs[r]));
    }
    int& epoch = kind == 0 ? h->barrier_epoch : h->barrier_epoch1;
    epoch += 1;
    launch_pdl(k_peer_barrier, dim3(1), dim3(32), 0, st, fp, rank, world, epoch, h->peer_err_dev, h->peer_err_pinned,
               kind == 0 ? 0 : RAE_FLAG_WORDS / 2);
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

// part 0: every dense tensor; 1: the decoder tensors C | C1 | C2 only; 2: the encoder bias Wb only (the split tail of the
// sharded step applies Wb - read by the next step's encoder - on the main stream and the rest on a side stream)
int launch_dense_apply_peers(rae_engine* h, const void* const* dense_bufs, int world, cudaStream_t st, int part) {
    PeerPtrs pp;
    int rc = fill_peers(h, dense_bufs, world, &pp, "rae_dist_step_end(dense_bufs)");
    if (rc) return rc;
    DenseSegs segs{};
    bool aligned = true;
    // the decoder tensors carry the regulariser when ext_reg (OieModel.py:60-62); Wb never does
    const bool regdec = h->reg && h->cfg.ext_reg;
    const float r1 = regdec ? (float)(h->cfg.adj * h->cfg.l1) : 0.f, r2 = regdec ? (float)(h->cfg.adj * h->cfg.l2) : 0.f;
    auto add = [&](int pid, int64_t begin, int64_t n, bool regularised) {
        if (n <= 0) return;
        DenseSeg& sg = segs.s[segs.count++];
        sg.p = h->P[pid]; sg.acc = h->ACC[pid]; sg.begin = (size_t)begin; sg.end = (size_t)(begin + n);
        sg.r1 = regularised ? r1 : 0.f; sg.r2 = regularised ? r2 : 0.f;
        if ((begin & 3) || (n & 3) || (((uintptr_t)sg.p | (uintptr_t)sg.acc) & 15)) aligned = false;
    };
    const int64_t dd = h->hasM ? (int64_t)h->d * h->d * h->K : 0, dk = h->hasSP ? (int64_t)h->d * h->K : 0;
    add(RAE_P_C, h->off_gC, dd, true);
    add(RAE_P_C1, h->off_gC1, dk, true);
    add(RAE_P_C2, h->off_gC2, dk, true);
    add(RAE_P_WB, h->off_gWb, h->K, false);
    for (int r = 0; r < world; ++r)
        if ((uintptr_t)pp.p[r] & 15) aligned = false;
    const size_t i_begin = part == 2 ? (size_t)h->off_gWb : 0, i_end = part == 1 ? (size_t)h->off_gWb : (size_t)h->n_dense;
    if (i_end <= i_begin) return RAE_OK;
    const size_t n = i_end - i_begin, work = aligned ? (n + 3) / 4 : n;
    const int blocks = (int)std::min<size_t>((work + 255) / 256, (size_t)h->num_sms * 8);
    launch_pdl(k_dense_apply_peers, dim3(blocks), dim3(256), 0, st, segs, pp, world, i_begin, i_end, nullptr, (float)h->cfg.lr,
               h->adagrad ? 1 : 0, aligned ? 1 : 0, h->peer_err_dev);
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

}  // namespace rae

using namespace rae;

extern "C" {

int rae_peer_alloc(int64_t bytes, void** ptr_out, void* handle_out) {
    if (!ptr_out || bytes <= 0) return fail(nullptr, RAE_EINVAL, "rae_peer_alloc: bad argument");
    *ptr_out = nullptr;
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, (size_t)bytes);
    if (e != cudaSuccess) return fail(nullptr, RAE_ENOMEM, "rae_peer_alloc: cudaMalloc(%lld) failed: %s", (long long)bytes, cudaGetErrorString(e));
    if ((e = cudaMemset(p, 0, (size_t)bytes)) != cudaSuccess) {
        cudaFree(p);
        return fail(nullptr, RAE_ECUDA, "rae_peer_alloc: cudaMemset failed: %s", cudaGetErrorString(e));
    }
    if (handle_out) {
        static_assert(sizeof(cudaIpcMemHandle_t) == RAE_IPC_HANDLE_BYTES, "IPC handle size");
        cudaIpcMemHandle_t hd;
        if ((e = cudaIpcGetMemHandle(&hd, p)) != cudaSuccess) {
            cudaFree(p);
            return fail(nullptr, RAE_ECUDA, "rae_peer_alloc: cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
        }
        memcpy(handle_out, &hd, sizeof(hd));
    }
    *ptr_out = p;
    return RAE_OK;
}

int rae_peer_free(void* ptr) {
    if (!ptr) return RAE_OK;
    cudaError_t e = cudaFree(ptr);
    if (e != cudaSuccess) return fail(nullptr, RAE_ECUDA, "rae_peer_free: %s", cudaGetErrorString(e));
    return RAE_OK;
}

int rae_peer_open(const void* handle, void** ptr_out) {
    if (!handle || !ptr_out) return fail(nullptr, RAE_EINVAL, "rae_peer_open: null argument");
    cudaIpcMemHandle_t hd;
    memcpy(&hd, handle, sizeof(hd));
    cudaError_t e = cudaIpcOpenMemHandle(ptr_out, hd, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
        *ptr_out = nullptr;
        return fail(nullptr, RAE_ECUDA, "rae_peer_open: cudaIpcOpenMemHandle failed: %s", cudaGetErrorString(e));
    }
    return RAE_OK;
}

int rae_peer_close(void* ptr) {
    if (!ptr) return RAE_OK;
    cudaError_t e = cudaIpcCloseMemHandle(ptr);
    if (e != cudaSuccess) return fail(nullptr, RAE_ECUDA, "rae_peer_close: %s", cudaGetErrorString(e));
    return RAE_OK;
}

int rae_fetch_rows(rae_engine* h, const void* const* tables, int32_t world, int64_t width, const int32_t* ids, int64_t n,
                   float* out, void* stream) {
    if (!h || !tables || width < 1 || n < 0 || (n > 0 && (!ids || !out))) return fail(h, RAE_EINVAL, "rae_fetch_rows: bad argument");
    return launch_fetch_rows(h, tables, world, width, ids, n, out, (cudaStream_t)stream);
}

int rae_pull_apply(rae_engine* h, float* table, float* acc, int64_t width, const int32_t* rows_local, const int32_t* ent_off,
                   const int32_t* ent_src, const int32_t* ent_slot, int64_t n_rows, const void* const* grads, int32_t world,
                   void* stream) {
    if (!h || !table || !grads || width < 1 || n_rows < 0) return fail(h, RAE_EINVAL, "rae_pull_apply: bad argument");
    if (h->adagrad && !acc) return fail(h, RAE_EINVAL, "rae_pull_apply: AdaGrad needs the accumulator table");
    if (n_rows > 0 && (!rows_local || !ent_off || !ent_src || !ent_slot)) return fail(h, RAE_EINVAL, "rae_pull_apply: null plan arrays");
    return launch_pull_apply(h, table, acc, width, rows_local, ent_off, ent_src, ent_slot, n_rows, grads, world, (cudaStream_t)stream);
}

int rae_shard_apply(rae_engine* h, float* table, float* acc, int64_t width, const int32_t* rows_local, const int32_t* ent_off,
                    const int32_t* ent_src, const int32_t* ent_slot, int64_t n_rows, const void* const* grads, int32_t world,
                    int64_t shard_rows, void* stream) {
    if (!h || !grads || width < 1 || n_rows < 0 || shard_rows < 0 || (shard_rows > 0 && !table))
        return fail(h, RAE_EINVAL, "rae_shard_apply: bad argument");
    if (h->adagrad && shard_rows > 0 && !acc) return fail(h, RAE_EINVAL, "rae_shard_apply: AdaGrad needs the accumulator table");
    if (n_rows > 0 && (!rows_local || !ent_off || !ent_src || !ent_slot)) return fail(h, RAE_EINVAL, "rae_shard_apply: null plan arrays");
    return launch_shard_apply(h, table, acc, width, rows_local, ent_off, ent_src, ent_slot, n_rows, grads, world, shard_rows,
                              (cudaStream_t)stream);
}

int rae_peer_barrier(rae_engine* h, const void* const* flag_bufs, int32_t world, int32_t rank, void* stream) {
    // a stand-alone barrier orders EVERYTHING this handle has issued: the side streams' tails join the caller's stream first
    if (h && h->s1 && h->s2) {
        cudaStream_t st0 = (cudaStream_t)stream;
        if (cudaEventRecord(h->ev_join1, h->s1) == cudaSuccess) cudaStreamWaitEvent(st0, h->ev_join1, 0);
        if (cudaEventRecord(h->ev_join2, h->s2) == cudaSuccess) cudaStreamWaitEvent(st0, h->ev_join2, 0);
    }
    if (!h || !flag_bufs) return fail(h, RAE_EINVAL, "rae_peer_barrier: null argument");
    return launch_peer_barrier(h, flag_bufs, world, rank, (cudaStream_t)stream);
}

int rae_peer_status(rae_engine* h, void* stream) {
    if (!h) return RAE_EINVAL;
    int32_t v = 0;
    RAE_CUDA(h, cudaMemcpyAsync(&v, h->peer_err_dev, sizeof(v), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    RAE_CUDA(h, cudaStreamSynchronize((cudaStream_t)stream));
    if (v != 0) return fail(h, RAE_ECUDA, "a peer barrier timed out: a rank of the node did not arrive");
    return peer_failed(h);
}

#define RAE_DMARK(name, strm, sid)                                                         \
    do {                                                                                   \
        if (h->timeline && h->tl_n < RAE_TL_MAX) {                                         \
            RAE_CUDA(h, cudaEventRecord(h->tl_ev[h->tl_n], strm));                         \
            h->tl_name[h->tl_n] = name; h->tl_stream[h->tl_n] = sid; ++h->tl_n;            \
        }                                                                                  \
    } while (0)

int rae_bind_push_targets(rae_engine* h, const void* const* gw, const void* const* ga, const void* const* gab, int32_t world,
                          int32_t rank, int64_t f_cap, int64_t n_cap) {
    if (!h || !gw || !ga || !gab) return fail(h, RAE_EINVAL, "rae_bind_push_targets: null argument");
    if (!h->emit_only) return fail(h, RAE_EINVAL, "rae_bind_push_targets needs RAE_FLAG_EMIT_ONLY");
    if (world < 1 || world > RAE_MAX_PEERS || rank < 0 || rank >= world || f_cap <= 0 || n_cap <= 0)
        return fail(h, RAE_EINVAL, "rae_bind_push_targets: bad world / rank / capacity");
    float* host[3][RAE_MAX_PEERS] = {};
    for (int r = 0; r < world; ++r) {
        if (!gw[r] || !ga[r] || !gab[r]) return fail(h, RAE_EINVAL, "rae_bind_push_targets: null receive buffer of rank %d", r);
        host[0][r] = static_cast<float*>(const_cast<void*>(gw[r]));
        host[1][r] = static_cast<float*>(const_cast<void*>(ga[r]));
        host[2][r] = static_cast<float*>(const_cast<void*>(gab[r]));
    }
    if (h->push.w_dev == nullptr) {
        float** blk = nullptr;
        RAE_CUDA(h, cudaMalloc((void**)&blk, 3 * RAE_MAX_PEERS * sizeof(float*)));
        h->push.w_dev = blk; h->push.a_dev = blk + RAE_MAX_PEERS; h->push.ab_dev = blk + 2 * RAE_MAX_PEERS;
    }
    RAE_CUDA(h, cudaMemcpy(h->push.w_dev, host, sizeof(host), cudaMemcpyHostToDevice));
    h->push.world = world; h->push.rank = rank; h->push.f_cap = f_cap; h->push.n_cap = n_cap;
    h->push.on = true;
    return RAE_OK;
}

int rae_dist_set_dense_wait(rae_engine* h, void* event) {
    if (!h) return RAE_EINVAL;
    h->dense_wait = event;
    return RAE_OK;
}

int rae_dist_step_begin(rae_engine* h, const rae_dist_step* d, void* stream) {
    if (!h || !d) return fail(h, RAE_EINVAL, "rae_dist_step_begin: null argument");
    if (peer_failed(h)) return RAE_ECUDA;
    h->push.f_ids = d->f_ids;
    h->push.e_ids = d->e_ids;
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    h->tl_n = 0;
    h->tl_keep = true;
    RAE_DMARK("dist_start", st, 0);
    const bool side = h->s1 != nullptr && !h->profiling;
    if (side) {
        // entity rows arrive on the side stream that sorts the entity occurrences next; the main stream (W rows ->
        // encoder) only waits for them where the decoder first reads A
        RAE_CUDA(h, cudaEventRecord(h->ev_dfork, st));
        RAE_CUDA(h, cudaStreamWaitEvent(h->s1, h->ev_dfork, 0));
        if ((rc = rae_fetch_rows(h, d->a_shards, d->world, h->d, d->e_ids, d->n_e, d->Ac, h->s1))) return rc;
        if ((rc = rae_fetch_rows(h, d->ab_shards, d->world, 1, d->e_ids, d->n_e, d->Abc, h->s1))) return rc;
        RAE_CUDA(h, cudaEventRecord(h->ev_dfetch, h->s1));
        RAE_DMARK("fetch_entities", h->s1, 1);
        h->pending_wait = h->ev_dfetch;
    }
    if ((rc = rae_fetch_rows(h, d->w_shards, d->world, h->K, d->f_ids, d->n_f, d->Wc, stream))) return rc;
    RAE_DMARK("fetch_w", st, 0);
    if (!side) {
        if ((rc = rae_fetch_rows(h, d->a_shards, d->world, h->d, d->e_ids, d->n_e, d->Ac, stream))) return rc;
        if ((rc = rae_fetch_rows(h, d->ab_shards, d->world, 1, d->e_ids, d->n_e, d->Abc, stream))) return rc;
    }
    return rae_train_step_begin(h, d->batch_index, d->a1c, d->a2c, d->n1c, d->n2c, d->neg_ld, stream);
}

int rae_dist_step_begin_host(rae_engine* h, const rae_dist_step* d, const int32_t* neg1_host, int64_t ld1,
                             const int32_t* neg2_host, int64_t ld2, void* stream) {
    if (!h || !d) return fail(h, RAE_EINVAL, "rae_dist_step_begin_host: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    // the copy and the check ride on the W-update stream, which is idle until the step forks: off the critical path
    cudaStream_t sc = (h->s2 != nullptr && !h->profiling) ? h->s2 : st;
    int32_t *g1 = nullptr, *g2 = nullptr;
    int rc = stage_host_negatives(h, neg1_host, ld1, neg2_host, ld2, sc, &g1, &g2);
    if (rc) return rc;
    const int64_t n = (int64_t)h->S * h->B;
    if (n > 0) {
        const int blocks = (int)std::min<int64_t>((n + 255) / 256, (int64_t)h->num_sms);
        k_check_negatives<<<blocks, 256, 0, sc>>>(d->e_ids, d->n_e, d->n1c, d->n2c, d->neg_ld, g1, g2, h->S, h->B, h->neg_err_pinned);
        RAE_CUDA(h, cudaGetLastError());
    }
    return rae_dist_step_begin(h, d, stream);
}

int rae_dist_read_cost(rae_engine* h, double* cost_host) {
    if (!h || !cost_host) return fail(h, RAE_EINVAL, "rae_dist_read_cost: null argument");
    if (!h->gcost_pending) return fail(h, RAE_ENOTBOUND, "rae_dist_read_cost: no step with global_cost set has been issued");
    RAE_CUDA(h, cudaEventSynchronize(h->ev_gcost));
    if (peer_failed(h)) return RAE_ECUDA;
    *cost_host = *(volatile double*)h->gcost_pinned;
    if (*(volatile int32_t*)h->neg_err_pinned != 0) {
        *(volatile int32_t*)h->neg_err_pinned = 0;
        return fail(h, RAE_EINVAL, "the negatives passed for this batch are not the columns of the bound epoch negatives");
    }
    return RAE_OK;
}

int rae_dist_step_end(rae_engine* h, const rae_dist_step* d, void* stream) {
    if (!h || !d) return fail(h, RAE_EINVAL, "rae_dist_step_end: null argument");
    if (peer_failed(h)) return RAE_ECUDA;
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    const bool flags = d->flag_bufs != nullptr;
    const bool gcost = flags && d->global_cost != 0;
    FlagPtrs fp;
    if (h->reg) {
        // The regulariser's share of this rank, from the parameters before this step's update (every apply of the step is
        // behind barrier A below): its own W shard, and on rank 0 the decoder tensors, which every rank holds.  The cost is
        // re-run on the score partials of the local step; the rank-order sum of the local costs is then the global cost.
        if (d->w_rows < 0 || (d->w_rows > 0 && !d->W)) return fail(h, RAE_EINVAL, "rae_dist_step_end: bad W shard / w_rows");
        if ((rc = launch_cost(h, st, d->W, d->w_rows * h->K, d->rank == 0))) return rc;
        RAE_DMARK("reg_cost", st, 0);
    }
    if (gcost) {
        if (d->world > RAE_MAX_PEERS || d->rank < 0 || d->rank >= d->world) return fail(h, RAE_EINVAL, "rae_dist_step_end: bad world / rank");
        memset(&fp, 0, sizeof(fp));
        for (int r = 0; r < d->world; ++r) fp.p[r] = static_cast<int32_t*>(const_cast<void*>(d->flag_bufs[r]));
        // the local cost goes into the own flag buffer before the barrier publishes this rank's arrival
        if ((rc = rae_copy_cost(h, reinterpret_cast<double*>(fp.p[d->rank] + RAE_MAX_PEERS), stream))) return rc;
    }
    // (A) every rank has emitted its gradient rows and its dense gradient
    RAE_DMARK("local_step_done", st, 0);
    if (flags && (rc = launch_peer_barrier(h, d->flag_bufs, d->world, d->rank, st, 0))) return rc;
    RAE_DMARK("barrier_emitted", st, 0);
    if (gcost) {
        // the caller gets the global cost here, while the pulls below still run (rae_dist_read_cost)
        launch_pdl(k_global_cost, dim3(1), dim3(32), 0, st, fp, d->world, d->cost_dev, h->gcost_pinned);
        h->launches++;
        RAE_CUDA(h, cudaGetLastError());
        RAE_CUDA(h, cudaEventRecord(h->ev_gcost, st));
        h->gcost_pending = true;
    }
    const bool side = h->s1 != nullptr && h->s2 != nullptr && !h->profiling;
    if (side) {
        // the three owner-side pulls are independent: entity rows and biases on the side streams, W rows + the dense update here
        RAE_CUDA(h, cudaEventRecord(h->ev_dfork, st));
        RAE_CUDA(h, cudaStreamWaitEvent(h->s1, h->ev_dfork, 0));
        RAE_CUDA(h, cudaStreamWaitEvent(h->s2, h->ev_dfork, 0));
    }
    cudaStream_t sa = side ? h->s1 : st, sb = side ? h->s2 : st;
    // three independent branches: entity rows on s1, the dense update (reads nothing the applies write) and the biases on
    // s2, W rows here
    const bool peer_dense = flags && d->dense_bufs != nullptr;
    if (peer_dense) {
        // Wb is read by the NEXT step's encoder on this stream: applied here (K elements); the decoder tensors are next read
        // by the operand preparation, which runs on s2 itself
        if (side) {
            if ((rc = launch_dense_apply_peers(h, d->dense_bufs, d->world, st, 2))) return rc;
            if ((rc = launch_dense_apply_peers(h, d->dense_bufs, d->world, sb, 1))) return rc;
        } else if ((rc = launch_dense_apply_peers(h, d->dense_bufs, d->world, st, 0))) {
            return rc;
        }
        RAE_DMARK("dense_apply_peers", sb, side ? 2 : 0);
    }
    if (d->n_er > 0) {
        if ((rc = rae_pull_apply(h, d->A, d->accA, h->d, d->er_rows, d->er_off, d->e_src, d->e_slot, d->n_er, d->ga_bufs, d->world, sa))) return rc;
        RAE_DMARK("apply_A", sa, side ? 1 : 0);
        if ((rc = rae_pull_apply(h, d->Ab, d->accAb, 1, d->er_rows, d->er_off, d->e_src, d->e_slot, d->n_er, d->gab_bufs, d->world, sb))) return rc;
        RAE_DMARK("apply_Ab", sb, side ? 2 : 0);
    }
    if (h->reg) {
        // every row of the shard moves: the touched rows' contributions, then the regulariser, then the rule
        RAE_DMARK("w_shard_begin", st, 0);
        if ((rc = rae_shard_apply(h, d->W, d->accW, h->K, d->fr_rows, d->fr_off, d->f_src, d->f_slot, d->n_fr, d->gw_bufs, d->world,
                                  d->w_rows, stream))) return rc;
    } else if (d->n_fr > 0 && (rc = rae_pull_apply(h, d->W, d->accW, h->K, d->fr_rows, d->fr_off, d->f_src, d->f_slot, d->n_fr,
                                                   d->gw_bufs, d->world, stream))) {
        return rc;
    }
    RAE_DMARK("apply_W", st, 0);
    if (!peer_dense) {
        // the caller all-reduced the dense gradient itself - possibly on another stream, beside the barrier and the applies
        // above (rae_dist_set_dense_wait): the dense update is the first thing here that needs the sum
        if (h->dense_wait != nullptr) {
            RAE_CUDA(h, cudaStreamWaitEvent(st, (cudaEvent_t)h->dense_wait, 0));
            h->dense_wait = nullptr;
        }
        if ((rc = rae_train_step_end(h, stream))) return rc;
    }
    if (side && flags) {
        // Split tail.  The next step's first consumers of the tables are the W fetch and the encoder on this stream: they
        // need every owner's W apply only.  The entity rows are fetched on s1, so "every owner has applied A, Ab and the
        // dense update" is a second barrier sequence (kind 1) on s1, behind which s1's next work (the entity fetch of
        // the next step) is ordered by the stream itself; this stream meets it where the decoder first reads A
        // (pending_wait).  The applies of A / Ab / the dense parameters thus run beside the next step's head.
        RAE_CUDA(h, cudaEventRecord(h->ev_join2, h->s2));
        RAE_CUDA(h, cudaStreamWaitEvent(h->s1, h->ev_join2, 0));
        if ((rc = launch_peer_barrier(h, d->flag_bufs, d->world, d->rank, h->s1, 1))) return rc;
        RAE_DMARK("barrier_rest_applied", h->s1, 1);
        if ((rc = launch_peer_barrier(h, d->flag_bufs, d->world, d->rank, st, 0))) return rc;
        RAE_DMARK("barrier_w_applied", st, 0);
    } else {
        if (side) {
            RAE_CUDA(h, cudaEventRecord(h->ev_join1, h->s1));
            RAE_CUDA(h, cudaEventRecord(h->ev_join2, h->s2));
            RAE_CUDA(h, cudaStreamWaitEvent(st, h->ev_join1, 0));
            RAE_CUDA(h, cudaStreamWaitEvent(st, h->ev_join2, 0));
        }
        // (B) every owner has applied: the next step may fetch, the compact gradient buffers may be overwritten
        if (flags && (rc = launch_peer_barrier(h, d->flag_bufs, d->world, d->rank, st, 0))) return rc;
        RAE_DMARK("barrier_applied", st, 0);
    }
    h->push.f_ids = nullptr;        // valid for the step whose descriptor set them only
    h->push.e_ids = nullptr;
    if (d->cost_dev && !gcost) return rae_copy_cost(h, d->cost_dev, stream);
    return RAE_OK;
}

}  // extern "C"
