// Kernel 1: encoder.  One warp per example: gather-sum of the example's W rows from the binary CSR batch, + Wb,
// fused K-way softmax, entropy (training), argmax (labelling) or the k best relations (top-k labelling).
//   reference: sparse.dot(x_feats, W) + Wb ; T.nnet.softmax ; T.argmax   learning/models/encoders/RelationClassifier.py:35-36,45-47
//              entropy = alpha * -sum(log(q) * q)                       learning/OieModel.py:81
// HBM-bound: nnz*K*4 bytes of W rows per batch; every lane keeps UNROLL x KT independent row loads in flight.
#include "rae_common.cuh"
#include "rae_internal.h"

namespace rae {

// Where row f of W is: a compile-time policy of the encoder bodies below.  The warp of an example reads its feature ids 32
// at a time (one per lane), turns each into a lookup key, and broadcasts the key of the row it loads next.
//   DenseTable : one table, row f at W + f*K (the engine's bound W: the single-GPU step and labelling, the compact tables of
//                the sharded step).  int example index; probs are always written.
//   ShardTables: W row-sharded over `world` ranks, row f at p[f % world] + (f / world)*K (rae_label_shards).  The <= 16
//                peer pointers are copied into shared memory at kernel entry, so the lookup never indexes the parameter
//                space dynamically (no local copy, no stack frame); the key is the row pointer itself.  int64 example
//                index (a whole split per launch); q == NULL skips the probability stores.
struct DenseTable {
    typedef const float* __restrict__ Arg;
    typedef int Index;
    typedef int Key;
    static constexpr bool kOptionalQ = false;
    const float* W;
    __device__ __forceinline__ explicit DenseTable(const float* w) : W(w) {}
    static __device__ __forceinline__ Index example() { return (blockIdx.x * blockDim.x + threadIdx.x) >> 5; }
    __device__ __forceinline__ Key key(int f, int) const { return f; }
    static __device__ __forceinline__ Key shfl(Key k, int src) { return __shfl_sync(kFull, k, src); }
    __device__ __forceinline__ const float* row(Key f, int K) const { return W + (size_t)f * K; }
};

struct ShardPtrs {
    const float* p[RAE_MAX_PEERS];
    int world;
};

struct ShardTables {
    typedef ShardPtrs Arg;
    typedef int64_t Index;
    typedef const float* Key;
    static constexpr bool kOptionalQ = true;
    const float* const* tab;       // shared memory
    int world;
    // every thread of the CTA must construct it (one barrier) before any thread leaves
    __device__ __forceinline__ explicit ShardTables(const ShardPtrs& a) : world(a.world) {
        __shared__ const float* s_tab[RAE_MAX_PEERS];
        if (threadIdx.x == 0) {
#pragma unroll
            for (int r = 0; r < RAE_MAX_PEERS; ++r) s_tab[r] = a.p[r];
        }
        __syncthreads();
        tab = s_tab;
    }
    static __device__ __forceinline__ Index example() {
        return (Index)(((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    }
    __device__ __forceinline__ Key key(int f, int K) const { return tab[f % world] + (size_t)(f / world) * K; }
    static __device__ __forceinline__ Key shfl(Key k, int src) {
        return reinterpret_cast<Key>(__shfl_sync(kFull, reinterpret_cast<unsigned long long>(k), src));
    }
    __device__ __forceinline__ const float* row(Key k, int) const { return k; }
};

// The warp's row again, read from the special registers at the store: the gather loop of the scalar KT = 8 body keeps
// every register busy, and a row index kept live across it spills.
__device__ __forceinline__ size_t row_of_warp() {
    unsigned cta, tid, ntid;
    asm volatile("mov.u32 %0, %%ctaid.x;" : "=r"(cta));
    asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid));
    asm volatile("mov.u32 %0, %%ntid.x;" : "=r"(ntid));
    return ((size_t)cta * ntid + tid) >> 5;
}

// Top-k output (TopK = true, rae_label_topk): the k best relations of the warp's row b, by score descending and then
// relation id ascending (the first-max rule of the labels, extended), into ids[b*k ..] and, when q is not NULL, their softmax
// probabilities expf(z - lse) into q[b*k ..].  e[s] is the score of relation id(s) of this lane: lane + 32s on the scalar
// path, 4(lane + 32(s/4)) + s%4 on the 16-byte path.  Each lane keeps its best score not taken yet; k rounds of butterfly
// arg-max pick the winner, and only the lane that owns it marks it in its bitmask and rescans.  Lane j keeps the winner of
// round j, so a row's k results leave in one coalesced store.  Everything stays in registers: e is only indexed by
// unrolled (compile-time) s, and slots past K start out taken so that the rescan needs no relation ids.
template <bool V4>
__device__ __forceinline__ int topk_id(int lane, int s) { return V4 ? 4 * (lane + 32 * (s >> 2)) + (s & 3) : lane + 32 * s; }

template <int N, bool V4>
__device__ __forceinline__ void best_untaken(const float (&e)[N], int lane, unsigned taken, float& bv, int& bi) {
    bv = -INFINITY;
    int bs = -1;
#pragma unroll
    for (int s = 0; s < N; ++s)
        if (!((taken >> s) & 1u) && e[s] > bv) { bv = e[s]; bs = s; }       // ascending id: first max wins
    bi = bs < 0 ? 0x7fffffff : topk_id<V4>(lane, bs);
}

template <int N, bool V4>
__device__ __forceinline__ void store_topk(const float (&e)[N], int K, int lane, float lse, size_t b, int k,
                                           int32_t* __restrict__ ids, float* __restrict__ q) {
    static_assert(N <= 32, "one bit per owned score");
    unsigned taken = 0u;
#pragma unroll
    for (int s = 0; s < N; ++s)
        if (topk_id<V4>(lane, s) >= K) taken |= 1u << s;
    float bv;
    int bi;
    best_untaken<N, V4>(e, lane, taken, bv, bi);
    float my_v = 0.f;
    int my_i = 0;
    for (int j = 0; j < k; ++j) {
        float wv = bv;
        int wi = bi;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(kFull, wv, o);
            const int oi = __shfl_xor_sync(kFull, wi, o);
            if (ov > wv || (ov == wv && oi < wi)) { wv = ov; wi = oi; }
        }
        if (lane == j) { my_v = wv; my_i = wi; }
        const int owner = V4 ? (wi >> 2) & 31 : wi & 31;
        if (wi < K && owner == lane) {
            taken |= 1u << (V4 ? ((wi >> 7) << 2) | (wi & 3) : wi >> 5);
            best_untaken<N, V4>(e, lane, taken, bv, bi);
        }
    }
    if (lane < k) {
        ids[b * k + lane] = my_i;
        if (q != nullptr) q[b * k + lane] = expf(my_v - lse);
    }
}

template <int KT, class Rows = DenseTable, bool TopK = false>
__global__ void __launch_bounds__(256) k_encoder_forward(const int32_t* __restrict__ indptr,
                                                         const int32_t* __restrict__ indices,
                                                         typename Rows::Arg W, const float* __restrict__ Wb,
                                                         typename Rows::Index B, int K, float alpha, float* __restrict__ q,
                                                         float* __restrict__ logq, float* __restrict__ sc_ent,
                                                         int sc_stride, int64_t* __restrict__ labels, int topk,
                                                         int32_t* __restrict__ topk_ids) {
    const Rows rows(W);
    const int lane = threadIdx.x & 31;
    const typename Rows::Index b = Rows::example();
    if (b >= B) return;
    const int beg = indptr[b], end = indptr[b + 1];
    float z[KT];
#pragma unroll
    for (int t = 0; t < KT; ++t) {
        int k = lane + 32 * t;
        z[t] = (k < K) ? Wb[k] : 0.f;
    }
    constexpr int UNROLL = (KT <= 4) ? 8 : 2;
    for (int base = beg; base < end; base += 32) {
        const typename Rows::Key mine = rows.key((base + lane < end) ? indices[base + lane] : 0, K);
        const int cnt = min(32, end - base);
        for (int t0 = 0; t0 < cnt; t0 += UNROLL) {
            float v[UNROLL][KT];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const typename Rows::Key f = Rows::shfl(mine, (t0 + u) & 31);
                const bool ok = (t0 + u) < cnt;
                const float* row = rows.row(f, K);
#pragma unroll
                for (int t = 0; t < KT; ++t) {
                    int k = lane + 32 * t;
                    v[u][t] = (ok && k < K) ? ld_nc(row + k) : 0.f;
                }
            }
            // fixed summation order (feature order of the CSR row) -> run-to-run reproducible
#pragma unroll
            for (int u = 0; u < UNROLL; ++u)
#pragma unroll
                for (int t = 0; t < KT; ++t) z[t] += v[u][t];
        }
    }
    // softmax over K
    float m = -INFINITY;
    int arg = 0x7fffffff;
#pragma unroll
    for (int t = 0; t < KT; ++t) {
        int k = lane + 32 * t;
        if (k < K && z[t] > m) { m = z[t]; arg = k; }   // ascending k per lane: first max wins
    }
    if (!TopK && labels != nullptr) {
        float bm = m;
        int ba = arg;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            float om = __shfl_xor_sync(kFull, bm, o);
            int oa = __shfl_xor_sync(kFull, ba, o);
            if (om > bm || (om == bm && oa < ba)) { bm = om; ba = oa; }
        }
        if (lane == 0) labels[b] = (int64_t)ba;
    }
    m = warp_max(m);
    float s = 0.f;
#pragma unroll
    for (int t = 0; t < KT; ++t) {
        int k = lane + 32 * t;
        if (k < K) s += expf(z[t] - m);
    }
    s = warp_sum(s);
    const float lse = m + logf(s);
    if (TopK) {
        store_topk<KT, false>(z, K, lane, lse, row_of_warp(), topk, topk_ids, q);
        return;
    }
    float ent = 0.f;
    const bool store_q = !Rows::kOptionalQ || q != nullptr;
#pragma unroll
    for (int t = 0; t < KT; ++t) {
        int k = lane + 32 * t;
        if (k < K) {
            float lq = z[t] - lse;
            float p = expf(lq);
            if (store_q) q[(size_t)b * K + k] = p;
            if (logq != nullptr) logq[(size_t)b * K + k] = lq;
            ent -= p * lq;
        }
    }
    if (sc_ent != nullptr) {
        ent = warp_sum(ent);
        if (lane == 0) sc_ent[(size_t)b * sc_stride] = alpha * ent;
    }
}

// K % 4 == 0: every lane owns QT float4 (16-byte row loads, one instruction per W row for K <= 128) and UNROLL rows
// are in flight together.
template <int QT, class Rows = DenseTable, bool TopK = false>
__global__ void __launch_bounds__(256) k_encoder_forward_v4(const int32_t* __restrict__ indptr,
                                                            const int32_t* __restrict__ indices,
                                                            typename Rows::Arg W, const float* __restrict__ Wb,
                                                            typename Rows::Index B, int K, float alpha, float* __restrict__ q,
                                                            float* __restrict__ logq, float* __restrict__ sc_ent,
                                                            int sc_stride, int64_t* __restrict__ labels, int topk,
                                                            int32_t* __restrict__ topk_ids) {
    pdl_enter();
    const Rows rows(W);
    const int lane = threadIdx.x & 31;
    const typename Rows::Index b = Rows::example();
    if (b >= B) return;
    const int beg = indptr[b], end = indptr[b + 1];
    const int nq = K >> 2;
    float4 z[QT];
#pragma unroll
    for (int t = 0; t < QT; ++t) {
        const int qi = lane + 32 * t;
        z[t] = (qi < nq) ? __ldg(reinterpret_cast<const float4*>(Wb) + qi) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    constexpr int UNROLL = (QT == 1) ? 16 : (QT == 2 ? 8 : 4);
    for (int base = beg; base < end; base += 32) {
        const typename Rows::Key mine = rows.key((base + lane < end) ? indices[base + lane] : 0, K);
        const int cnt = min(32, end - base);
        for (int t0 = 0; t0 < cnt; t0 += UNROLL) {
            float4 v[UNROLL][QT];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const typename Rows::Key f = Rows::shfl(mine, (t0 + u) & 31);
                const bool ok = (t0 + u) < cnt;
                const float4* row = reinterpret_cast<const float4*>(rows.row(f, K));
#pragma unroll
                for (int t = 0; t < QT; ++t) {
                    const int qi = lane + 32 * t;
                    v[u][t] = (ok && qi < nq) ? __ldg(row + qi) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
            // fixed summation order (feature order of the CSR row) -> run-to-run reproducible
#pragma unroll
            for (int u = 0; u < UNROLL; ++u)
#pragma unroll
                for (int t = 0; t < QT; ++t) {
                    z[t].x += v[u][t].x; z[t].y += v[u][t].y; z[t].z += v[u][t].z; z[t].w += v[u][t].w;
                }
        }
    }
    float m = -INFINITY;
    int arg = 0x7fffffff;
#pragma unroll
    for (int t = 0; t < QT; ++t) {
        const int qi = lane + 32 * t;
        if (qi < nq) {
            const float e[4] = {z[t].x, z[t].y, z[t].z, z[t].w};
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (e[c] > m) { m = e[c]; arg = 4 * qi + c; }     // ascending k per lane: first max wins
        }
    }
    if (!TopK && labels != nullptr) {
        float bm = m;
        int ba = arg;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float om = __shfl_xor_sync(kFull, bm, o);
            const int oa = __shfl_xor_sync(kFull, ba, o);
            if (om > bm || (om == bm && oa < ba)) { bm = om; ba = oa; }
        }
        if (lane == 0) labels[b] = (int64_t)ba;
    }
    m = warp_max(m);
    float s = 0.f;
#pragma unroll
    for (int t = 0; t < QT; ++t) {
        const int qi = lane + 32 * t;
        if (qi < nq) s += (expf(z[t].x - m) + expf(z[t].y - m)) + (expf(z[t].z - m) + expf(z[t].w - m));
    }
    s = warp_sum(s);
    const float lse = m + logf(s);
    if (TopK) {
        float e[4 * QT];
#pragma unroll
        for (int t = 0; t < QT; ++t) {
            e[4 * t] = z[t].x; e[4 * t + 1] = z[t].y; e[4 * t + 2] = z[t].z; e[4 * t + 3] = z[t].w;
        }
        store_topk<4 * QT, true>(e, K, lane, lse, row_of_warp(), topk, topk_ids, q);
        return;
    }
    float ent = 0.f;
    const bool store_q = !Rows::kOptionalQ || q != nullptr;
#pragma unroll
    for (int t = 0; t < QT; ++t) {
        const int qi = lane + 32 * t;
        if (qi < nq) {
            const float4 lq = make_float4(z[t].x - lse, z[t].y - lse, z[t].z - lse, z[t].w - lse);
            const float4 pr = make_float4(expf(lq.x), expf(lq.y), expf(lq.z), expf(lq.w));
            if (store_q) reinterpret_cast<float4*>(q + (size_t)b * K)[qi] = pr;
            if (logq != nullptr) reinterpret_cast<float4*>(logq + (size_t)b * K)[qi] = lq;
            ent -= (pr.x * lq.x + pr.y * lq.y) + (pr.z * lq.z + pr.w * lq.w);
        }
    }
    if (sc_ent != nullptr) {
        ent = warp_sum(ent);
        if (lane == 0) sc_ent[(size_t)b * sc_stride] = alpha * ent;
    }
}

namespace {

// One launch of the encoder over n examples with the W lookup of policy Rows.  w_aligned: every row of W starts on 16 bytes
// when K % 4 == 0 (the 16-byte path also needs Wb, q and log q aligned; the top-k output stores q one float per lane, so
// there only Wb counts and the path is the one rae_label_shards takes with probs NULL or aligned).
template <class Rows, bool TopK = false>
int launch_encoder(rae_engine* h, const int32_t* indptr, const int32_t* indices, typename Rows::Arg W, bool w_aligned,
                   typename Rows::Index n, float* q, float* logq, float* sc_ent, int64_t* labels, cudaStream_t st,
                   int topk = 0, int32_t* topk_ids = nullptr) {
    const int K = h->K;
    const int threads = 256;
    const int64_t blocks64 = ((int64_t)n * 32 + threads - 1) / threads;
    if (blocks64 > 0x7fffffff) return fail(h, RAE_EINVAL, "encoder: %lld rows are too many for one launch", (long long)n);
    const int blocks = (int)blocks64;
    const float* Wb = h->P[RAE_P_WB];
    const float alpha = (float)h->cfg.alpha;
    const int kt = (K + 31) / 32;
    // 16-byte path: rows of W, q and log q must be 16-byte aligned (K % 4 == 0 and aligned base pointers)
    const uintptr_t outs = TopK ? 0 : ((uintptr_t)q | (uintptr_t)logq);
    const bool vec = (K & 3) == 0 && K <= 512 && w_aligned && (((uintptr_t)Wb | outs) & 15) == 0;
    if (vec) {
        const int qt = (K / 4 + 31) / 32;
#define RAE_ENC4(QT)                                                                                                 \
    launch_pdl(k_encoder_forward_v4<QT, Rows, TopK>, dim3(blocks), dim3(threads), 0, st, indptr, indices, W, Wb, n, K, alpha, q, logq, \
               sc_ent, SC_N, labels, topk, topk_ids)
        if (qt <= 1) RAE_ENC4(1);
        else if (qt <= 2) RAE_ENC4(2);
        else RAE_ENC4(4);
#undef RAE_ENC4
        h->launches++;
        RAE_CUDA(h, cudaGetLastError());
        return RAE_OK;
    }
#define RAE_ENC(KT)                                                                                                  \
    k_encoder_forward<KT, Rows, TopK><<<blocks, threads, 0, st>>>(indptr, indices, W, Wb, n, K, alpha, q, logq, sc_ent, SC_N, labels, \
                                                                 topk, topk_ids)
    if (kt <= 1) RAE_ENC(1);
    else if (kt <= 2) RAE_ENC(2);
    else if (kt <= 4) RAE_ENC(4);
    else if (kt <= 8) RAE_ENC(8);
    else if (kt <= 16) RAE_ENC(16);
    else if (kt <= 32) RAE_ENC(32);
    else return fail(h, RAE_EINVAL, "K=%d > 1024 is not supported by the encoder kernel", K);
#undef RAE_ENC
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

// the peer-pointer table of a row-sharded W (rae_label_shards, rae_label_topk); aligned: every shard starts on 16 bytes
int shard_ptrs(rae_engine* h, const char* who, const void* const* w_shards, int world, ShardPtrs& sp, bool& aligned) {
    if (world < 1 || world > RAE_MAX_PEERS) return fail(h, RAE_EINVAL, "%s: world %d out of range [1, %d]", who, world, RAE_MAX_PEERS);
    sp = ShardPtrs{};
    sp.world = world;
    aligned = true;
    for (int r = 0; r < world; ++r) {
        if (!w_shards[r]) return fail(h, RAE_EINVAL, "%s: null W shard for rank %d", who, r);
        sp.p[r] = static_cast<const float*>(w_shards[r]);
        aligned = aligned && ((uintptr_t)sp.p[r] & 15) == 0;
    }
    return RAE_OK;
}

}  // namespace

int launch_encoder_forward(rae_engine* h, const int32_t* indptr, const int32_t* indices, int B, float* q, float* logq,
                           float* sc_ent, int64_t* labels, cudaStream_t st) {
    const float* W = h->P[RAE_P_W];
    return launch_encoder<DenseTable>(h, indptr, indices, W, ((uintptr_t)W & 15) == 0, B, q, logq, sc_ent, labels, st);
}

int launch_label_shards(rae_engine* h, const void* const* w_shards, int world, const int32_t* indptr, const int32_t* indices,
                        int64_t n_rows, int64_t* labels, float* probs, cudaStream_t st) {
    ShardPtrs sp;
    bool aligned;
    if (int rc = shard_ptrs(h, "rae_label_shards", w_shards, world, sp, aligned)) return rc;
    if (n_rows == 0) return RAE_OK;
    return launch_encoder<ShardTables>(h, indptr, indices, sp, aligned, n_rows, probs, nullptr, nullptr, labels, st);
}

int launch_label_topk(rae_engine* h, const void* const* w_shards, int world, const int32_t* indptr, const int32_t* indices,
                      int64_t n_rows, int k, int32_t* ids, float* probs, cudaStream_t st) {
    if (k < 1 || k > h->K || k > RAE_MAX_TOPK)
        return fail(h, RAE_EINVAL, "rae_label_topk: k = %d outside [1, min(K = %d, %d)]", k, h->K, RAE_MAX_TOPK);
    ShardPtrs sp;
    bool aligned;
    if (int rc = shard_ptrs(h, "rae_label_topk", w_shards, world, sp, aligned)) return rc;
    if (n_rows == 0) return RAE_OK;
    return launch_encoder<ShardTables, true>(h, indptr, indices, sp, aligned, n_rows, probs, nullptr, nullptr, nullptr, st, k, ids);
}

}  // namespace rae
