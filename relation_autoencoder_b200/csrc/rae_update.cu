// Kernel 3: deterministic segmented scatter + sparse-row AdaGrad, dense-parameter update, cost reduction.
//
//   reference: T.grad(cost, params) + AdaGrad.update / SGD.update   learning/Optimizers.py:18-33,38-52
//              (Theano accumulates duplicate rows through AdvancedIncSubtensor1 BEFORE the optimiser squares the
//               gradient, so duplicates must be summed first: sort-by-row, segment-reduce in sorted order, then ONE
//               read-modify-write per unique row.  No atomics in the data path -> bitwise reproducible.)
//              regulariser  learning/OieModel.py:54-62, learning/OieInduction.py:131-135
//
// Rows with zero gradient are fixed points of Optimizers.py:29-32 (acc' = acc, p' = p - lr*0/(sqrt(acc)+1e-6) = p), so
// visiting only the touched rows is exactly the reference's dense sweep when lambda1 = lambda2 = 0.
#include <algorithm>
#include <cub/cub.cuh>

#include "rae_common.cuh"
#include "rae_internal.h"

namespace rae {

namespace {

__global__ void k_entity_keys(const int32_t* __restrict__ a1, const int32_t* __restrict__ a2,
                              const int32_t* __restrict__ neg1, const int32_t* __restrict__ neg2, int64_t neg_ld, int B,
                              int S, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    pdl_enter();
    // occurrence id o = slot*B + b ; slot 0: args1, 1: args2, 2+s: neg1[s], 2+S+s: neg2[s]
    const int n = (2 + 2 * S) * B;
    for (int o = blockIdx.x * blockDim.x + threadIdx.x; o < n; o += gridDim.x * blockDim.x) {
        const int slot = o / B, b = o - slot * B;
        int row;
        if (slot == 0) row = a1[b];
        else if (slot == 1) row = a2[b];
        else if (slot < 2 + S) row = neg1[(size_t)(slot - 2) * neg_ld + b];
        else row = neg2[(size_t)(slot - 2 - S) * neg_ld + b];
        keys[o] = (uint32_t)row;
        vals[o] = (uint32_t)o;
    }
}

__global__ void k_feature_keys(const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices, int B,
                               uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    // one warp per example: key = feature id, value = example index within the batch
    const int lane = threadIdx.x & 31;
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= B) return;
    const int base = indptr[0];
    for (int p = indptr[b] + lane; p < indptr[b + 1]; p += 32) {
        keys[p - base] = (uint32_t)indices[p];
        vals[p - base] = (uint32_t)b;
    }
}

// ---- segment boundaries (introspection / parity tests only: the update kernels work from the sorted keys) ----
__global__ void k_flag_heads(const uint32_t* __restrict__ keys_s, int n, int32_t* __restrict__ flags) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        flags[i] = (i == 0 || keys_s[i] != keys_s[i - 1]) ? 1 : 0;
}

__global__ void k_scatter_heads(const int32_t* __restrict__ flags, const int32_t* __restrict__ pos, int n,
                                int32_t* __restrict__ seg_start, int32_t* __restrict__ n_seg) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (flags[i]) seg_start[pos[i]] = i;
        if (i == n - 1) {
            const int ns = pos[i] + flags[i];
            seg_start[ns] = n;
            *n_seg = ns;
        }
    }
    if (n == 0 && blockIdx.x == 0 && threadIdx.x == 0) { seg_start[0] = 0; *n_seg = 0; }
}

// integer count of distinct keys (statistics only; integer atomics do not affect any result)
__global__ void k_count_heads(const uint32_t* __restrict__ keys_s, int n, int32_t* __restrict__ out) {
    int c = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        c += (i == 0 || keys_s[i] != keys_s[i - 1]) ? 1 : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(kFull, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

// ---- segmented reduction of sorted occurrences, balanced over warps -------------------------------------------------
// Level 1 (k_rows_chunk): one warp per chunk of 32 sorted positions.
//   phase 1  lanes = COLUMNS (one float4 each, tiles of 128 columns): the chunk's payload rows are streamed 8 at a time
//            (coalesced row reads, all 8 in flight) and accumulated in position order; at every run boundary - warp-uniform,
//            taken from the ballot of the keys - the finished run's sum is parked in the warp's shared-memory slab;
//   phase 2  the runs are visited 4 at a time: table + accumulator rows of 4 runs are in flight together, the optimiser
//            rule is applied once per row and the row is written back coalesced (or the reduced gradient row is emitted).
//   A segment that spans exactly TWO chunks (about every second chunk boundary cuts one) is ABSORBED by the chunk it starts
//   in: that warp reads on through the segment's positions in the next chunk (at most 32 more) and the next chunk skips
//   them - both sides take the decision from the sorted keys alone.  Only segments spanning three or more chunks (rows with
//   more than 32 occurrences) park their per-chunk partial rows in scratch slot 2c / 2c+1.
// Level 2 (k_*_long2): the CTA of the chunk in which such a long segment STARTS finds its extent, sums the partial rows
// in chunk order and applies the update.  Hot rows (Zipf) are thereby spread over many warps; the summation order is a
// fixed function of the sorted layout -> bitwise reproducible.  No atomics.

// where an emitted (reduced) gradient row goes: the local buffer, or - gradient push - the owner's receive buffer
struct PushTo { float* const* base; float* const* bias; const int32_t* ids; int world; long long rowoff; };
__device__ __forceinline__ float* emit_row(const PushTo& t, float* local, uint32_t row, int width) {
    if (t.base == nullptr) return local + (size_t)row * width;
    return t.base[t.ids[row] % t.world] + ((size_t)t.rowoff + row) * width;
}
__device__ __forceinline__ float* emit_bias(const PushTo& t, float* local, uint32_t row) {
    if (t.bias == nullptr) return local + row;
    return t.bias[t.ids[row] % t.world] + (size_t)t.rowoff + row;
}

// arguments of both levels.  MODE 0: feature rows of W (payload = dz).  MODE 1: entity rows of A and, through the
// bias partial at column dp of every partial slot, of Ab.
struct RowsArgs {
    PushTo push;
    const uint32_t* keys_s; const uint32_t* vals_s; int n;
    const float* payload;      // W: dz [B,K] ; entity: ev
    int width;                 // floats per table row (K or d)
    int pitch;                 // floats per partial slot in `part` (W: K ; entity: dp + 4, bias partial at [dp])
    float* table; float* acc; float* g_out; float* part;
    float lr; int adagrad, emit, apply;
    // entity rows only
    int B, S, dp; const float* sc; const float* gn1; const float* gn2;
    float* tableb; float* accb; float* gb_out;
};

// A segment that spans exactly two chunks is absorbed by level 1 for feature rows only: measured, the probes and the
// tail pass cost the entity kernel more than level 2 saves.
template <int MODE>
constexpr bool kAbsorbs = MODE == 0;

// does a multi-chunk segment start in chunk c?  returns its first partial slot (or -1) and its row
__device__ __forceinline__ int long_segment_start(const uint32_t* __restrict__ keys_s, int n, int c, uint32_t* row, bool absorbing) {
    const int p0 = c << 5;
    const int cnt = min(32, n - p0);
    if (p0 + cnt >= n) return -1;
    const uint32_t keyl = keys_s[p0 + cnt - 1];
    if (keys_s[p0 + cnt] != keyl) return -1;          // last run ends with the chunk
    *row = keyl;
    const bool starts_here = !(keys_s[p0] == keyl && p0 > 0 && keys_s[p0 - 1] == keyl);
    if (absorbing && starts_here && (p0 + 64 >= n || keys_s[p0 + 64] != keyl)) return -1;     // spans two chunks: absorbed by level 1
    if (keys_s[p0] == keyl) {                          // run covers the chunk from its first position
        if (p0 > 0 && keys_s[p0 - 1] == keyl) return -1;   // ... and continues an earlier chunk: not the start
        return 2 * c;
    }
    return 2 * c + 1;
}

struct ScanCtx {
    unsigned same;      // bit i: lane - 2^i belongs to the same run
    bool live, is_last, partial;
    int slot;           // partial slot 2c or 2c+1 (valid on is_last && partial)
    uint32_t key;
};

__device__ __forceinline__ ScanCtx scan_ctx(const uint32_t* __restrict__ keys_s, int n, int c, int lane) {
    ScanCtx s;
    const int p0 = c << 5;
    const int cnt = min(32, n - p0);
    s.live = lane < cnt;
    s.key = s.live ? keys_s[p0 + lane] : 0xffffffffu;
    s.same = 0u;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        const uint32_t up = __shfl_up_sync(kFull, s.key, 1 << i);
        if (s.live && lane >= (1 << i) && up == s.key) s.same |= 1u << i;
    }
    const uint32_t dn = __shfl_down_sync(kFull, s.key, 1);
    s.is_last = s.live && (lane == cnt - 1 || dn != s.key);
    const unsigned heads = __ballot_sync(kFull, s.live && !(s.same & 1u));
    const int rs = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));     // first lane of this lane's run
    const uint32_t key0 = __shfl_sync(kFull, s.key, 0), keyl = __shfl_sync(kFull, s.key, cnt - 1);
    const bool cont_prev = p0 > 0 && keys_s[p0 - 1] == key0;
    const bool cont_next = p0 + cnt < n && keys_s[p0 + cnt] == keyl;
    s.partial = (rs == 0 && cont_prev) || (lane == cnt - 1 && cont_next);
    s.slot = 2 * c + (rs == 0 ? 0 : 1);
    return s;
}

__device__ __forceinline__ float seg_scan(float v, unsigned same) {
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        const float t = __shfl_up_sync(kFull, v, 1 << i);
        if (same & (1u << i)) v += t;
    }
    return v;
}

// columns q .. q+3 of a row (p points at column q < width): one 16-byte access when VEC, else the columns below `width`
// one by one (the others read as 0 / are not written).  Plain loads on purpose: the row-update kernels issue a whole
// batch of them before the first add, so a warp waits one memory latency per batch, not one per row.
template <bool VEC>
__device__ __forceinline__ float4 ld4(const float* p, int q, int width) {
    if (VEC) return *reinterpret_cast<const float4*>(p);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    v.x = p[0];
    if (q + 1 < width) v.y = p[1];
    if (q + 2 < width) v.z = p[2];
    if (q + 3 < width) v.w = p[3];
    return v;
}
template <bool VEC>
__device__ __forceinline__ void st4(float* p, const float4& v, int q, int width) {
    if (VEC) {
        *reinterpret_cast<float4*>(p) = v;
        return;
    }
    p[0] = v.x;
    if (q + 1 < width) p[1] = v.y;
    if (q + 2 < width) p[2] = v.z;
    if (q + 3 < width) p[3] = v.w;
}

constexpr int ROWS_TILE = 128;     // columns per pass (one float4 per lane)

// MODE 0: feature rows (payload row = dz[val,:], coefficient 1).  MODE 1: entity rows (occurrence decode, coefficient,
// bias scalar).  VEC: the table rows are 16-byte aligned (width % 4 == 0).
template <int MODE, bool VEC>
__global__ void __launch_bounds__(256) k_rows_chunk(RowsArgs p, int slab_cols) {
    pdl_enter();
    extern __shared__ float4 slab4[];                      // [warps of the CTA][32 runs][slab_cols / 4]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nw = (gridDim.x * blockDim.x) >> 5;
    const int nchunks = (p.n + 31) >> 5;
    const int sq = slab_cols >> 2;
    float4* S = slab4 + (size_t)warp * 32 * sq;
    for (int c = gw; c < nchunks; c += nw) {
        const ScanCtx s = scan_ctx(p.keys_s, p.n, c, lane);
        const int p0 = c << 5;
        const int cnt = min(32, p.n - p0);
        const uint32_t mine = s.live ? p.vals_s[p0 + lane] : 0u;
        const unsigned heads = __ballot_sync(kFull, s.live && !(s.same & 1u));
        const int nr = __popc(heads);
        // chunk-level continuation flags (recomputed from lane-local data of scan_ctx: partial is set on the last lane of a
        // partial run; the run-level predicate is rebuilt below from the first / last run)
        const uint32_t key0 = __shfl_sync(kFull, s.key, 0), keyl = __shfl_sync(kFull, s.key, cnt - 1);
        const bool cont_prev = p0 > 0 && p.keys_s[p0 - 1] == key0;
        const bool cont_next = p0 + cnt < p.n && p.keys_s[p0 + cnt] == keyl;
        // two-chunk segments: absorbed by their first chunk, skipped by the second (header comment); cnt == 32 whenever
        // the chunk has a successor
        const bool single = nr == 1;
        bool absorb = false, skip = false;
        if (kAbsorbs<MODE>) {
            if (cont_next && !(single && cont_prev)) absorb = p0 + 64 >= p.n || p.keys_s[p0 + 64] != keyl;
            if (cont_prev && !(single && cont_next)) skip = p.keys_s[p0 - 32] != key0 || p0 == 32 || p.keys_s[p0 - 33] != key0;
        }
        const int skipn = skip ? ((heads & ~1u) ? (__ffs(heads & ~1u) - 1) : cnt) : 0;     // positions of the skipped first run
        int ext = 0;                    // positions of the absorbed tail in the next chunk
        uint32_t mine_x = 0u;
        if (absorb) {
            const int px = p0 + 32 + lane;
            const bool same = px < p.n && p.keys_s[px] == keyl;
            const unsigned bal = __ballot_sync(kFull, same);
            ext = (bal == 0xffffffffu) ? 32 : (__ffs(~bal) - 1);
            if (lane < ext) mine_x = p.vals_s[px];
        }
        // occurrence -> payload row offset, coefficient, bias contribution
        auto decode = [&](uint32_t occ, bool live, int& off, float& coef, float& bias) {
            coef = 1.f; bias = 0.f;
            if (MODE == 0) {
                off = (int)occ * p.width;
            } else {
                const int slot_m = (int)(occ / (uint32_t)p.B);
                const int b_m = (int)(occ - (uint32_t)slot_m * (uint32_t)p.B);
                int vs;
                if (slot_m == 0) { vs = E_GA1; coef = 1.f; bias = p.sc[(size_t)b_m * SC_N + SC_GU1]; }
                else if (slot_m == 1) { vs = E_GA2; coef = 1.f; bias = p.sc[(size_t)b_m * SC_N + SC_GU2]; }
                else if (slot_m < 2 + p.S) { vs = E_V1; coef = p.gn1[(size_t)(slot_m - 2) * p.B + b_m]; bias = coef; }
                else { vs = E_V2; coef = p.gn2[(size_t)(slot_m - 2 - p.S) * p.B + b_m]; bias = coef; }
                if (!live) { coef = 0.f; bias = 0.f; }
                off = (b_m * E_NV + vs) * p.dp;
            }
        };
        int off_m, off_x = 0;
        float coef_m, coef_x = 0.f, bias_m, bias_x = 0.f;
        decode(mine, s.live, off_m, coef_m, bias_m);
        if (absorb) decode(mine_x, lane < ext, off_x, coef_x, bias_x);
        if (MODE == 1) {
            // bias column: lane = position, segmented scan, the last lane of a run applies / parks it
            float gb = seg_scan(bias_m, s.same);
            if (absorb) {
                // the absorbed tail's bias terms, summed in position order (lanes below ext), added to the last run
                float xs = bias_x;
#pragma unroll
                for (int i = 0; i < 5; ++i) {
                    const float t = __shfl_up_sync(kFull, xs, 1 << i);
                    if (lane >= (1 << i)) xs += t;
                }
                xs = __shfl_sync(kFull, xs, ext - 1);
                if (lane == cnt - 1) gb += xs;
            }
            const bool in_first = (s.slot & 1) == 0;
            const bool parked = s.partial && !(lane == cnt - 1 && absorb);
            if (s.is_last && !(in_first && skip)) {
                if (parked) {
                    p.part[(size_t)s.slot * p.pitch + p.dp] = gb;
                } else {
                    if (p.emit) *emit_bias(p.push, p.gb_out, s.key) = gb;
                    if (p.apply) {
                        float w = p.tableb[s.key], a = p.adagrad ? p.accb[s.key] : 0.f;
                        opt_step(w, a, gb, p.lr, p.adagrad);
                        if (p.adagrad) p.accb[s.key] = a;
                        p.tableb[s.key] = w;
                    }
                }
            }
        }
        constexpr bool pay_vec = MODE == 1 || VEC;         // ev rows are always 16-byte aligned; dz rows iff K % 4 == 0
        for (int col0 = 0; col0 < p.width; col0 += ROWS_TILE) {
            const int q = col0 + 4 * lane;                 // first column of this lane
            const bool inq = q < p.width;
            // ---- phase 1: accumulate runs in position order ----
            float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
            int r = -1;
            // positions [lo, hi) of one chunk, the occurrence of position i in lane i's (off_l, coef_l); a run starts at
            // every set bit of hd
            auto gather = [&](int off_l, float coef_l, int lo, int hi, unsigned hd) {
                constexpr int UN = 16;     // payload rows in flight per warp
                for (int b0 = 0; b0 < hi; b0 += UN) {
                    float4 v[UN];
                    float cf[UN];
#pragma unroll
                    for (int u = 0; u < UN; ++u) {
                        const int pp = (b0 + u) & 31;
                        const int off = __shfl_sync(kFull, off_l, pp);
                        cf[u] = __shfl_sync(kFull, coef_l, pp);
                        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (b0 + u < hi && b0 + u >= lo && inq) v[u] = ld4<pay_vec>(p.payload + (size_t)off + q, q, p.width);
                    }
#pragma unroll
                    for (int u = 0; u < UN; ++u) {
                        const int pp = b0 + u;
                        if (pp < hi) {
                            if ((hd >> pp) & 1u) {
                                if (r >= 0 && lane < sq) S[r * sq + lane] = a;
                                ++r;
                                a = make_float4(0.f, 0.f, 0.f, 0.f);
                            }
                            if (MODE == 0) { a.x += v[u].x; a.y += v[u].y; a.z += v[u].z; a.w += v[u].w; }
                            else { a.x = fmaf(cf[u], v[u].x, a.x); a.y = fmaf(cf[u], v[u].y, a.y); a.z = fmaf(cf[u], v[u].z, a.z); a.w = fmaf(cf[u], v[u].w, a.w); }
                        }
                    }
                }
            };
            gather(off_m, coef_m, skipn, cnt, heads);
            gather(off_x, coef_x, 0, ext, 0u);     // absorbed tail: the last run continues through `ext` positions of the next chunk
            if (r >= 0 && lane < sq) S[r * sq + lane] = a;
            __syncwarp();
            // ---- phase 2: one optimiser read-modify-write (or one emitted gradient row) per run ----
            constexpr int RN = 8;      // table + accumulator rows in flight per warp
            unsigned hm = heads;                          // run heads still to visit (lowest set bit = next run)
            for (int r0 = 0; r0 < nr; r0 += RN) {
                float4 w[RN], ac[RN];
                uint32_t row[RN];
                int kind[RN];            // 0 nothing, 1 complete run, 2 partial -> slot 2c, 3 partial -> slot 2c+1
#pragma unroll
                for (int u = 0; u < RN; ++u) {
                    const int rr = r0 + u;
                    kind[u] = 0;
                    row[u] = 0;
                    w[u] = ac[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (rr < nr) {
                        const int hp = __ffs(hm) - 1;                   // position of the rr-th run head
                        hm &= hm - 1;
                        row[u] = __shfl_sync(kFull, s.key, hp);
                        const bool partial = (rr == 0 && cont_prev) || (rr == nr - 1 && cont_next && !absorb);
                        kind[u] = partial ? (hp == 0 ? 2 : 3) : 1;
                        if (rr == 0 && skip) kind[u] = 0;            // absorbed by the previous chunk
                        if (kind[u] == 1 && p.apply && inq) {
                            const size_t idx = (size_t)row[u] * p.width + q;
                            w[u] = ld4<VEC>(p.table + idx, q, p.width);
                            if (p.adagrad) ac[u] = ld4<VEC>(p.acc + idx, q, p.width);
                        }
                    }
                }
#pragma unroll
                for (int u = 0; u < RN; ++u) {
                    if (kind[u] == 0 || !inq || lane >= sq) continue;
                    const float4 g = S[(r0 + u) * sq + lane];
                    if (kind[u] >= 2) {
                        // a run-time test on purpose: the same choice made at compile time (pay_vec) measured 1.5 us slower
                        // in the entity update at T (B200, 1000 W power limit)
                        float* o = p.part + (size_t)(2 * c + (kind[u] - 2)) * p.pitch + q;
                        if ((p.pitch & 3) == 0) st4<true>(o, g, q, p.width);
                        else st4<false>(o, g, q, p.width);
                        continue;
                    }
                    const size_t idx = (size_t)row[u] * p.width + q;
                    if (p.emit) st4<VEC>(emit_row(p.push, p.g_out, row[u], p.width) + q, g, q, p.width);
                    if (p.apply) {
                        float4 wv = w[u], av = ac[u];
                        opt_step(wv, av, g, p.lr, p.adagrad);
                        st4<VEC>(p.table + idx, wv, q, p.width);
                        if (p.adagrad) st4<VEC>(p.acc + idx, av, q, p.width);
                    }
                }
            }
            __syncwarp();
        }
    }
}


// level 2: a CTA looks at 8 consecutive chunks at a time, one per warp.  If a multi-chunk segment starts in the warp's chunk,
// its lanes probe the first key of the next chunks 32 at a time to find its extent m.  Short segments (m <= LONG_WARP_MAX
// following chunks - nearly all of them: a run cut by one chunk boundary) are finished by the warp itself: the partial rows,
// the table row and the accumulator row are all in flight together, summed in chunk order, one optimiser read-modify-write.
// The few hot rows (Zipf head, hundreds of chunks) are left to the whole CTA: 8 warps sum disjoint strided subsets of the
// partial rows and the CTA combines them in warp order.
constexpr int LONG_WARP_MAX = 8;

__device__ __forceinline__ int long_extent(const uint32_t* __restrict__ keys_s, int nchunks, int c0, uint32_t row, int lane) {
    int m = 0;
    for (int base = c0 + 1; base < nchunks; base += 32) {
        const int c = base + lane;
        const bool cont = c < nchunks && keys_s[(size_t)c << 5] == row;
        const unsigned bal = __ballot_sync(kFull, cont);
        if (bal == 0xffffffffu) { m += 32; continue; }
        m += __ffs(~bal) - 1;
        break;
    }
    return m;
}

// warp path: row[0..width) of (table, acc) updated with part[slot0] + sum_{i<m} part[2 (c0+1+i)] (pitch floats per slot)
__device__ __forceinline__ void long2_warp_row(const float* __restrict__ part, int pitch, int width, int slot0, int c0, int m,
                                               float* __restrict__ trow, float* __restrict__ arow, float* __restrict__ grow, float lr,
                                               int adagrad, int emit, int apply, int lane) {
    const bool vec = ((width | pitch) & 3) == 0;
    if (vec) {
        for (int q = 4 * lane; q < width; q += 128) {
            float4 x[LONG_WARP_MAX];
            const float4 g0 = *reinterpret_cast<const float4*>(part + (size_t)slot0 * pitch + q);
#pragma unroll
            for (int u = 0; u < LONG_WARP_MAX; ++u)
                x[u] = u < m ? *reinterpret_cast<const float4*>(part + (size_t)(2 * (c0 + 1 + u)) * pitch + q) : make_float4(0.f, 0.f, 0.f, 0.f);
            float4 w = make_float4(0.f, 0.f, 0.f, 0.f), a = w;
            if (apply) {
                w = *reinterpret_cast<const float4*>(trow + q);
                if (adagrad) a = *reinterpret_cast<const float4*>(arow + q);
            }
            float4 g = g0;
#pragma unroll
            for (int u = 0; u < LONG_WARP_MAX; ++u) { g.x += x[u].x; g.y += x[u].y; g.z += x[u].z; g.w += x[u].w; }
            if (emit) *reinterpret_cast<float4*>(grow + q) = g;
            if (apply) {
                opt_step(w, a, g, lr, adagrad);
                *reinterpret_cast<float4*>(trow + q) = w;
                if (adagrad) *reinterpret_cast<float4*>(arow + q) = a;
            }
        }
    } else {
        for (int q = lane; q < width; q += 32) {
            float g = part[(size_t)slot0 * pitch + q];
            for (int u = 0; u < m; ++u) g += part[(size_t)(2 * (c0 + 1 + u)) * pitch + q];
            if (emit) grow[q] = g;
            if (apply) {
                float w = trow[q], a = adagrad ? arow[q] : 0.f;
                opt_step(w, a, g, lr, adagrad);
                if (adagrad) arow[q] = a;
                trow[q] = w;
            }
        }
    }
}

// level 2 of both row kinds: the entity rows carry the bias partial at column dp of every slot, which the warp path finishes
// in lane 0 and the CTA path as one more column
template <int MODE>
__device__ __forceinline__ void rows_long2(const RowsArgs& p) {
    pdl_enter();
    extern __shared__ float red[];      // [8][pitch]
    __shared__ int sh_slot[8], sh_m[8];
    __shared__ uint32_t sh_row[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nchunks = (p.n + 31) >> 5;
    const int ncol = MODE == 1 ? p.dp + 1 : p.width;       // columns of a slot the CTA path sums
    for (int cb = blockIdx.x * 8; cb < nchunks; cb += gridDim.x * 8) {
        {
            const int c = cb + warp;
            uint32_t row = 0;
            int slot0 = -1, m = 0;
            if (c < nchunks) slot0 = long_segment_start(p.keys_s, p.n, c, &row, kAbsorbs<MODE>);
            if (slot0 >= 0) m = long_extent(p.keys_s, nchunks, c, row, lane);
            if (slot0 >= 0 && m <= LONG_WARP_MAX) {
                const size_t ro = (size_t)row * p.width;
                long2_warp_row(p.part, p.pitch, p.width, slot0, c, m, p.table + ro, p.acc + ro, emit_row(p.push, p.g_out, row, p.width),
                               p.lr, p.adagrad, p.emit, p.apply, lane);
                if (MODE == 1 && lane == 0) {
                    float g = p.part[(size_t)slot0 * p.pitch + p.dp];
                    for (int u = 0; u < m; ++u) g += p.part[(size_t)(2 * (c + 1 + u)) * p.pitch + p.dp];
                    if (p.emit) *emit_bias(p.push, p.gb_out, row) = g;
                    if (p.apply) {
                        float wv = p.tableb[row], a = p.adagrad ? p.accb[row] : 0.f;
                        opt_step(wv, a, g, p.lr, p.adagrad);
                        if (p.adagrad) p.accb[row] = a;
                        p.tableb[row] = wv;
                    }
                }
                slot0 = -1;
            }
            if (lane == 0) { sh_slot[warp] = slot0; sh_m[warp] = m; sh_row[warp] = row; }
        }
        __syncthreads();
        for (int ci = 0; ci < 8; ++ci) {
            const int c0 = cb + ci;
            const int slot0 = sh_slot[ci], m = sh_m[ci];
            const uint32_t row = sh_row[ci];
            if (slot0 < 0) continue;
            // warp w sums partial rows of chunks c0+1+w, c0+1+w+8, ...
            for (int j0 = 0; j0 < ncol; j0 += 32) {
                const int j = j0 + lane;
                float acc = 0.f;
                constexpr int UN = 8;
                for (int i = warp; i < m; i += 8 * UN) {
                    float x[UN];
#pragma unroll
                    for (int u = 0; u < UN; ++u) {
                        const int ii = i + 8 * u;
                        x[u] = (ii < m && j < ncol) ? p.part[(size_t)(2 * (c0 + 1 + ii)) * p.pitch + j] : 0.f;
                    }
#pragma unroll
                    for (int u = 0; u < UN; ++u) acc += x[u];
                }
                if (j < ncol) red[warp * p.pitch + j] = acc;
            }
            __syncthreads();
            for (int j = threadIdx.x; j < ncol; j += 256) {
                const bool bias = MODE == 1 && j == p.dp;
                if (MODE == 1 && j >= p.width && !bias) continue;
                float g = p.part[(size_t)slot0 * p.pitch + j];
#pragma unroll
                for (int w = 0; w < 8; ++w) g += red[w * p.pitch + j];
                float* P = bias ? p.tableb + row : p.table + (size_t)row * p.width + j;
                float* AC = bias ? p.accb + row : p.acc + (size_t)row * p.width + j;
                if (p.emit) *(bias ? emit_bias(p.push, p.gb_out, row) : emit_row(p.push, p.g_out, row, p.width) + j) = g;
                if (p.apply) {
                    float wv = *P, a = p.adagrad ? *AC : 0.f;
                    opt_step(wv, a, g, p.lr, p.adagrad);
                    if (p.adagrad) *AC = a;
                    *P = wv;
                }
            }
            __syncthreads();        // `red` is reused by the CTA's next segment
        }
        __syncthreads();            // sh_* are rewritten by the next round
    }
}

// two kernels (not one template) so that profiles and phase labels keep telling the row kinds apart
__global__ void __launch_bounds__(256) k_w_long2(RowsArgs p) { rows_long2<0>(p); }
__global__ void __launch_bounds__(256) k_entity_long2(RowsArgs p) { rows_long2<1>(p); }

// ---- dense parameters ----
// sum the batch-split partials of dC/dC1/dC2 and the per-CTA partials of dWb into the flat dense gradient buffer.
// blocks [0, n_elem_blocks): 4 consecutive elements per thread (float4 when aligned), the splits summed in split order;
// blocks [n_elem_blocks, +K): one CTA per column k of dWb - thread t sums partial rows t, t+256, ... and a fixed-shape
// shared-memory tree combines the 256 values (deterministic).
// slots of the partial buffer that hold element i0 of [C | C1 | C2]: uniform (SIMT path, tile_slots == nullptr) or, on the
// tensor path, the slot count of the 128-row operand tile the element's row n = (i, j) | C1 row | C2 row falls in (a small
// per-tile table made at create time: rae_decoder_tc.cu)
struct DenseSlots { const int32_t* tile_slots; int uniform; int d, K, DP, n_bil_rows, hasM; };
__device__ __forceinline__ int dense_slots_of(const DenseSlots& ds, size_t i0) {
    if (ds.tile_slots == nullptr) return ds.uniform;
    const int r = (int)(i0 / (size_t)ds.K);                    // row of the [units*d, K] layout
    const int nb = ds.hasM ? ds.d * ds.d : 0;
    int n;
    if (r < nb) { const int i = r / ds.d; n = i * ds.DP + (r - i * ds.d); }
    else { const int m = r - nb, which = m / ds.d; n = ds.n_bil_rows + which * ds.DP + (m - which * ds.d); }
    return ds.tile_slots[n >> 7];
}

// sum of the `nsplit` partial slots of 4 consecutive elements, in slot order, 8 or 16 slots per round trip: the loads of a round
// are issued back to back (volatile asm; slots beyond nsplit re-read the last valid one - a cache hit - and are dropped by
// the select).  The C1 / C2 tiles of the one-tile dC kernel have 64 slots: read one after the other (a load - add chain)
// they made 25 CTAs of this kernel run 40 us after the other 1700 had finished (ncu: SMs active 38 % of the duration).
__device__ __forceinline__ float4 sum_slots(const float* __restrict__ part, size_t plane, size_t i0, int nsplit) {
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    int sp0 = 0;
    for (; sp0 + 8 < nsplit; sp0 += 16) {              // more than 8 slots left: 16 per round trip
        float4 x[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) x[u] = ldg_stream4(part + (size_t)min(sp0 + u, nsplit - 1) * plane + i0);
#pragma unroll
        for (int u = 0; u < 16; ++u)
            if (sp0 + u < nsplit) { s.x += x[u].x; s.y += x[u].y; s.z += x[u].z; s.w += x[u].w; }
    }
    for (; sp0 < nsplit; sp0 += 8) {
        float4 x[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) x[u] = ldg_stream4(part + (size_t)min(sp0 + u, nsplit - 1) * plane + i0);
#pragma unroll
        for (int u = 0; u < 8; ++u)
            if (sp0 + u < nsplit) { s.x += x[u].x; s.y += x[u].y; s.z += x[u].z; s.w += x[u].w; }
    }
    return s;
}

// fused optimiser step (single-GPU production path): the summed gradient goes straight into the AdaGrad / SGD rule of its
// element of C | C1 | C2 | Wb instead of through the flat gradient buffer and a second kernel (Optimizers.py:29-32,51).
// Only taken when every tensor is 16-byte aligned and K % 4 == 0 (launch_dense_finalize checks).
struct DenseFuse { float* p[4]; float* acc[4]; size_t off[4]; float lr, r1, r2; int adagrad; int on; };
__device__ __forceinline__ void dense_rule(float& w, float& a, float g, const DenseFuse& f, bool reg) {
    if (reg) {
        const float sgn = (w > 0.f) ? 1.f : ((w < 0.f) ? -1.f : 0.f);
        g += f.r1 * sgn + 2.f * f.r2 * w;
    }
    opt_step(w, a, g, f.lr, f.adagrad);
}

__global__ void __launch_bounds__(256) k_dense_finalize(const float* __restrict__ part, DenseSlots ds, size_t n_units_elems,
                                                        const float* __restrict__ dzsum_part, int n_dz_part, int K,
                                                        float* __restrict__ out, size_t off_wb, int n_elem_blocks, DenseFuse fz) {
    pdl_enter();
    if ((int)blockIdx.x < n_elem_blocks) {
        // element blocks in REVERSE order: the C1 / C2 rows at the end of the flat layout have the most partial slots (64 at
        // the target shape, several load round trips): their CTAs start in the first wave instead of the last
        const size_t i0 = ((size_t)(n_elem_blocks - 1 - (int)blockIdx.x) * blockDim.x + threadIdx.x) * 4;
        if (i0 >= n_units_elems) return;
        if (fz.on) {
            const int t = i0 >= fz.off[2] ? 2 : (i0 >= fz.off[1] ? 1 : 0);
            const size_t li = i0 - (t == 2 ? fz.off[2] : (t == 1 ? fz.off[1] : fz.off[0]));
            float* const pp = (t == 2 ? fz.p[2] : (t == 1 ? fz.p[1] : fz.p[0])) + li;
            float* const pa = (t == 2 ? fz.acc[2] : (t == 1 ? fz.acc[1] : fz.acc[0])) + li;
            const int nsplit = dense_slots_of(ds, i0);
            // Every load of the element - parameter, accumulator and up to 8 slots - is issued before the first add (volatile
            // asm stays in program order): ONE memory latency per thread.  Written as conditional loads the compiler chained
            // them, load - add - load - add through one register (38 us for 46 MB, ncu).  Slots beyond nsplit re-read the last
            // valid one (a cache hit) and are dropped by the select.
            float4 w = *reinterpret_cast<const float4*>(pp);
            float4 a = fz.adagrad ? *reinterpret_cast<const float4*>(pa) : make_float4(0.f, 0.f, 0.f, 0.f);
            const float4 s = sum_slots(part, n_units_elems, i0, nsplit);
            const bool reg = fz.r1 != 0.f || fz.r2 != 0.f;
            dense_rule(w.x, a.x, s.x, fz, reg); dense_rule(w.y, a.y, s.y, fz, reg);
            dense_rule(w.z, a.z, s.z, fz, reg); dense_rule(w.w, a.w, s.w, fz, reg);
            *reinterpret_cast<float4*>(pp) = w;
            if (fz.adagrad) *reinterpret_cast<float4*>(pa) = a;
            return;
        }
        if ((n_units_elems & 3) == 0 && (K & 3) == 0) {        // the 4 elements share a row
            const int nsplit = dense_slots_of(ds, i0);
            // all slot loads are issued before the first add (one memory latency, not one per slot); summed in slot order
            const float4 s = sum_slots(part, n_units_elems, i0, nsplit);
            *reinterpret_cast<float4*>(out + i0) = s;
        } else {
            for (size_t i = i0; i < min(i0 + 4, n_units_elems); ++i) {
                const int nsplit = dense_slots_of(ds, i);
                float s = 0.f;
                for (int sp = 0; sp < nsplit; ++sp) s += part[(size_t)sp * n_units_elems + i];
                out[i] = s;
            }
        }
        return;
    }
    // dWb[k] = sum over the examples of dz[b][k] is a heavily cancelling sum (every row of dz sums to zero): the partial rows
    // are combined in double so that the reduction itself adds nothing to the fp32 error of the terms
    __shared__ double red[256];
    const int k = (int)blockIdx.x - n_elem_blocks;
    double s = 0.0;
    for (int c = threadIdx.x; c < n_dz_part; c += 256) s += (double)dzsum_part[(size_t)c * K + k];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        if (fz.on) {
            float w = fz.p[3][k], a = fz.adagrad ? fz.acc[3][k] : 0.f;
            dense_rule(w, a, (float)red[0], fz, false);
            fz.p[3][k] = w;
            if (fz.adagrad) fz.acc[3][k] = a;
        } else {
            out[off_wb + k] = (float)red[0];
        }
    }
}

// elementwise optimiser over up to 5 dense tensors in one launch (blockIdx.y = tensor):
// g = grad (+ adj*(l1*sign(p) + 2*l2*p)); AdaGrad (Optimizers.py:29-32) or SGD (:51).
// Also used for W when the regulariser makes its gradient dense (OieModel.py:54-56).
struct DenseJob { float* p; float* acc; float* grad; size_t n; float reg_l1, reg_l2; int write_back; };
struct DenseJobs { DenseJob j[5]; int count; float lr; int adagrad; };

__global__ void __launch_bounds__(256) k_dense_apply(DenseJobs jobs) {
    pdl_enter();
    const DenseJob jb = jobs.j[blockIdx.y];
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < jb.n; i += (size_t)gridDim.x * blockDim.x) {
        float w = jb.p[i];
        float g = jb.grad[i];
        if (jb.reg_l1 != 0.f || jb.reg_l2 != 0.f) {
            const float sgn = (w > 0.f) ? 1.f : ((w < 0.f) ? -1.f : 0.f);
            g += jb.reg_l1 * sgn + 2.f * jb.reg_l2 * w;
            if (jb.write_back) jb.grad[i] = g;
        }
        float a = jobs.adagrad ? jb.acc[i] : 0.f;
        opt_step(w, a, g, jobs.lr, jobs.adagrad);
        if (jobs.adagrad) jb.acc[i] = a;
        jb.p[i] = w;
    }
}

// deterministic partial sums of |p| and p^2 (regulariser value, OieModel.py:54-56,60-62)
__global__ void k_reg_norms(const float* __restrict__ p, size_t n, double* __restrict__ part /* [grid][2] */) {
    __shared__ double s1[256], s2[256];
    double a = 0.0, b = 0.0;
    // each thread visits i, i + stride, ... in that order; the loads of NU consecutive visits are issued before their adds
    // (one memory latency per NU elements instead of per element), the summation order is unchanged
    constexpr int NU = 16;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + (NU - 1) * stride < n; i += NU * stride) {
        float x[NU];
#pragma unroll
        for (int u = 0; u < NU; ++u) x[u] = p[i + u * stride];
#pragma unroll
        for (int u = 0; u < NU; ++u) {
            const double v = (double)x[u];
            a += fabs(v);
            b += v * v;
        }
    }
    for (; i < n; i += stride) {
        const double v = (double)p[i];
        a += fabs(v);
        b += v * v;
    }
    s1[threadIdx.x] = a; s2[threadIdx.x] = b;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) { s1[threadIdx.x] += s1[threadIdx.x + o]; s2[threadIdx.x] += s2[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { part[2 * blockIdx.x] = s1[0]; part[2 * blockIdx.x + 1] = s2[0]; }
}

// cost = -(sum of score partials)/Z + adj*(l1*L1 + l2*L2)       (OieModel.py:90, OieInduction.py:134-135)
// one CTA; thread t owns elements t, t+256, ... and the tree below has a fixed shape -> deterministic
__global__ void __launch_bounds__(256) k_cost(const double* __restrict__ loss_part, int n_loss,
                                              const double* __restrict__ reg_part, int n_reg, double invZ,
                                              double adj_l1, double adj_l2, double* __restrict__ cost,
                                              double* __restrict__ cost_mapped) {
    pdl_enter();
    __shared__ double s0[256], s1[256], s2[256];
    double a = 0.0, b = 0.0, c = 0.0;
    for (int i = threadIdx.x; i < n_loss; i += 256) a += loss_part[i];
    for (int i = threadIdx.x; i < n_reg; i += 256) { b += reg_part[2 * i]; c += reg_part[2 * i + 1]; }
    s0[threadIdx.x] = a; s1[threadIdx.x] = b; s2[threadIdx.x] = c;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            s0[threadIdx.x] += s0[threadIdx.x + o];
            s1[threadIdx.x] += s1[threadIdx.x + o];
            s2[threadIdx.x] += s2[threadIdx.x + o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double v = -s0[0] * invZ + adj_l1 * s1[0] + adj_l2 * s2[0];
        *cost = v;
        *cost_mapped = v;      // pinned host word (UVA): the caller reads it after the event behind this kernel, no D2H copy
    }
}

int ensure_part(rae_engine* h, float** buf, size_t* cap, size_t need) {
    if (need <= *cap) return RAE_OK;
    if (*buf) cudaFree(*buf);
    *buf = nullptr;
    *cap = 0;
    const size_t want = need + need / 4;
    cudaError_t e = cudaMalloc((void**)buf, want * sizeof(float));
    if (e != cudaSuccess) return fail(h, RAE_ENOMEM, "cudaMalloc(partials %zu floats) failed: %s", want, cudaGetErrorString(e));
    *cap = want;
    return RAE_OK;
}

}  // namespace

size_t segwork_temp_bytes(int64_t n) {
    size_t a = 0, b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const uint32_t*)nullptr,
                                    (uint32_t*)nullptr, (int)n, 0, 32, (cudaStream_t)0);
    cub::DeviceScan::ExclusiveSum(nullptr, b, (const int32_t*)nullptr, (int32_t*)nullptr, (int)n, (cudaStream_t)0);
    const size_t own = radix_sort_temp_bytes(n, 256);      // rae_sort.cu (any SM count up to 256)
    return std::max(std::max(a, b), own) + 256;
}

// pairs up to this count go through the one-kernel cooperative sort (rae_sort.cu); device-wide sorts of more pairs than
// that (bind-time sorts of a whole split, config 5's global batch on one GPU) are bandwidth-bound and stay with the
// library's onesweep
static bool own_sort(const rae_engine* h, int64_t n) { return h->coop_launch && n <= RAE_OWN_SORT_MAX; }

int sort_entities(rae_engine* h, const int32_t* a1, const int32_t* a2, const int32_t* neg1, const int32_t* neg2, int64_t neg_ld,
                  cudaStream_t st) {
    const int64_t n = (int64_t)(2 + 2 * h->S) * h->B;
    if (own_sort(h, n))
        return radix_sort_entities(h, a1, a2, neg1, neg2, neg_ld, h->ent.keys_s, h->ent.vals_s, h->ent.key_bits, st, h->ent_cub_tmp,
                                   h->ent_cub_bytes);
    int rc = build_entity_keys(h, a1, a2, neg1, neg2, neg_ld, st);
    if (rc) return rc;
    return sort_pairs(h, h->ent, n, st, h->ent_cub_tmp, h->ent_cub_bytes);
}

int build_entity_keys(rae_engine* h, const int32_t* a1, const int32_t* a2, const int32_t* neg1, const int32_t* neg2,
                      int64_t neg_ld, cudaStream_t st) {
    const int n = (2 + 2 * h->S) * h->B;
    const int blocks = std::min((n + 255) / 256, 4 * h->num_sms);
    launch_pdl(k_entity_keys, dim3(blocks), dim3(256), 0, st, a1, a2, neg1, neg2, neg_ld, h->B, h->S, h->ent.keys, h->ent.vals);
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

int build_feature_keys(rae_engine* h, const int32_t* indptr, const int32_t* indices, cudaStream_t st) {
    const int blocks = (h->B * 32 + 255) / 256;
    k_feature_keys<<<blocks, 256, 0, st>>>(indptr, indices, h->B, h->feat.keys, h->feat.vals);
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

int sort_pairs(rae_engine* h, SegWork& w, int64_t n, cudaStream_t st, void* tmp, size_t tmp_bytes) {
    if (n > w.capacity) return fail(h, RAE_EINVAL, "internal: sort workspace too small (%lld > %lld)", (long long)n, (long long)w.capacity);
    if (n <= 0) return RAE_OK;
    if (own_sort(h, n)) return radix_sort_pairs(h, w.keys, w.vals, w.keys_s, w.vals_s, n, w.key_bits, st, tmp, tmp_bytes);
    size_t bytes = tmp_bytes;
    // LSD radix sort is stable: equal rows keep ascending occurrence order == np.argsort(kind='stable')
    RAE_CUDA(h, cub::DeviceRadixSort::SortPairs(tmp, bytes, w.keys, w.keys_s, w.vals, w.vals_s, (int)n, 0,
                                                w.key_bits, st));
    h->launches += (w.key_bits + 7) / 8 + 2;
    return RAE_OK;
}

int segment_heads(rae_engine* h, const uint32_t* keys_s, int64_t n, SegWork& w, cudaStream_t st) {
    if (n > w.capacity) return fail(h, RAE_EINVAL, "internal: segment workspace too small");
    if (n > 0) {
        const int blocks = std::min((int)((n + 255) / 256), 4 * h->num_sms);
        k_flag_heads<<<blocks, 256, 0, st>>>(keys_s, (int)n, w.flags);
        size_t bytes = h->cub_bytes;
        RAE_CUDA(h, cub::DeviceScan::ExclusiveSum(h->cub_tmp, bytes, w.flags, w.pos, (int)n, st));
        k_scatter_heads<<<blocks, 256, 0, st>>>(w.flags, w.pos, (int)n, w.seg_start, w.n_seg);
    } else {
        k_scatter_heads<<<1, 32, 0, st>>>(w.flags, w.pos, 0, w.seg_start, w.n_seg);
    }
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

int count_unique(rae_engine* h, const uint32_t* keys_s, int64_t n, int32_t* out_dev, cudaStream_t st) {
    RAE_CUDA(h, cudaMemsetAsync(out_dev, 0, sizeof(int32_t), st));
    if (n > 0) {
        const int blocks = std::min((int)((n + 255) / 256), 4 * h->num_sms);
        k_count_heads<<<blocks, 256, 0, st>>>(keys_s, (int)n, out_dev);
        RAE_CUDA(h, cudaGetLastError());
    }
    return RAE_OK;
}

// one sorted-occurrence update: sizes the partial buffer, then level 1 (k_rows_chunk) and level 2 (k_*_long2)
template <int MODE>
static int rows_update(rae_engine* h, RowsArgs& p, cudaStream_t st) {
    if (p.n <= 0) return RAE_OK;
    const int64_t nchunks = ((int64_t)p.n + 31) / 32;
    int rc = MODE == 1 ? ensure_part(h, &h->ent_part, &h->ent_part_cap, (size_t)(2 * nchunks) * p.pitch)
                       : ensure_part(h, &h->feat_part, &h->feat_part_cap, (size_t)(2 * nchunks) * p.pitch);
    if (rc) return rc;
    p.part = MODE == 1 ? h->ent_part : h->feat_part;
    const int slab_cols = std::min(ROWS_TILE, (p.width + 3) & ~3);
    // The kernel is bound by DRAM latency (one optimiser read-modify-write per unique row) and the per-warp slab limits how
    // many warps an SM holds: CTAs of TWO warps pack 7 CTAs = 14 warps into the 227 KB of an SM where one CTA of 8 warps
    // (128 KB at 128 columns) left room for nothing else.
    constexpr int WARPS = 2;
    const size_t smem = (size_t)WARPS * 32 * slab_cols * sizeof(float);
    const bool vec = (p.width & 3) == 0;
    auto kern = vec ? k_rows_chunk<MODE, true> : k_rows_chunk<MODE, false>;
    static bool attr_done[2] = {false, false};
    if (!attr_done[vec ? 1 : 0]) {
        RAE_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, WARPS * 32 * ROWS_TILE * (int)sizeof(float)));
        attr_done[vec ? 1 : 0] = true;
    }
    const int blocks = (int)std::min<int64_t>((nchunks + WARPS - 1) / WARPS, (int64_t)h->num_sms * 32);
    launch_pdl(kern, dim3(blocks), dim3(32 * WARPS), smem, st, p, slab_cols);
    RAE_CUDA(h, cudaGetLastError());
    const int blocks2 = (int)std::min<int64_t>((nchunks + 7) / 8, (int64_t)h->num_sms * 8);
    launch_pdl(MODE == 1 ? k_entity_long2 : k_w_long2, dim3(blocks2), dim3(256), sizeof(float) * 8 * p.pitch, st, p);
    h->launches += 2;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

// entity rows: A[row,:] and Ab[row] updated with the coefficient-weighted sum of the occurrences' ev rows and bias terms
int launch_entity_update(rae_engine* h, const uint32_t* keys_s, const uint32_t* vals_s, int64_t n_occ, bool emit_dense,
                         bool apply, cudaStream_t st) {
    RowsArgs p{};
    p.keys_s = keys_s; p.vals_s = vals_s; p.n = (int)n_occ;
    p.payload = h->ev; p.width = h->d; p.pitch = h->dp + 4;
    p.table = h->P[RAE_P_A]; p.acc = h->ACC[RAE_P_A]; p.g_out = h->gA_dense;
    p.lr = (float)h->cfg.lr; p.adagrad = h->adagrad; p.emit = emit_dense; p.apply = apply;
    p.B = h->B; p.S = h->S; p.dp = h->dp; p.sc = h->sc; p.gn1 = h->gn1; p.gn2 = h->gn2;
    p.tableb = h->P[RAE_P_AB]; p.accb = h->ACC[RAE_P_AB]; p.gb_out = h->gAb_dense;
    if (h->emit_only && h->push.on && h->push.e_ids != nullptr)
        p.push = PushTo{h->push.a_dev, h->push.ab_dev, h->push.e_ids, h->push.world, (long long)h->push.rank * h->push.n_cap};
    return rows_update<1>(h, p, st);
}

// feature rows: W[row,:] updated with the sum of dz[val,:] over the row's sorted occurrences
int launch_w_update(rae_engine* h, const uint32_t* keys_s, const uint32_t* vals_s, int64_t nnz, bool emit_dense,
                    bool apply, cudaStream_t st) {
    RowsArgs p{};
    p.keys_s = keys_s; p.vals_s = vals_s; p.n = (int)nnz;
    p.payload = h->dz; p.width = h->K; p.pitch = h->K;
    p.table = h->P[RAE_P_W]; p.acc = h->ACC[RAE_P_W]; p.g_out = h->gW_dense;
    p.lr = (float)h->cfg.lr; p.adagrad = h->adagrad; p.emit = emit_dense; p.apply = apply;
    if (h->emit_only && h->push.on && h->push.f_ids != nullptr)
        p.push = PushTo{h->push.w_dev, nullptr, h->push.f_ids, h->push.world, (long long)h->push.rank * h->push.f_cap};
    return rows_update<0>(h, p, st);
}

int launch_dense_finalize(rae_engine* h, cudaStream_t st, bool fuse_apply) {
    const size_t n_units = (size_t)h->off_gWb;   // elements of [C | C1 | C2]
    DenseFuse fz{};
    h->dense_fused = false;
    if (fuse_apply && !h->debug_dense && !h->emit_only && (n_units & 3) == 0 && (h->K & 3) == 0) {
        const bool regdec = (h->cfg.l1 != 0.0 || h->cfg.l2 != 0.0) && h->cfg.ext_reg;
        fz.lr = (float)h->cfg.lr; fz.adagrad = h->adagrad;
        fz.r1 = regdec ? (float)(h->cfg.adj * h->cfg.l1) : 0.f;
        fz.r2 = regdec ? (float)(h->cfg.adj * h->cfg.l2) : 0.f;
        // tensors in the order of the flat layout [C | C1 | C2]; absent ones have zero extent (their offsets coincide)
        const int pid[4] = {RAE_P_C, RAE_P_C1, RAE_P_C2, RAE_P_WB};
        const size_t off[4] = {(size_t)h->off_gC, (size_t)h->off_gC1, (size_t)h->off_gC2, (size_t)h->off_gWb};
        bool ok = true;
        for (int t = 0; t < 4; ++t) {
            fz.p[t] = h->P[pid[t]]; fz.acc[t] = h->ACC[pid[t]]; fz.off[t] = off[t];
            const bool present = t == 3 || (t == 0 ? h->hasM : h->hasSP);
            if (!present) continue;
            if (fz.p[t] == nullptr || (h->adagrad && fz.acc[t] == nullptr)) ok = false;
            if (t < 3 && (((uintptr_t)fz.p[t] | (uintptr_t)fz.acc[t]) & 15)) ok = false;
        }
        if (!h->hasM) fz.off[0] = 0;      // C absent: element 0 belongs to C1 (off_gC1 == 0)
        fz.on = ok ? 1 : 0;
        h->dense_fused = ok;
    }
    const int n_elem_blocks = (int)((n_units + 1023) / 1024);
    DenseSlots ds{};
    ds.uniform = h->gC_nsplit;
    ds.d = h->d; ds.K = h->K; ds.hasM = h->hasM ? 1 : 0;
    if (h->use_tc) { ds.tile_slots = h->tc.tile_slots; ds.DP = h->tc.DP; ds.n_bil_rows = h->tc.n_bil_rows; }
    launch_pdl(k_dense_finalize, dim3(n_elem_blocks + h->K), dim3(256), 0, st, h->gC_part, ds, n_units, h->dzsum_part, h->dz_part_used, h->K,
                                                          h->dense_grad, (size_t)h->off_gWb, n_elem_blocks, fz);
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

int launch_dense_apply(rae_engine* h, cudaStream_t st) {
    const bool reg = h->reg;
    if (h->dense_fused && !h->dense_w) return RAE_OK;      // applied inside k_dense_finalize
    const bool regdec = reg && h->cfg.ext_reg;
    const size_t dd = (size_t)h->d * h->d * h->K, dk = (size_t)h->d * h->K;
    const float r1 = (float)(h->cfg.adj * h->cfg.l1), r2 = (float)(h->cfg.adj * h->cfg.l2);
    DenseJobs jobs{};
    jobs.lr = (float)h->cfg.lr;
    jobs.adagrad = h->adagrad;
    size_t nmax = 0;
    auto add = [&](int pid, float* grad, size_t n, bool regularised) {
        if (n == 0) return;
        DenseJob& j = jobs.j[jobs.count++];
        j.p = h->P[pid]; j.acc = h->ACC[pid]; j.grad = grad; j.n = n;
        j.reg_l1 = regularised ? r1 : 0.f;
        j.reg_l2 = regularised ? r2 : 0.f;
        j.write_back = h->debug_dense ? 1 : 0;
        nmax = std::max(nmax, n);
    };
    if (!h->dense_fused) {
        if (h->hasM) add(RAE_P_C, h->dense_grad + h->off_gC, dd, regdec);
        if (h->hasSP) {
            add(RAE_P_C1, h->dense_grad + h->off_gC1, dk, regdec);
            add(RAE_P_C2, h->dense_grad + h->off_gC2, dk, regdec);
        }
        add(RAE_P_WB, h->dense_grad + h->off_gWb, (size_t)h->K, false);
    }
    // regulariser makes dW dense: gW_dense holds the data gradient (zero rows elsewhere)
    if (h->dense_w) add(RAE_P_W, h->gW_dense, (size_t)h->cfg.F * h->K, reg);
    const int bx = (int)std::min<size_t>((nmax + 255) / 256, (size_t)h->num_sms * 8);
    launch_pdl(k_dense_apply, dim3(bx, jobs.count), dim3(256), 0, st, jobs);
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

int launch_cost(rae_engine* h, cudaStream_t st, const float* w_shard, int64_t w_elems, bool with_dec) {
    int n_reg = 0;
    if (h->reg) {
        // fixed grid per tensor -> fixed summation order
        auto norms = [&](const float* p, size_t n) -> int {
            if (n == 0) return RAE_OK;
            const int blocks = 64;
            if (n_reg + blocks > h->n_reg_part) return fail(h, RAE_EINVAL, "internal: reg_part too small");
            k_reg_norms<<<blocks, 256, 0, st>>>(p, n, h->reg_part + 2 * (size_t)n_reg);
            n_reg += blocks;
            h->launches++;
            return RAE_OK;
        };
        int rc;
        // an emit-only handle's W is the step's compact copy, not the parameter: its norms come from the shard
        if (!h->emit_only && (rc = norms(h->P[RAE_P_W], (size_t)h->cfg.F * h->K))) return rc;
        if (w_shard && (rc = norms(w_shard, (size_t)w_elems))) return rc;
        if (h->cfg.ext_reg && (!h->emit_only || with_dec)) {
            if (h->hasM && (rc = norms(h->P[RAE_P_C], (size_t)h->d * h->d * h->K))) return rc;
            if (h->hasSP) {
                if ((rc = norms(h->P[RAE_P_C1], (size_t)h->d * h->K))) return rc;
                if ((rc = norms(h->P[RAE_P_C2], (size_t)h->d * h->K))) return rc;
            }
        }
    }
    const int n_loss = h->n_loss_part;
    launch_pdl(k_cost, dim3(1), dim3(256), 0, st, h->loss_part, n_loss, h->reg_part, n_reg, 1.0 / h->Z, h->cfg.adj * h->cfg.l1,
                              h->cfg.adj * h->cfg.l2, h->cost_dev, h->cost_pinned);
    h->launches++;
    RAE_CUDA(h, cudaGetLastError());
    return RAE_OK;
}

int launch_zero(rae_engine* h, void* p, size_t bytes, cudaStream_t st) {
    RAE_CUDA(h, cudaMemsetAsync(p, 0, bytes, st));
    return RAE_OK;
}

}  // namespace rae
