// C-ABI entry points (include/rae.h) and the per-step kernel schedule.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "rae_internal.h"

namespace rae {

bool g_pdl_enabled = true;      // process-wide: cleared when any handle is created with RAE_FLAG_NO_PDL

static char g_create_err[512] = "";

int fail(rae_engine* h, int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    char* dst = h ? h->err : g_create_err;
    vsnprintf(dst, 512, fmt, ap);
    va_end(ap);
    return code;
}

template <typename T>
static int dev_alloc(rae_engine* h, T** p, size_t n) {
    *p = nullptr;
    if (n == 0) n = 1;
    cudaError_t e = cudaMalloc((void**)p, n * sizeof(T));
    if (e != cudaSuccess) return fail(h, RAE_ENOMEM, "cudaMalloc(%zu bytes) failed: %s", n * sizeof(T), cudaGetErrorString(e));
    return RAE_OK;
}

static int alloc_segwork(rae_engine* h, SegWork& w, int64_t cap, int key_bits) {
    int rc;
    if ((rc = dev_alloc(h, &w.keys, cap))) return rc;
    if ((rc = dev_alloc(h, &w.vals, cap))) return rc;
    if ((rc = dev_alloc(h, &w.keys_s, cap))) return rc;
    if ((rc = dev_alloc(h, &w.vals_s, cap))) return rc;
    if ((rc = dev_alloc(h, &w.flags, cap))) return rc;
    if ((rc = dev_alloc(h, &w.pos, cap))) return rc;
    if ((rc = dev_alloc(h, &w.seg_start, cap + 1))) return rc;
    if ((rc = dev_alloc(h, &w.n_seg, 1))) return rc;
    w.capacity = cap;
    w.key_bits = key_bits;
    return RAE_OK;
}

static void free_segwork(SegWork& w) {
    cudaFree(w.keys); cudaFree(w.vals); cudaFree(w.keys_s); cudaFree(w.vals_s);
    cudaFree(w.flags); cudaFree(w.pos); cudaFree(w.seg_start); cudaFree(w.n_seg);
    w = SegWork{};
}

static int bits_for(int64_t n) {
    int b = 1;
    while (b < 32 && ((int64_t)1 << b) < n) ++b;
    return b;
}

static int ensure_cub(rae_engine* h, int64_t n) {
    size_t need = segwork_temp_bytes(n);
    if (need > h->cub_bytes) {
        if (h->cub_tmp) cudaFree(h->cub_tmp);
        h->cub_tmp = nullptr;
        cudaError_t e = cudaMalloc(&h->cub_tmp, need);
        if (e != cudaSuccess) return fail(h, RAE_ENOMEM, "cudaMalloc(cub temp %zu) failed: %s", need, cudaGetErrorString(e));
        h->cub_bytes = need;
    }
    return RAE_OK;
}

static int ensure_feat_capacity(rae_engine* h, int64_t nnz) {
    if (nnz <= h->feat.capacity) return RAE_OK;
    free_segwork(h->feat);
    int rc = alloc_segwork(h, h->feat, nnz + nnz / 8 + 1024, bits_for(h->cfg.F));
    if (rc) return rc;
    return ensure_cub(h, h->feat.capacity);
}

static void free_feature_cache(FeatureCache& c) {
    cudaFree(c.keys_s); cudaFree(c.vals_s);
    delete[] c.batch_off;
    c = FeatureCache{};
}

// one training step on device-resident inputs.  nnz_hint < 0: unknown (explicit API reads indptr back once).
static int run_step(rae_engine* h, const int32_t* indptr, const int32_t* indices, int64_t nnz, const int32_t* a1,
                    const int32_t* a2, const int32_t* neg1, const int32_t* neg2, int64_t neg_ld,
                    const uint32_t* f_keys_s, const uint32_t* f_vals_s, cudaStream_t st, bool finish_dense = true) {
    int rc;
    h->launches = 0;
    const bool emit = h->debug_dense || h->dense_w || h->emit_only;
    int phase = 0;
#define RAE_PHASE()                                                                    \
    do {                                                                               \
        if (h->profiling) RAE_CUDA(h, cudaEventRecord(h->ev_phase[phase], st));        \
        ++phase;                                                                       \
    } while (0)
    if (!h->tl_keep) h->tl_n = 0;
    h->tl_keep = false;
#define RAE_MARK(name, strm, sid)                                                          \
    do {                                                                                   \
        if (h->timeline && h->tl_n < RAE_TL_MAX) {                                         \
            RAE_CUDA(h, cudaEventRecord(h->tl_ev[h->tl_n], strm));                         \
            h->tl_name[h->tl_n] = name; h->tl_stream[h->tl_n] = sid; ++h->tl_n;            \
        }                                                                                  \
    } while (0)
    RAE_MARK("start", st, 0);
    // Independent branches run on two handle-owned side streams (forked from / joined into the caller's stream):
    //   s1: entity keys + stable sort (needs only the indices) ... entity-row update
    //   s2: W-row update
    // while the caller's stream carries encoder -> decoder -> dense gradients -> cost -> dense update.
    // Disabled when gradients are emitted densely (debug / regulariser) or per-phase profiling is on.
    const bool overlap = !h->dense_w && !h->debug_dense && !h->profiling && h->s1 != nullptr;
    // The dense-operand preparation depends only on the parameters: it runs beside the encoder on side stream 2.  (Moving
    // the q^T operand / L, R gather there as well was measured 13 us SLOWER per step: two more cross-stream edges.)
    const bool prepc_side = overlap && h->use_tc;
    cudaStream_t se = overlap ? h->s1 : st, sw = overlap ? h->s2 : st;
    const int64_t n_occ = (int64_t)(2 + 2 * h->S) * h->B;
    if (overlap) {
        RAE_CUDA(h, cudaEventRecord(h->ev_fork0, st));
        RAE_CUDA(h, cudaStreamWaitEvent(h->s1, h->ev_fork0, 0));
        if (prepc_side) {
            // the pre-split dense operands depend only on the parameters: prepared beside the encoder
            RAE_CUDA(h, cudaStreamWaitEvent(h->s2, h->ev_fork0, 0));
            if ((rc = tc_prepare_c(h, h->s2))) return rc;
            RAE_CUDA(h, cudaEventRecord(h->ev_prepc, h->s2));
            RAE_MARK("prep_c", h->s2, 2);
        }
        if ((rc = sort_entities(h, a1, a2, neg1, neg2, neg_ld, se))) return rc;
        RAE_MARK("entity_sort", se, 1);
    }
    RAE_PHASE();   // 0 encoder forward: q, log q, entropy
    if ((rc = launch_encoder_forward(h, indptr, indices, h->B, h->q, h->logq, h->sc + SC_ENT, nullptr, st))) return rc;
    RAE_MARK("encoder", st, 0);
    RAE_PHASE();   // 1 entity occurrence keys -> stable sort -> segments (depends on the indices only)
    if (!overlap) {
        if ((rc = sort_entities(h, a1, a2, neg1, neg2, neg_ld, st))) return rc;
    }
    RAE_PHASE();   // 2 feature sort (skipped when the per-batch transposed index was cached at bind time)
    if (f_keys_s == nullptr) {
        if ((rc = ensure_feat_capacity(h, nnz))) return rc;
        if ((rc = build_feature_keys(h, indptr, indices, st))) return rc;
        if ((rc = sort_pairs(h, h->feat, nnz, st, h->cub_tmp, h->cub_bytes))) return rc;
        f_keys_s = h->feat.keys_s; f_vals_s = h->feat.vals_s;
    }
    if (h->pending_wait) {
        // multi-GPU: the compact entity tables are being fetched on a side stream (rae_dist_step_begin)
        RAE_CUDA(h, cudaStreamWaitEvent(st, h->pending_wait, 0));
        h->pending_wait = nullptr;
    }
    RAE_PHASE();   // 3 dense / q-dependent operand preparation of the tensor path
    if (h->use_tc) {
        if (prepc_side) RAE_CUDA(h, cudaStreamWaitEvent(st, h->ev_prepc, 0));
        else if ((rc = tc_prepare_c(h, st))) return rc;
        if ((rc = tc_prepare_p(h, a1, a2, st))) return rc;
        RAE_MARK("prep_p", st, 0);
    }
    RAE_PHASE();   // 4 forward contraction: v = M R, w = M^T L, c1, c2
    if (h->use_tc) {
        if ((rc = tc_forward(h, st))) return rc;
    } else {
        if ((rc = launch_bilinear_forward_simt(h, a1, a2, st))) return rc;
    }
    RAE_MARK("contract_forward", st, 0);
    RAE_PHASE();   // 5 scoring / loss / d cost / d score
    if (h->neg_wait) {
        // rae_train_step_host: the negatives were copied on the entity stream, beside the encoder
        RAE_CUDA(h, cudaStreamWaitEvent(st, h->neg_wait, 0));
        h->neg_wait = nullptr;
    }
    if ((rc = launch_score(h, a1, a2, neg1, neg2, neg_ld, st))) return rc;
    RAE_MARK("score", st, 0);
    h->cost_on_event = false;
    if (overlap) {
        // The cost needs the score partials and the pre-update parameters only: it is reduced beside the backward pass
        // (off the critical path) and signalled by its own event, so a caller that wants the number (func['train']
        // returns it) gets it while the rest of the step still runs - the updates stay ordered on the streams.
        RAE_CUDA(h, cudaEventRecord(h->ev_score, st));
        RAE_CUDA(h, cudaStreamWaitEvent(h->s2, h->ev_score, 0));
        if ((rc = launch_cost(h, h->s2))) return rc;
        RAE_CUDA(h, cudaEventRecord(h->ev_cost, h->s2));
        RAE_MARK("cost", h->s2, 2);
        h->cost_on_event = true;
    }
    RAE_PHASE();   // 6 (profiling / no-overlap order only) entity-row update, see below
    RAE_PHASE();   // 7
    RAE_PHASE();   // 8 backward: recompute M c, M^T a
    if (h->use_tc) {
        if ((rc = tc_backward_recompute(h, st))) return rc;
    } else {
        if ((rc = launch_bilinear_backward_simt(h, st))) return rc;
    }
    RAE_MARK("contract_recompute", st, 0);
    RAE_PHASE();   // 9 backward: dq contraction
    if (h->use_tc && (rc = tc_backward_dq(h, st))) return rc;
    RAE_MARK("contract_dq", st, 0);
    RAE_PHASE();   // 10 backward: per-example finish -> dz
    if (h->use_tc && (rc = tc_backward_finish(h, st))) return rc;
    RAE_MARK("backward_finish", st, 0);
    if (overlap) {
        // dz and the per-example vectors are final: the sparse-row updates can start on their own streams
        RAE_CUDA(h, cudaEventRecord(h->ev_fork1, st));
        RAE_CUDA(h, cudaStreamWaitEvent(h->s1, h->ev_fork1, 0));
        RAE_CUDA(h, cudaStreamWaitEvent(h->s2, h->ev_fork1, 0));
        // (each side stream's last mark goes in before its join event, so that the step's "end" mark, recorded behind
        // the joins, is never stamped before it when the side streams finish last)
        if ((rc = launch_entity_update(h, h->ent.keys_s, h->ent.vals_s, n_occ, h->emit_only, !h->emit_only, se))) return rc;
        RAE_MARK("entity_update", h->s1, 1);
        RAE_CUDA(h, cudaEventRecord(h->ev_join1, h->s1));
        if ((rc = launch_w_update(h, f_keys_s, f_vals_s, nnz, emit, !h->emit_only, sw))) return rc;
        RAE_MARK("w_update", h->s2, 2);
        RAE_CUDA(h, cudaEventRecord(h->ev_join2, h->s2));
    }
    RAE_PHASE();   // 11 dense-parameter gradients: dC contraction
    if (h->use_tc) {
        if ((rc = tc_grad_dense(h, st))) return rc;
    } else {
        if ((rc = launch_grad_dense_simt(h, st))) return rc;
    }
    RAE_MARK("contract_dc", st, 0);
    RAE_PHASE();   // 12 sum of the batch-split partials
    // without a regulariser nothing reads the dense parameters between here and their update: the optimiser rule is
    // applied by the same kernel that sums the partials
    if ((rc = launch_dense_finalize(h, st, finish_dense && h->cfg.l1 == 0.0 && h->cfg.l2 == 0.0))) return rc;
    RAE_MARK("dense_finalize", st, 0);
    RAE_PHASE();   // 13 cost (uses the pre-update parameters for the regulariser value); overlapped order: see phase 5.
    // Emit-only: the score part only - rae_dist_step_end adds the regulariser of the own shard and re-runs the cost
    if (!overlap && (rc = launch_cost(h, st))) return rc;
    // emit-only (row-sharded multi-GPU): the tables are per-step compact copies whose every row is touched, so the
    // emitted gradient buffers need no clearing and nothing is applied here (the owner shard applies, rae_pull_apply)
    if (emit && !h->emit_only) {
        if ((rc = launch_zero(h, h->gW_dense, sizeof(float) * (size_t)h->cfg.F * h->K, st))) return rc;
    }
    if (h->debug_dense && !h->emit_only) {
        if ((rc = launch_zero(h, h->gA_dense, sizeof(float) * (size_t)h->cfg.N * h->d, st))) return rc;
        if ((rc = launch_zero(h, h->gAb_dense, sizeof(float) * (size_t)h->cfg.N, st))) return rc;
    }
    if (!overlap) {
        // sparse-row updates in stream order; their phase slots (6, 7) are timed separately below
        if (h->profiling) RAE_CUDA(h, cudaEventRecord(h->ev_upd[0], st));
        if ((rc = launch_entity_update(h, h->ent.keys_s, h->ent.vals_s, n_occ, h->debug_dense || h->emit_only, !h->emit_only, st))) return rc;
        if (h->profiling) RAE_CUDA(h, cudaEventRecord(h->ev_upd[1], st));
        if ((rc = launch_w_update(h, f_keys_s, f_vals_s, nnz, emit, !h->dense_w && !h->emit_only, st))) return rc;
        if (h->profiling) RAE_CUDA(h, cudaEventRecord(h->ev_upd[2], st));
    }
    RAE_PHASE();   // 14 dense-parameter optimiser step
    if (finish_dense && (rc = launch_dense_apply(h, st))) return rc;
    RAE_MARK("dense_apply", st, 0);
    if (overlap) {
        RAE_CUDA(h, cudaStreamWaitEvent(st, h->ev_join1, 0));
        RAE_CUDA(h, cudaStreamWaitEvent(st, h->ev_join2, 0));
    }
    RAE_MARK("end", st, 0);
    RAE_PHASE();   // end
#undef RAE_PHASE
#undef RAE_MARK
    h->stats.nnz = nnz;
    h->stats.entity_occ = n_occ;
    h->stats.kernel_launches = h->launches;
    h->stats.tensor_path = h->use_tc ? 1 : 0;
    h->stats.unique_w_rows = -1;
    h->stats.unique_e_rows = -1;
    h->last_f_keys_s = f_keys_s;
    h->last_f_n = nnz;
    return RAE_OK;
}

static int finish_cost(rae_engine* h, double* cost_host, cudaStream_t st) {
    if (cost_host == nullptr) return RAE_OK;
    if (h->cost_on_event) {
        // the cost kernel stored the value in the pinned word itself; the parameter updates behind it keep running and
        // every later call on this handle is ordered after them by the streams
        RAE_CUDA(h, cudaEventSynchronize(h->ev_cost));
    } else {
        RAE_CUDA(h, cudaStreamSynchronize(st));
    }
    *cost_host = *(volatile double*)h->cost_pinned;
    return RAE_OK;
}

static int check_ready(rae_engine* h, bool need_train_split, bool need_neg) {
    if (!h) return RAE_EINVAL;
    if (!h->params_bound) return fail(h, RAE_ENOTBOUND, "parameters are not bound (rae_bind_params)");
    if (h->adagrad && !h->acc_bound) return fail(h, RAE_ENOTBOUND, "AdaGrad accumulators are not bound (rae_bind_accumulators)");
    if (need_train_split && !h->split[RAE_SPLIT_TRAIN].bound) return fail(h, RAE_ENOTBOUND, "train split is not bound (rae_bind_split)");
    if (need_neg && (h->neg1 == nullptr || h->neg2 == nullptr)) return fail(h, RAE_ENOTBOUND, "epoch negatives are not bound (rae_bind_epoch_negatives)");
    return RAE_OK;
}

int build_feature_cache(rae_engine* h, cudaStream_t st) {
    SplitBinding& sp = h->split[RAE_SPLIT_TRAIN];
    free_feature_cache(h->fcache);
    const int64_t nb = sp.n_rows / h->B;     // trailing partial batch dropped (OieInduction.py:96-98)
    if (nb == 0) return RAE_OK;
    std::vector<int32_t> ip((size_t)nb + 1);
    RAE_CUDA(h, cudaMemcpy2DAsync(ip.data(), sizeof(int32_t), sp.indptr, sizeof(int32_t) * (size_t)h->B, sizeof(int32_t),
                                  (size_t)nb + 1, cudaMemcpyDeviceToHost, st));
    RAE_CUDA(h, cudaStreamSynchronize(st));
    FeatureCache& c = h->fcache;
    c.n_batches = nb;
    c.batch_off = new int64_t[nb + 1];
    int64_t mx = 0;
    for (int64_t b = 0; b <= nb; ++b) {
        c.batch_off[b] = ip[b] - ip[0];
        if (b > 0 && ip[b] - ip[b - 1] > mx) mx = ip[b] - ip[b - 1];
    }
    sp.max_batch_nnz = mx;
    const int64_t used = c.batch_off[nb];
    int rc;
    if ((rc = dev_alloc(h, &c.keys_s, used))) return rc;
    if ((rc = dev_alloc(h, &c.vals_s, used))) return rc;
    if ((rc = ensure_feat_capacity(h, mx))) return rc;
    for (int64_t b = 0; b < nb; ++b) {
        const int64_t n = c.batch_off[b + 1] - c.batch_off[b];
        const int32_t* ipb = sp.indptr + b * h->B;
        if ((rc = build_feature_keys(h, ipb, sp.indices, st))) return rc;
        if ((rc = sort_pairs(h, h->feat, n, st, h->cub_tmp, h->cub_bytes))) return rc;
        RAE_CUDA(h, cudaMemcpyAsync(c.keys_s + c.batch_off[b], h->feat.keys_s, sizeof(uint32_t) * n, cudaMemcpyDeviceToDevice, st));
        RAE_CUDA(h, cudaMemcpyAsync(c.vals_s + c.batch_off[b], h->feat.vals_s, sizeof(uint32_t) * n, cudaMemcpyDeviceToDevice, st));
    }
    RAE_CUDA(h, cudaStreamSynchronize(st));
    c.valid = true;
    return RAE_OK;
}

static bool is_pinned_host(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// Host int32 [S,B] negatives (row strides ld1 / ld2 elements) -> the next half of the double-buffered device staging, on
// stream sc; records ev_neg behind the copy.  The previous step's tail may still read the other half.
int stage_host_negatives(rae_engine* h, const int32_t* neg1_host, int64_t ld1, const int32_t* neg2_host, int64_t ld2,
                         cudaStream_t sc, int32_t** d1_out, int32_t** d2_out) {
    if ((!neg1_host || !neg2_host) && h->S > 0) return fail(h, RAE_EINVAL, "host negatives: null pointer");
    if (h->S > 1 && (ld1 < h->B || ld2 < h->B)) return fail(h, RAE_EINVAL, "host negatives: row stride below B");
    const size_t n = (size_t)h->S * h->B, row = sizeof(int32_t) * (size_t)h->B;
    int32_t* d1 = h->stage_neg + (size_t)h->stage_flip * 2 * n;
    int32_t* d2 = d1 + n;
    h->stage_flip ^= 1;
    *d1_out = d1;
    *d2_out = d2;
    if (n == 0) return RAE_OK;
    h->neg_direct = false;
    if (is_pinned_host(neg1_host) && is_pinned_host(neg2_host)) {
        // page-locked caller memory: strided rows straight to the device, no host staging (the copy reads the CALLER's
        // buffer asynchronously: rae_train_step_host_ld waits for it before returning when no cost read does so already)
        h->neg_direct = true;
        RAE_CUDA(h, cudaMemcpy2DAsync(d1, row, neg1_host, sizeof(int32_t) * (size_t)ld1, row, h->S, cudaMemcpyHostToDevice, sc));
        RAE_CUDA(h, cudaMemcpy2DAsync(d2, row, neg2_host, sizeof(int32_t) * (size_t)ld2, row, h->S, cudaMemcpyHostToDevice, sc));
    } else {
        // the pinned staging buffer is reused: wait until the previous step's copy has left it
        if (h->neg_staged) RAE_CUDA(h, cudaEventSynchronize(h->ev_neg));
        for (int s = 0; s < h->S; ++s) {
            memcpy(h->pinned_neg + (size_t)s * h->B, neg1_host + (size_t)s * ld1, row);
            memcpy(h->pinned_neg + n + (size_t)s * h->B, neg2_host + (size_t)s * ld2, row);
        }
        RAE_CUDA(h, cudaMemcpyAsync(d1, h->pinned_neg, 2 * n * sizeof(int32_t), cudaMemcpyHostToDevice, sc));
        h->neg_staged = true;
    }
    RAE_CUDA(h, cudaEventRecord(h->ev_neg, sc));
    return RAE_OK;
}

}  // namespace rae

using namespace rae;

extern "C" {

int rae_abi_version(void) { return RAE_ABI_VERSION; }

const char* rae_last_error(const rae_engine* h) { return h ? h->err : g_create_err; }

int rae_create(const rae_config* cfg, rae_engine** out) {
    if (out) *out = nullptr;
    if (!cfg || !out) return fail(nullptr, RAE_EINVAL, "rae_create: null argument");
    if (cfg->abi_version != RAE_ABI_VERSION) return fail(nullptr, RAE_EINVAL, "rae_create: ABI version %d != %d", cfg->abi_version, RAE_ABI_VERSION);
    if (cfg->model < RAE_MODEL_A || cfg->model > RAE_MODEL_AC) return fail(nullptr, RAE_EINVAL, "rae_create: unknown model %d", cfg->model);
    if (cfg->optimizer != RAE_OPT_ADAGRAD && cfg->optimizer != RAE_OPT_SGD)
        return fail(nullptr, RAE_EINVAL, "Optimizer '%d' not implemented", cfg->optimizer);   // OieInduction.py:269
    if (cfg->K < 1 || cfg->K > 1024 || cfg->d < 1 || cfg->d > 256 || cfg->S < 0 || cfg->B < 1 || cfg->F < 1 || cfg->N < 1)
        return fail(nullptr, RAE_EINVAL, "rae_create: unsupported sizes K=%d d=%d S=%d B=%d F=%lld N=%lld (need 1<=K<=1024, 1<=d<=256)",
                    cfg->K, cfg->d, cfg->S, cfg->B, (long long)cfg->F, (long long)cfg->N);
    if ((int64_t)(2 + 2 * cfg->S) * cfg->B >= ((int64_t)1 << 31)) return fail(nullptr, RAE_EINVAL, "rae_create: (2+2S)*B too large");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, RAE_ENODEVICE, "no CUDA device available: librae has no CPU fallback");
    }
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, RAE_EINVAL, "rae_create: device %d out of range (%d devices)", cfg->device, ndev);
    rae_engine* h = new (std::nothrow) rae_engine();
    if (!h) return fail(nullptr, RAE_ENOMEM, "out of host memory");
    memset((void*)h, 0, sizeof(*h));
    h->ent = SegWork{}; h->feat = SegWork{}; h->fcache = FeatureCache{};
    for (int i = 0; i < RAE_NUM_SPLITS; ++i) h->split[i] = SplitBinding{};
    h->cfg = *cfg;
    h->K = cfg->K; h->d = cfg->d; h->S = cfg->S; h->B = cfg->B;
    h->dp = (cfg->d + 3) & ~3;
    h->hasM = cfg->model != RAE_MODEL_C;
    h->hasSP = cfg->model != RAE_MODEL_A;
    h->quirk = cfg->model == RAE_MODEL_C && !(cfg->flags & RAE_FLAG_FIX_SP_QUIRK);
    h->adagrad = cfg->optimizer == RAE_OPT_ADAGRAD;
    h->reg = (cfg->l1 != 0.0 || cfg->l2 != 0.0);
    h->debug_dense = (cfg->flags & RAE_FLAG_DENSE_GRADS) != 0;
    h->emit_only = (cfg->flags & RAE_FLAG_EMIT_ONLY) != 0;
    // row-sharded (emit-only): the step emits W's data gradient only; the owner of each shard adds the regulariser to every
    // row of it after the cross-rank sum (rae_shard_apply)
    h->dense_w = h->reg && !h->emit_only;
    h->Z = cfg->z_total > 0 ? (double)cfg->z_total : (double)(4.0 * cfg->B + 2.0 * cfg->B * cfg->S);
#define RAE_CREATE_CUDA(expr)                                                                                  \
    do {                                                                                                       \
        cudaError_t _e = (expr);                                                                               \
        if (_e != cudaSuccess) {                                                                               \
            fail(nullptr, RAE_ECUDA, "%s failed: %s", #expr, cudaGetErrorString(_e));                          \
            rae_destroy(h);                                                                                    \
            return RAE_ECUDA;                                                                                  \
        }                                                                                                      \
    } while (0)
#define RAE_CREATE_RC(expr)                                                                                    \
    do {                                                                                                       \
        int _rc = (expr);                                                                                      \
        if (_rc) {                                                                                             \
            strncpy(g_create_err, h->err, sizeof(g_create_err) - 1);                                           \
            rae_destroy(h);                                                                                    \
            return _rc;                                                                                        \
        }                                                                                                      \
    } while (0)
    RAE_CREATE_CUDA(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    RAE_CREATE_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
    h->num_sms = prop.multiProcessorCount;
    h->coop_launch = prop.cooperativeLaunch != 0;
    h->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    if (prop.major < 10) {
        fail(nullptr, RAE_ENODEVICE, "device %d is sm_%d%d: librae is built for sm_100a only", cfg->device, prop.major, prop.minor);
        rae_destroy(h);
        return RAE_ENODEVICE;
    }
    char why[256];
    if (!simt_supported(h, why, sizeof(why))) {
        fail(nullptr, RAE_EINVAL, "%s", why);
        rae_destroy(h);
        return RAE_EINVAL;
    }
    h->tc = TcState{};
    h->use_tc = false;
    g_pdl_enabled = !(cfg->flags & RAE_FLAG_NO_PDL);
    if (!(cfg->flags & RAE_FLAG_FORCE_SIMT) && tc_supported(h)) {
        RAE_CREATE_RC(tc_init(h));
        h->use_tc = true;
    } else if (cfg->flags & RAE_FLAG_FORCE_TENSOR) {
        fail(nullptr, RAE_EINVAL, "RAE_FLAG_FORCE_TENSOR: the tcgen05 path needs a bilinear model with 16 < d <= 128, K <= 104 and B <= 2^24 (K=%d d=%d B=%d)", cfg->K, cfg->d, cfg->B);
        rae_destroy(h);
        return RAE_EINVAL;
    }
    const size_t BK = (size_t)h->B * h->K;
    RAE_CREATE_RC(dev_alloc(h, &h->q, BK));
    RAE_CREATE_RC(dev_alloc(h, &h->logq, BK));
    RAE_CREATE_RC(dev_alloc(h, &h->dz, BK));
    RAE_CREATE_RC(dev_alloc(h, &h->ev, (size_t)h->B * E_NV * h->dp));
    RAE_CREATE_RC(dev_alloc(h, &h->sc, (size_t)h->B * SC_N));
    RAE_CREATE_RC(dev_alloc(h, &h->gn1, (size_t)h->S * h->B));
    RAE_CREATE_RC(dev_alloc(h, &h->gn2, (size_t)h->S * h->B));
    RAE_CREATE_CUDA(cudaMemset(h->ev, 0, sizeof(float) * (size_t)h->B * E_NV * h->dp));
    RAE_CREATE_CUDA(cudaMemset(h->sc, 0, sizeof(float) * (size_t)h->B * SC_N));
    h->n_loss_part = (h->B + 3) / 4;   // one partial per CTA of k_score (4 examples each)
    RAE_CREATE_RC(dev_alloc(h, &h->loss_part, (size_t)h->n_loss_part));
    h->n_reg_part = 64 * 4;
    RAE_CREATE_RC(dev_alloc(h, &h->reg_part, (size_t)2 * h->n_reg_part));
    RAE_CREATE_RC(dev_alloc(h, &h->cost_dev, 1));
    RAE_CREATE_CUDA(cudaMallocHost((void**)&h->cost_pinned, 4 * sizeof(double)));
    memset(h->cost_pinned, 0, 4 * sizeof(double));
    h->gcost_pinned = h->cost_pinned + 1;                                  // same page-locked block: [cost | global cost | flag | barrier status]
    h->neg_err_pinned = reinterpret_cast<int32_t*>(h->cost_pinned + 2);
    h->peer_err_pinned = reinterpret_cast<int32_t*>(h->cost_pinned + 3);
    h->n_dz_part = h->B;   // upper bound on CTAs of the backward kernel (>= 8 examples per CTA)
    RAE_CREATE_RC(dev_alloc(h, &h->dzsum_part, (size_t)h->n_dz_part * h->K));
    const int64_t dd = h->hasM ? (int64_t)h->d * h->d * h->K : 0, dk = h->hasSP ? (int64_t)h->d * h->K : 0;
    h->off_gC = 0; h->off_gC1 = dd; h->off_gC2 = dd + dk; h->off_gWb = dd + 2 * dk; h->n_dense = dd + 2 * dk + h->K;
    RAE_CREATE_RC(dev_alloc(h, &h->dense_grad, (size_t)h->n_dense));
    {
        const int nunits = (h->hasM ? h->d : 0) + (h->hasSP ? 2 : 0);
        int ns = nunits > 0 ? (2 * h->num_sms + nunits - 1) / nunits : 1;
        const int max_by_batch = (h->B + 63) / 64;
        if (ns > max_by_batch) ns = max_by_batch;
        if (ns < 1) ns = 1;
        if (h->use_tc) ns = h->tc.slots_dc;  // the tensor path deals the batch over slots its own way
        h->gC_nsplit = ns;
        RAE_CREATE_RC(dev_alloc(h, &h->gC_part, (size_t)ns * (size_t)(dd + 2 * dk)));
    }
    if (h->dense_w || h->debug_dense || h->emit_only) RAE_CREATE_RC(dev_alloc(h, &h->gW_dense, (size_t)cfg->F * h->K));
    if (h->debug_dense || h->emit_only) {
        RAE_CREATE_RC(dev_alloc(h, &h->gA_dense, (size_t)cfg->N * h->d));
        RAE_CREATE_RC(dev_alloc(h, &h->gAb_dense, (size_t)cfg->N));
    }
    h->own_gW = h->gW_dense; h->own_gA = h->gA_dense; h->own_gAb = h->gAb_dense; h->own_dense = h->dense_grad;
    const int64_t n_occ = (int64_t)(2 + 2 * h->S) * h->B;
    RAE_CREATE_RC(alloc_segwork(h, h->ent, n_occ, bits_for(cfg->N)));
    RAE_CREATE_RC(ensure_cub(h, n_occ));
    h->ent_cub_bytes = segwork_temp_bytes(n_occ);
    RAE_CREATE_CUDA(cudaMalloc(&h->ent_cub_tmp, h->ent_cub_bytes));
    RAE_CREATE_CUDA(cudaStreamCreateWithFlags(&h->s1, cudaStreamNonBlocking));
    RAE_CREATE_CUDA(cudaStreamCreateWithFlags(&h->s2, cudaStreamNonBlocking));
    RAE_CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_fork0, cudaEventDisableTiming));
    RAE_CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_fork1, cudaEventDisableTiming));
    RAE_CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_join1, cudaEventDisableTiming));
    RAE_CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_join2, cudaEventDisableTiming));
    RAE_CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_prepc, cudaEventDisableTiming));
    RAE_CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_q, cudaEventDisableTiming));
    RAE_CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_qt, cudaEventDisableTiming));
    RAE_CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_dfork, cudaEventDisableTiming));
    RAE_CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_dfetch, cudaEventDisableTiming));
    RAE_CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_score, cudaEventDisableTiming));
    RAE_CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_cost, cudaEventDisableTiming));
    RAE_CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_neg, cudaEventDisableTiming));
    RAE_CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_gcost, cudaEventDisableTiming));
    RAE_CREATE_RC(dev_alloc(h, &h->stage_neg, 4 * (size_t)(h->S > 0 ? h->S : 1) * h->B));
    RAE_CREATE_CUDA(cudaMallocHost((void**)&h->pinned_neg, sizeof(int32_t) * 2 * (size_t)(h->S > 0 ? h->S : 1) * h->B));
    RAE_CREATE_RC(dev_alloc(h, &h->peer_err_dev, 1));
    RAE_CREATE_CUDA(cudaMemset(h->peer_err_dev, 0, sizeof(int32_t)));
    RAE_CREATE_RC(dev_alloc(h, &h->stat_dev, 2));
    RAE_CREATE_CUDA(cudaMemset(h->stat_dev, 0, 2 * sizeof(int32_t)));
    RAE_CREATE_RC(dev_alloc(h, &h->label_dev, (size_t)h->B));
    RAE_CREATE_RC(dev_alloc(h, &h->prob_dev, BK));
#undef RAE_CREATE_CUDA
#undef RAE_CREATE_RC
    *out = h;
    return RAE_OK;
}

void rae_destroy(rae_engine* h) {
    if (!h) return;
    cudaFree(h->q); cudaFree(h->logq); cudaFree(h->dz); cudaFree(h->ev); cudaFree(h->sc); cudaFree(h->gn1); cudaFree(h->gn2);
    cudaFree(h->loss_part); cudaFree(h->reg_part); cudaFree(h->cost_dev); cudaFree(h->dzsum_part); cudaFree(h->own_dense);
    cudaFree(h->gC_part); cudaFree(h->own_gW); cudaFree(h->own_gA); cudaFree(h->own_gAb); cudaFree(h->cub_tmp);
    cudaFree(h->ent_part); cudaFree(h->feat_part); cudaFree(h->stat_dev); cudaFree(h->peer_err_dev);
    cudaFree(h->stage_neg); cudaFree(h->label_dev); cudaFree(h->prob_dev);
    if (h->ev_created) {
        for (int i = 0; i <= RAE_NUM_PHASES; ++i) cudaEventDestroy(h->ev_phase[i]);
        for (int i = 0; i < 3; ++i) cudaEventDestroy(h->ev_upd[i]);
    }
    cudaFree(h->push.w_dev);
    if (h->tl_created) {
        for (int i = 0; i < RAE_TL_MAX; ++i) cudaEventDestroy(h->tl_ev[i]);
    }
    if (h->s1) cudaStreamDestroy(h->s1);
    if (h->s2) cudaStreamDestroy(h->s2);
    if (h->ev_fork0) cudaEventDestroy(h->ev_fork0);
    if (h->ev_fork1) cudaEventDestroy(h->ev_fork1);
    if (h->ev_join1) cudaEventDestroy(h->ev_join1);
    if (h->ev_join2) cudaEventDestroy(h->ev_join2);
    if (h->ev_score) cudaEventDestroy(h->ev_score);
    if (h->ev_cost) cudaEventDestroy(h->ev_cost);
    if (h->ev_neg) cudaEventDestroy(h->ev_neg);
    if (h->ev_gcost) cudaEventDestroy(h->ev_gcost);
    if (h->ev_prepc) cudaEventDestroy(h->ev_prepc);
    if (h->ev_q) cudaEventDestroy(h->ev_q);
    if (h->ev_qt) cudaEventDestroy(h->ev_qt);
    if (h->ev_dfork) cudaEventDestroy(h->ev_dfork);
    if (h->ev_dfetch) cudaEventDestroy(h->ev_dfetch);
    cudaFree(h->ent_cub_tmp);
    if (h->cost_pinned) cudaFreeHost(h->cost_pinned);
    if (h->pinned_neg) cudaFreeHost(h->pinned_neg);
    free_segwork(h->ent);
    free_segwork(h->feat);
    free_feature_cache(h->fcache);
    tc_free(h);
    cudaGetLastError();
    delete h;
}

int rae_bind_params(rae_engine* h, float* W, float* Wb, float* A, float* Ab, float* C, float* C1, float* C2) {
    if (!h) return RAE_EINVAL;
    if (!W || !Wb || !A || !Ab) return fail(h, RAE_EINVAL, "rae_bind_params: W, Wb, A, Ab must be non-null");
    if (h->hasM && !C) return fail(h, RAE_EINVAL, "rae_bind_params: this model needs C (R) [d,d,K]");
    if (h->hasSP && (!C1 || !C2)) return fail(h, RAE_EINVAL, "rae_bind_params: this model needs C1 and C2 [d,K]");
    float* v[RAE_NUM_PARAMS] = {W, Wb, A, Ab, C, C1, C2};
    for (int i = 0; i < RAE_NUM_PARAMS; ++i) h->P[i] = v[i];
    h->params_bound = true;
    return RAE_OK;
}

int rae_bind_accumulators(rae_engine* h, float* W, float* Wb, float* A, float* Ab, float* C, float* C1, float* C2) {
    if (!h) return RAE_EINVAL;
    if (!Wb || (!h->emit_only && (!W || !A || !Ab)))
        return fail(h, RAE_EINVAL, "rae_bind_accumulators: W, Wb, A, Ab must be non-null (W, A, Ab may be NULL with RAE_FLAG_EMIT_ONLY)");
    if (h->hasM && !C) return fail(h, RAE_EINVAL, "rae_bind_accumulators: this model needs C (R) [d,d,K]");
    if (h->hasSP && (!C1 || !C2)) return fail(h, RAE_EINVAL, "rae_bind_accumulators: this model needs C1 and C2 [d,K]");
    float* v[RAE_NUM_PARAMS] = {W, Wb, A, Ab, C, C1, C2};
    for (int i = 0; i < RAE_NUM_PARAMS; ++i) h->ACC[i] = v[i];
    h->acc_bound = true;
    return RAE_OK;
}

int rae_bind_split(rae_engine* h, int32_t split_id, const int32_t* indptr, const int32_t* indices, int64_t n_rows,
                   const int32_t* args1, const int32_t* args2, void* stream) {
    if (!h) return RAE_EINVAL;
    if (split_id < 0 || split_id >= RAE_NUM_SPLITS) return fail(h, RAE_EINVAL, "rae_bind_split: bad split id %d", split_id);
    if (!indptr || !indices || n_rows < 0) return fail(h, RAE_EINVAL, "rae_bind_split: null CSR");
    if (split_id == RAE_SPLIT_TRAIN && (!args1 || !args2)) return fail(h, RAE_EINVAL, "rae_bind_split: the train split needs args1/args2");
    cudaStream_t st = (cudaStream_t)stream;
    SplitBinding& sp = h->split[split_id];
    sp.indptr = indptr; sp.indices = indices; sp.a1 = args1; sp.a2 = args2; sp.n_rows = n_rows;
    int32_t ends[2] = {0, 0};
    RAE_CUDA(h, cudaMemcpyAsync(&ends[0], indptr, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    RAE_CUDA(h, cudaMemcpyAsync(&ends[1], indptr + n_rows, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    RAE_CUDA(h, cudaStreamSynchronize(st));
    sp.nnz = (int64_t)ends[1] - ends[0];
    sp.bound = true;
    if (split_id == RAE_SPLIT_TRAIN) {
        if (!(h->cfg.flags & RAE_FLAG_NO_FEATURE_CACHE)) {
            int rc = build_feature_cache(h, st);
            if (rc) return rc;
        } else {
            free_feature_cache(h->fcache);
        }
    }
    return RAE_OK;
}

int rae_bind_epoch_negatives(rae_engine* h, const int32_t* neg1, const int32_t* neg2, int64_t n_cols) {
    if (!h) return RAE_EINVAL;
    if ((!neg1 || !neg2) && h->S > 0) return fail(h, RAE_EINVAL, "rae_bind_epoch_negatives: null pointer");
    h->neg1 = neg1; h->neg2 = neg2; h->neg_cols = n_cols;
    return RAE_OK;
}

static int train_batch(rae_engine* h, int64_t batch_index, const int32_t* neg1, const int32_t* neg2, int64_t neg_ld,
                       cudaStream_t st) {
    SplitBinding& sp = h->split[RAE_SPLIT_TRAIN];
    const int64_t nb = sp.n_rows / h->B;
    if (batch_index < 0 || batch_index >= nb) return fail(h, RAE_EINVAL, "batch_index %lld out of range [0,%lld)", (long long)batch_index, (long long)nb);
    const int64_t r0 = batch_index * h->B;
    if (h->fcache.valid) {
        const FeatureCache& c = h->fcache;
        const int64_t nnz = c.batch_off[batch_index + 1] - c.batch_off[batch_index];
        return run_step(h, sp.indptr + r0, sp.indices, nnz, sp.a1 + r0, sp.a2 + r0, neg1, neg2, neg_ld,
                        c.keys_s + c.batch_off[batch_index], c.vals_s + c.batch_off[batch_index], st);
    }
    int32_t ends[2];
    RAE_CUDA(h, cudaMemcpyAsync(&ends[0], sp.indptr + r0, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    RAE_CUDA(h, cudaMemcpyAsync(&ends[1], sp.indptr + r0 + h->B, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    RAE_CUDA(h, cudaStreamSynchronize(st));
    return run_step(h, sp.indptr + r0, sp.indices, (int64_t)ends[1] - ends[0], sp.a1 + r0, sp.a2 + r0, neg1, neg2, neg_ld,
                    nullptr, nullptr, st);
}

int rae_train_step(rae_engine* h, int64_t batch_index, double* cost_host, void* stream) {
    int rc = check_ready(h, true, true);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if ((batch_index + 1) * h->B > h->neg_cols) return fail(h, RAE_EINVAL, "batch %lld exceeds the bound negatives (%lld columns)", (long long)batch_index, (long long)h->neg_cols);
    const int64_t c0 = batch_index * h->B;
    if ((rc = train_batch(h, batch_index, h->neg1 + c0, h->neg2 + c0, h->neg_cols, st))) return rc;
    return finish_cost(h, cost_host, st);
}

int rae_train_step_host_ld(rae_engine* h, int64_t batch_index, const int32_t* neg1_host, int64_t ld1, const int32_t* neg2_host,
                           int64_t ld2, double* cost_host, void* stream) {
    int rc = check_ready(h, true, false);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    // Same predicate as run_step's `overlap`: the copy then rides on the entity stream, beside the encoder - its first
    // consumers are the entity keys (same stream) and the scoring kernel (waits for ev_neg).
    const bool side = !h->dense_w && !h->debug_dense && !h->profiling && h->s1 != nullptr;
    int32_t *d1 = nullptr, *d2 = nullptr;
    if ((rc = stage_host_negatives(h, neg1_host, ld1, neg2_host, ld2, side ? h->s1 : st, &d1, &d2))) return rc;
    if (side && h->S > 0) h->neg_wait = h->ev_neg;
    rc = train_batch(h, batch_index, d1, d2, h->B, st);
    h->neg_wait = nullptr;
    if (rc) return rc;
    // the caller may reuse its negative arrays as soon as this returns (the next epoch's sampler does): with a cost read
    // the wait below is implied (the cost follows the scoring kernel, which follows the copy), without one it is explicit
    if (cost_host == nullptr && h->neg_direct && h->S > 0) RAE_CUDA(h, cudaEventSynchronize(h->ev_neg));
    return finish_cost(h, cost_host, st);
}

int rae_train_step_host(rae_engine* h, int64_t batch_index, const int32_t* neg1_host, const int32_t* neg2_host,
                        double* cost_host, void* stream) {
    return rae_train_step_host_ld(h, batch_index, neg1_host, h ? h->B : 0, neg2_host, h ? h->B : 0, cost_host, stream);
}

int rae_train_step_explicit(rae_engine* h, const int32_t* indptr, const int32_t* indices, const int32_t* args1,
                            const int32_t* args2, const int32_t* neg1, const int32_t* neg2, int64_t neg_ld,
                            double* cost_host, void* stream) {
    int rc = check_ready(h, false, false);
    if (rc) return rc;
    if (!indptr || !indices || !args1 || !args2) return fail(h, RAE_EINVAL, "rae_train_step_explicit: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    int32_t ends[2];
    RAE_CUDA(h, cudaMemcpyAsync(&ends[0], indptr, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    RAE_CUDA(h, cudaMemcpyAsync(&ends[1], indptr + h->B, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    RAE_CUDA(h, cudaStreamSynchronize(st));
    if ((rc = run_step(h, indptr, indices, (int64_t)ends[1] - ends[0], args1, args2, neg1, neg2, neg_ld, nullptr, nullptr, st)))
        return rc;
    return finish_cost(h, cost_host, st);
}

int rae_label(rae_engine* h, int32_t split_id, int64_t batch_index, int64_t* labels, float* probs, void* stream) {
    if (!h) return RAE_EINVAL;
    if (!h->params_bound) return fail(h, RAE_ENOTBOUND, "parameters are not bound (rae_bind_params)");
    if (split_id < 0 || split_id >= RAE_NUM_SPLITS || !h->split[split_id].bound) return fail(h, RAE_ENOTBOUND, "split %d is not bound", split_id);
    if (!labels || !probs) return fail(h, RAE_EINVAL, "rae_label: null output");
    SplitBinding& sp = h->split[split_id];
    const int64_t nb = sp.n_rows / h->B;
    if (batch_index < 0 || batch_index >= nb) return fail(h, RAE_EINVAL, "batch_index %lld out of range [0,%lld)", (long long)batch_index, (long long)nb);
    h->launches = 0;
    return launch_encoder_forward(h, sp.indptr + batch_index * h->B, sp.indices, h->B, probs, nullptr, nullptr, labels,
                                  (cudaStream_t)stream);
}

int rae_label_host(rae_engine* h, int32_t split_id, int64_t batch_index, int64_t* labels_host, float* probs_host,
                   void* stream) {
    if (!h) return RAE_EINVAL;
    if (!labels_host || !probs_host) return fail(h, RAE_EINVAL, "rae_label_host: null output");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = rae_label(h, split_id, batch_index, h->label_dev, h->prob_dev, stream);
    if (rc) return rc;
    RAE_CUDA(h, cudaMemcpyAsync(labels_host, h->label_dev, sizeof(int64_t) * h->B, cudaMemcpyDeviceToHost, st));
    RAE_CUDA(h, cudaMemcpyAsync(probs_host, h->prob_dev, sizeof(float) * (size_t)h->B * h->K, cudaMemcpyDeviceToHost, st));
    RAE_CUDA(h, cudaStreamSynchronize(st));
    return RAE_OK;
}

int rae_bind_grad_buffers(rae_engine* h, float* gW, float* gA, float* gAb, float* dense) {
    if (!h) return RAE_EINVAL;
    h->gW_dense = gW ? gW : h->own_gW;
    h->gA_dense = gA ? gA : h->own_gA;
    h->gAb_dense = gAb ? gAb : h->own_gAb;
    h->dense_grad = dense ? dense : h->own_dense;
    return RAE_OK;
}

int64_t rae_dense_grad_size(const rae_engine* h) { return h ? h->n_dense : 0; }

int rae_train_step_begin(rae_engine* h, int64_t batch_index, const int32_t* args1, const int32_t* args2, const int32_t* neg1,
                         const int32_t* neg2, int64_t neg_ld, void* stream) {
    int rc = check_ready(h, true, false);
    if (rc) return rc;
    if (!args1 || !args2 || ((!neg1 || !neg2) && h->S > 0)) return fail(h, RAE_EINVAL, "rae_train_step_begin: null pointer");
    SplitBinding& sp = h->split[RAE_SPLIT_TRAIN];
    const int64_t nb = sp.n_rows / h->B;
    if (batch_index < 0 || batch_index >= nb) return fail(h, RAE_EINVAL, "batch_index %lld out of range [0,%lld)", (long long)batch_index, (long long)nb);
    if (!h->fcache.valid) return fail(h, RAE_EINVAL, "rae_train_step_begin needs the cached feature index (do not set RAE_FLAG_NO_FEATURE_CACHE)");
    const int64_t r0 = batch_index * h->B;
    const FeatureCache& c = h->fcache;
    const int64_t nnz = c.batch_off[batch_index + 1] - c.batch_off[batch_index];
    return run_step(h, sp.indptr + r0, sp.indices, nnz, args1, args2, neg1, neg2, neg_ld, c.keys_s + c.batch_off[batch_index],
                    c.vals_s + c.batch_off[batch_index], (cudaStream_t)stream, false);
}

int rae_copy_cost(rae_engine* h, double* dst_device, void* stream) {
    if (!h || !dst_device) return RAE_EINVAL;
    RAE_CUDA(h, cudaMemcpyAsync(dst_device, h->cost_dev, sizeof(double), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return RAE_OK;
}

int rae_label_shards(rae_engine* h, const void* const* w_shards, int32_t world, const int32_t* indptr,
                     const int32_t* indices, int64_t n_rows, int64_t* labels, float* probs, void* stream) {
    if (!h) return RAE_EINVAL;
    if (!h->params_bound) return fail(h, RAE_ENOTBOUND, "parameters are not bound (rae_bind_params)");
    if (!w_shards || !indptr || !indices || !labels || n_rows < 0) return fail(h, RAE_EINVAL, "rae_label_shards: bad argument");
    h->launches = 0;
    return launch_label_shards(h, w_shards, world, indptr, indices, n_rows, labels, probs, (cudaStream_t)stream);
}

int rae_label_topk(rae_engine* h, const void* const* w_shards, int32_t world, const int32_t* indptr,
                   const int32_t* indices, int64_t n_rows, int32_t k, int32_t* ids, float* probs, void* stream) {
    if (!h) return RAE_EINVAL;
    if (!h->params_bound) return fail(h, RAE_ENOTBOUND, "parameters are not bound (rae_bind_params)");
    if (!w_shards || !indptr || !indices || !ids || n_rows < 0) return fail(h, RAE_EINVAL, "rae_label_topk: bad argument");
    h->launches = 0;
    return launch_label_topk(h, w_shards, world, indptr, indices, n_rows, k, ids, probs, (cudaStream_t)stream);
}

int rae_rank_arguments(rae_engine* h, const int32_t* indptr, const int32_t* indices, const int32_t* args1, const int32_t* args2,
                       int64_t n_rows, int32_t* rank1, int32_t* rank2, void* stream) {
    if (!h) return RAE_EINVAL;
    if (!h->params_bound) return fail(h, RAE_ENOTBOUND, "parameters are not bound (rae_bind_params)");
    if (h->emit_only) return fail(h, RAE_EINVAL, "rae_rank_arguments: an emit-only handle holds compact copies of A, not the model's");
    if (!indptr || !indices || !args1 || !args2 || !rank1 || !rank2 || n_rows < 0)
        return fail(h, RAE_EINVAL, "rae_rank_arguments: bad argument");
    h->launches = 0;
    return launch_rank_arguments(h, indptr, indices, args1, args2, n_rows, rank1, rank2, (cudaStream_t)stream);
}

int rae_predict_arguments(rae_engine* h, const int32_t* indptr, const int32_t* indices, const int32_t* args1,
                          const int32_t* args2, int64_t n_rows, int32_t k, int32_t* ids1, float* scores1, int32_t* ids2,
                          float* scores2, void* stream) {
    if (!h) return RAE_EINVAL;
    if (!h->params_bound) return fail(h, RAE_ENOTBOUND, "parameters are not bound (rae_bind_params)");
    if (h->emit_only) return fail(h, RAE_EINVAL, "rae_predict_arguments: an emit-only handle holds compact copies of A, not the model's");
    if (!indptr || !indices || !args1 || !args2 || !ids1 || !scores1 || !ids2 || !scores2 || n_rows < 0)
        return fail(h, RAE_EINVAL, "rae_predict_arguments: bad argument");
    h->launches = 0;
    return launch_predict_arguments(h, indptr, indices, args1, args2, n_rows, k, ids1, scores1, ids2, scores2,
                                    (cudaStream_t)stream);
}

int rae_train_step_end(rae_engine* h, void* stream) {
    int rc = check_ready(h, false, false);
    if (rc) return rc;
    return launch_dense_apply(h, (cudaStream_t)stream);
}

int rae_read_cost(rae_engine* h, double* cost_host, void* stream) {
    if (!h || !cost_host) return RAE_EINVAL;
    return finish_cost(h, cost_host, (cudaStream_t)stream);
}

int rae_get_probs(rae_engine* h, float* dst, void* stream) {
    if (!h || !dst) return RAE_EINVAL;
    RAE_CUDA(h, cudaMemcpyAsync(dst, h->q, sizeof(float) * (size_t)h->B * h->K, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return RAE_OK;
}

int rae_get_dense_grad(rae_engine* h, int32_t param_id, float* dst, void* stream) {
    if (!h || !dst) return RAE_EINVAL;
    if (!h->debug_dense) return fail(h, RAE_EINVAL, "rae_get_dense_grad needs RAE_FLAG_DENSE_GRADS");
    const float* src = nullptr;
    size_t n = 0;
    switch (param_id) {
        case RAE_P_W: src = h->gW_dense; n = (size_t)h->cfg.F * h->K; break;
        case RAE_P_WB: src = h->dense_grad + h->off_gWb; n = (size_t)h->K; break;
        case RAE_P_A: src = h->gA_dense; n = (size_t)h->cfg.N * h->d; break;
        case RAE_P_AB: src = h->gAb_dense; n = (size_t)h->cfg.N; break;
        case RAE_P_C: if (h->hasM) { src = h->dense_grad + h->off_gC; n = (size_t)h->d * h->d * h->K; } break;
        case RAE_P_C1: if (h->hasSP) { src = h->dense_grad + h->off_gC1; n = (size_t)h->d * h->K; } break;
        case RAE_P_C2: if (h->hasSP) { src = h->dense_grad + h->off_gC2; n = (size_t)h->d * h->K; } break;
        default: break;
    }
    if (!src) return fail(h, RAE_EINVAL, "rae_get_dense_grad: parameter %d is not part of this model", param_id);
    RAE_CUDA(h, cudaMemcpyAsync(dst, src, sizeof(float) * n, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return RAE_OK;
}

int rae_get_entity_segments(rae_engine* h, int32_t* sorted_rows, int32_t* sorted_occ, int32_t* seg_start, int64_t* n_occ,
                            int64_t* n_seg, void* stream) {
    if (!h) return RAE_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = (int64_t)(2 + 2 * h->S) * h->B;
    int32_t ns = 0;
    {
        int rc = segment_heads(h, h->ent.keys_s, n, h->ent, st);
        if (rc) return rc;
    }
    RAE_CUDA(h, cudaMemcpyAsync(&ns, h->ent.n_seg, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    RAE_CUDA(h, cudaStreamSynchronize(st));
    if (sorted_rows) RAE_CUDA(h, cudaMemcpyAsync(sorted_rows, h->ent.keys_s, sizeof(int32_t) * n, cudaMemcpyDeviceToDevice, st));
    if (sorted_occ) RAE_CUDA(h, cudaMemcpyAsync(sorted_occ, h->ent.vals_s, sizeof(int32_t) * n, cudaMemcpyDeviceToDevice, st));
    if (seg_start) RAE_CUDA(h, cudaMemcpyAsync(seg_start, h->ent.seg_start, sizeof(int32_t) * ((size_t)ns + 1), cudaMemcpyDeviceToDevice, st));
    if (n_occ) *n_occ = n;
    if (n_seg) *n_seg = ns;
    return RAE_OK;
}

static const char* kPhaseNames[RAE_NUM_PHASES] = {"encoder_forward", "entity_sort", "feature_sort", "operand_prep", "contract_forward",
                                                   "score", "entity_update", "w_update", "contract_recompute", "contract_dq",
                                                   "backward_finish", "contract_dc", "dense_finalize", "cost", "dense_apply"};

const char* rae_phase_name(int32_t phase) { return (phase >= 0 && phase < RAE_NUM_PHASES) ? kPhaseNames[phase] : ""; }

int rae_set_profiling(rae_engine* h, int32_t on) {
    if (!h) return RAE_EINVAL;
    if (on && !h->ev_created) {
        for (int i = 0; i <= RAE_NUM_PHASES; ++i) RAE_CUDA(h, cudaEventCreate(&h->ev_phase[i]));
        for (int i = 0; i < 3; ++i) RAE_CUDA(h, cudaEventCreate(&h->ev_upd[i]));
        h->ev_created = true;
    }
    if (on == 2 && !h->tl_created) {
        for (int i = 0; i < RAE_TL_MAX; ++i) RAE_CUDA(h, cudaEventCreate(&h->tl_ev[i]));
        h->tl_created = true;
    }
    h->profiling = on == 1;
    h->timeline = on == 2;
    return RAE_OK;
}

int rae_get_timeline(rae_engine* h, char* buf, int64_t len) {
    if (!h || !buf || len <= 0) return RAE_EINVAL;
    buf[0] = 0;
    if (!h->tl_created || h->tl_n == 0) return fail(h, RAE_EINVAL, "rae_get_timeline: no step ran with rae_set_profiling(h, 2)");
    int64_t off = 0;
    for (int i = 0; i < h->tl_n; ++i) {
        RAE_CUDA(h, cudaEventSynchronize(h->tl_ev[i]));
        float ms = 0.f;
        RAE_CUDA(h, cudaEventElapsedTime(&ms, h->tl_ev[0], h->tl_ev[i]));
        const int w = snprintf(buf + off, (size_t)(len - off), "%s %d %.3f\n", h->tl_name[i], h->tl_stream[i], ms * 1e3f);
        if (w < 0 || off + w >= len) break;
        off += w;
    }
    return RAE_OK;
}

int rae_get_phase_times(rae_engine* h, float* ms) {
    if (!h || !ms) return RAE_EINVAL;
    if (!h->ev_created) return fail(h, RAE_EINVAL, "rae_get_phase_times: profiling was never enabled");
    RAE_CUDA(h, cudaEventSynchronize(h->ev_phase[RAE_NUM_PHASES]));
    for (int i = 0; i < RAE_NUM_PHASES; ++i) RAE_CUDA(h, cudaEventElapsedTime(&ms[i], h->ev_phase[i], h->ev_phase[i + 1]));
    // the sparse-row updates run after the cost kernel in the profiled (single-stream) order: their own events
    float eu = 0.f, wu = 0.f;
    RAE_CUDA(h, cudaEventElapsedTime(&eu, h->ev_upd[0], h->ev_upd[1]));
    RAE_CUDA(h, cudaEventElapsedTime(&wu, h->ev_upd[1], h->ev_upd[2]));
    ms[13] -= eu + wu;        // they sit between the cost kernel and the dense update
    ms[6] = eu;
    ms[7] = wu;
    return RAE_OK;
}

int rae_get_step_stats(rae_engine* h, rae_step_stats* out) {
    if (!h || !out) return RAE_EINVAL;
    // unique-row counts live on the device; reading them synchronises, so it happens only here
    int32_t cnt[2] = {0, 0};
    {
        int rc = count_unique(h, h->ent.keys_s, h->stats.entity_occ, h->stat_dev, 0);
        if (rc) return rc;
        if (h->last_f_keys_s && (rc = count_unique(h, h->last_f_keys_s, h->last_f_n, h->stat_dev + 1, 0))) return rc;
        RAE_CUDA(h, cudaMemcpy(cnt, h->stat_dev, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost));
    }
    const int32_t ue = cnt[0], uw = h->last_f_keys_s ? cnt[1] : 0;
    h->stats.unique_e_rows = ue;
    h->stats.unique_w_rows = uw;
    // SURVEY 8(d): fp32 params + fp32 accumulators, int32 ids
    const double rmw = h->adagrad ? 16.0 : 8.0;
    const double B = h->B, S = h->S, K = h->K, d = h->d, nnz = (double)h->stats.nnz;
    const double p_dense = (h->hasM ? d * d * K : 0.0) + (h->hasSP ? 2.0 * d * K : 0.0) + K;
    const double gath = h->hasM ? 4.0 * (2 + 2 * S) * B * (d + 1) : 4.0 * ((1 + 2 * S) * B * (d + 1) + B);
    h->stats.algorithmic_bytes = 4.0 * nnz * K + rmw * uw * K + gath + rmw * ue * (d + 1) + (4.0 + rmw) * p_dense +
                                 4.0 * (nnz + 2 * B + 2 * S * B);
    *out = h->stats;
    return RAE_OK;
}

}  // extern "C"
