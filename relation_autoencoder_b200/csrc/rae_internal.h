// Internal engine state and kernel-launcher declarations (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/rae.h"

namespace rae {

// per-example vector slots in ev[b][slot][dp]
enum EvSlot {
    E_L = 0,    // A[a1]
    E_R = 1,    // A[a2]  (A[a1] for model C with the reference's quirk, SelectionalPreferences.py:35)
    E_V1 = 2,   // fwd: v = M R ; after scoring: v + c1   (gradient direction of neg1 rows)
    E_V2 = 3,   // fwd: w = M^T L ; after scoring: w + c2 (gradient direction of neg2 rows)
    E_C1 = 4,   // c1 = C1 q
    E_C2 = 5,   // c2 = C2 q
    E_A = 6,    // a = gp L + X1
    E_CV = 7,   // c = gp R + Y2
    E_Y2 = 8,   // Y2 = sum_s gn2_s y_s
    E_GA1 = 9,  // d cost / d L
    E_GA2 = 10, // d cost / d R
    E_NV = 11
};
// per-example scalars sc[b][SC_N]
enum ScSlot { SC_GU1 = 0, SC_GU2 = 1, SC_GP = 2, SC_G1 = 3, SC_G2 = 4, SC_ENT = 5, SC_N = 8 };

struct SplitBinding {
    const int32_t* indptr = nullptr;
    const int32_t* indices = nullptr;
    const int32_t* a1 = nullptr;
    const int32_t* a2 = nullptr;
    int64_t n_rows = 0;
    int64_t nnz = 0;
    int64_t max_batch_nnz = 0;
    bool bound = false;
};

// sorted-occurrence workspace (one for entity rows, one for feature rows)
struct SegWork {
    uint32_t* keys = nullptr;      // unsorted keys (row ids)
    uint32_t* vals = nullptr;      // unsorted values (occurrence ids)
    uint32_t* keys_s = nullptr;    // sorted keys
    uint32_t* vals_s = nullptr;    // sorted values (stable)
    int32_t* flags = nullptr;      // segment-head flags
    int32_t* pos = nullptr;        // exclusive scan of flags
    int32_t* seg_start = nullptr;  // [n_seg + 1]
    int32_t* n_seg = nullptr;      // device scalar
    int64_t capacity = 0;
    int key_bits = 32;
};

// feature-side transposed index cached for every batch of the train split
struct FeatureCache {
    uint32_t* keys_s = nullptr;   // [nnz_used] feature ids, sorted within each batch
    uint32_t* vals_s = nullptr;   // [nnz_used] example index within the batch (stable order)
    int64_t* batch_off = nullptr; // host copy: offset of each batch into keys_s / vals_s (= indptr[b*B] - indptr[0])
    int64_t n_batches = 0;
    bool valid = false;
};

// Balanced schedule of the tensor-core contractions (rae_decoder_tc.cu).  The work of a contraction is `ntile` tiles of
// `upt` units each (a unit = one streamed operand chunk / pipeline stage); the T = ntile * upt units are dealt over G
// CTAs in contiguous ranges [start(x), start(x+1)), start(x) = floor(x T / G), so every SM gets the same number of
// MMAs whatever the tile count.  A range is cut at tile boundaries into segments; the segment of CTA x inside tile t
// writes its partial result into slot x - first_cta(t).  G <= T, so every CTA owns at least one unit and the CTAs that
// overlap a tile are consecutive.  G == 0 marks the rectangular layout of the SIMT path (`upt` = uniform slot count).
struct TcSched { int G, upt, ntile; };
__host__ __device__ __forceinline__ long long tcs_start(TcSched s, int x) { return (long long)x * s.upt * s.ntile / s.G; }
// the CTA whose range holds unit u: the largest x with floor(x T / G) <= u
__host__ __device__ __forceinline__ int tcs_cta_of(TcSched s, long long u) {
    const long long T = (long long)s.upt * s.ntile;
    return (int)(((u + 1) * s.G + T - 1) / T) - 1;
}
__host__ __device__ __forceinline__ int tcs_first(TcSched s, int tile) { return tcs_cta_of(s, (long long)tile * s.upt); }
__host__ __device__ __forceinline__ int tcs_nslots(TcSched s, int tile) {
    if (s.G == 0) return s.upt;
    return tcs_cta_of(s, (long long)(tile + 1) * s.upt - 1) - tcs_first(s, tile) + 1;
}

// tensor-core (tcgen05) contraction path state (rae_decoder_tc.cu)
struct TcState {
    bool ready = false;
    int DP = 0;            // columns per row of M, padded: 32 / 64 / 128
    int KH = 0;            // relations padded to a multiple of 16 (kind::f16 MMA depth)
    // operand rows n of Cf = [C rows (i, j) | C1 rows | C2 rows] in half chunks of 64 rows
    int n_bil_rows = 0, n_bil_half = 0, n_sp_half = 0;
    int n_rows_total = 0;  // (n_bil_half + n_sp_half) * 64: reduction length of dq, operand rows of dC
    int n_chunks_fwd = 0;  // 128-row chunks of the forward pass (bilinear + C1/C2 rows, padded to a whole chunk)
    int n_chunks_rec = 0;  // 128-row chunks of the backward recompute pass (bilinear rows only)
    int ntile = 0;         // example tiles of 128
    int fwd_stages = 2;    // B-operand shared-memory stages of the forward kernel
    size_t smem = 0;
    TcSched sch_fwd{}, sch_rec{}, sch_dq{}, sch_dc{}, sch_dc2{};
    int slots_vw = 0, slots_dq = 0, slots_dc = 0;   // partial-result slots per tile (maximum over tiles)
    float4* bop = nullptr; // forward B operand chunks [chunk][hi/lo][KQ][128]
    uint4* pimg = nullptr; // forward / recompute P operand images [tile][hi/lo][KQ][128] (q x 2^12 as FP16 pairs)
    float* vT = nullptr;   // [2][dp][B]            v partials, transposed (lane = example)
    float* wT = nullptr;   // [slots_vw][2][dp][B]  w partials, transposed
    float* spT = nullptr;  // [2][dp][B]            c1, c2, transposed
    uint32_t* scal = nullptr;   // device scalars: |max| words of the FP16 operand scales (rae_decoder_tc.cu: TcScal)
    int NK = 0; size_t smem_dq = 0, smem_dc = 0;
    float4* bop2 = nullptr; // Cf^T chunks [c32][hi/lo][8][NK]
    float* dqT = nullptr;   // [slots_dq][NK][B]  dq partials, transposed
    int n_ntiles = 0, n_bst = 0, dc_nacc = 2, dc_share = 0;   // dC: 128-row tiles, 64-example stages, accumulators, stages per CTA
    bool dc2 = false; int dc_tile0 = 0, dc_tiles = 0; size_t smem_dc2 = 0;   // two-tile FP16 dC kernel on the bilinear rows; tiles left to the one-tile kernel
    float4* pop4 = nullptr; float* Rimg = nullptr; float* Yimg = nullptr;     // its q^T operand and the stage images of R, Y2
    int32_t* tile_slots = nullptr;   // [n_ntiles] partial slots of every 128-row tile of dC (device; k_dense_finalize)
    float4* pop3 = nullptr; // q^T chunks [bc][hi/lo][8][NK]
    float* aT = nullptr; float* LT = nullptr; float* RT = nullptr; float* cT = nullptr; float* Y2T = nullptr;   // [dp][B] views
};

}  // namespace rae

constexpr int RAE_TL_MAX = 48;
struct rae_engine {
    rae_config cfg;
    int K, d, S, B;
    int dp;          // d rounded up to a multiple of 4 (row stride of ev)
    bool hasM, hasSP, quirk, adagrad, debug_dense, emit_only;
    bool reg;        // l1 or l2 != 0: W (and C | C1 | C2 when ext_reg) carry the regulariser
    bool dense_w;    // this handle applies the rule to every element of its own W through a dense dW (reg && !emit_only);
                     // an emit-only handle leaves W's regulariser to the owner's shard pass (rae_shard_apply)
    double Z;        // denominator of the mean
    float* P[RAE_NUM_PARAMS];
    float* ACC[RAE_NUM_PARAMS];
    bool params_bound, acc_bound;
    rae::SplitBinding split[RAE_NUM_SPLITS];
    const int32_t* neg1;
    const int32_t* neg2;
    int64_t neg_cols;

    // scratch (device)
    float* q;        // [B,K]
    float* logq;     // [B,K]
    float* dz;       // [B,K]
    float* ev;       // [B,E_NV,dp]
    float* sc;       // [B,SC_N]
    float* gn1;      // [S,B]
    float* gn2;      // [S,B]
    double* loss_part; int n_loss_part;
    double* reg_part;  int n_reg_part;
    double* cost_dev;  // [1]
    double* cost_pinned;
    float* dzsum_part; int n_dz_part; int dz_part_used;   // [n_dz_part, K]; rows written by the last backward
    float* dense_grad;  // flat [C | C1 | C2 | Wb]
    int64_t off_gC, off_gC1, off_gC2, off_gWb, n_dense;
    bool dense_fused;           // this step's k_dense_finalize applied the optimiser itself (launch_dense_apply has only W left)
    float* gC_part; int gC_nsplit;       // [nsplit, units*d*K]
    // debug / regularised dense gradients of the sparse tables
    float* gW_dense; float* gA_dense; float* gAb_dense;
    float* own_gW; float* own_gA; float* own_gAb; float* own_dense;   // internally allocated versions (freed at destroy)
    rae::SegWork ent, feat;
    float* ent_part; size_t ent_part_cap;     // level-1 partial rows of multi-chunk segments
    float* feat_part; size_t feat_part_cap;
    rae::FeatureCache fcache;
    rae::TcState tc; bool use_tc;
    void* cub_tmp; size_t cub_bytes;
    void* ent_cub_tmp; size_t ent_cub_bytes;      // the entity sort runs on its own stream: own temp storage
    cudaStream_t s1, s2;                           // side streams (entity sort + entity update; W update)
    cudaEvent_t ev_fork0, ev_fork1, ev_join1, ev_join2, ev_prepc, ev_dfork, ev_dfetch, ev_q, ev_qt;
    cudaEvent_t ev_score, ev_cost, ev_neg, ev_gcost;
    double* gcost_pinned;       // multi-GPU: the global cost (sum of the ranks' costs) lands here, behind ev_gcost
    int32_t* neg_err_pinned;    // multi-GPU: set by the check of host negatives against the routing plan
    bool gcost_pending;
    cudaEvent_t neg_wait;       // host-negatives copy in flight on a side stream: the scoring kernel waits for it
    bool cost_on_event;         // the last step recorded ev_cost behind its cost kernel
    bool neg_staged;            // ev_neg has been recorded at least once (pinned_neg may still be in flight)
    bool neg_direct;            // the last host-negatives copy read the caller's page-locked arrays in place
    int stage_flip;             // which half of the double-buffered device staging the next host step fills
    int barrier_epoch, barrier_epoch1; int32_t* peer_err_dev;      // peer-flag barriers issued so far; device status word (timeouts)
    int32_t* peer_err_pinned;                      // page-locked copy of the status word: checked by every rae_dist_* call
    cudaEvent_t pending_wait;                      // if set: the step's main stream waits for it before the decoder reads A
    // explicit-step staging
    int32_t* stage_neg;                          // device [2 (flip)][2 (neg1, neg2)][S,B]
    int32_t* pinned_neg;                         // host pinned [2,S,B]
    int64_t* label_dev; float* prob_dev;         // label_host staging
    // bookkeeping
    rae_step_stats stats;
    bool profiling; cudaEvent_t ev_phase[RAE_NUM_PHASES + 1]; cudaEvent_t ev_upd[3]; bool ev_created;
    // timeline (rae_set_profiling(h, 2)): the step runs with its normal three-stream overlap and an event is recorded behind
    // every kernel group on the stream it ran on -> the real concurrent schedule (rae_get_timeline)
    // row-sharded multi-GPU, gradient PUSH (rae_bind_push_targets): the emit-only row-update kernels store each reduced
    // gradient row straight into its OWNER's receive buffer, region [rank][compact slot] (posted stores over NVLink,
    // overlapping the dense contraction that runs beside them); the owner then applies from local memory
    struct { float** w_dev; float** a_dev; float** ab_dev; int world, rank; int64_t f_cap, n_cap; bool on;
             const int32_t* f_ids; const int32_t* e_ids; } push;
    void* dense_wait;           // cudaEvent_t the next rae_dist_step_end waits for before its dense update (caller's all-reduce)
    bool tl_keep;               // the next run_step appends to the marks recorded by rae_dist_step_begin instead of restarting
    bool timeline; int tl_n; cudaEvent_t tl_ev[RAE_TL_MAX]; const char* tl_name[RAE_TL_MAX]; int tl_stream[RAE_TL_MAX]; bool tl_created;
    const uint32_t* last_f_keys_s; int64_t last_f_n;   // sorted feature keys of the last step (statistics)
    int32_t* stat_dev;   // [2] device scratch for unique-row counts
    int launches;
    int num_sms;
    bool coop_launch;           // the device supports cooperative launches (rae_sort.cu)
    int max_smem_optin;
    char err[512];
};

namespace rae {

// ---- error helpers ----
int fail(rae_engine* h, int code, const char* fmt, ...);
#define RAE_CUDA(h, expr)                                                                          \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            return rae::fail((h), RAE_ECUDA, "%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, \
                             cudaGetErrorString(_e));                                              \
    } while (0)

// ---- encoder (rae_encoder.cu) ----
int launch_encoder_forward(rae_engine* h, const int32_t* indptr, const int32_t* indices, int B, float* q, float* logq,
                           float* sc_ent /* sc + SC_ENT, stride SC_N, may be null */, int64_t* labels, cudaStream_t st);
// the same encoder over n_rows examples whose W is row-sharded over `world` ranks (rae_label_shards); probs may be null
int launch_label_shards(rae_engine* h, const void* const* w_shards, int world, const int32_t* indptr, const int32_t* indices,
                        int64_t n_rows, int64_t* labels, float* probs, cudaStream_t st);
// the k best relations per row of the same encoder (rae_label_topk): ids int32 [n_rows, k], probs [n_rows, k] or null
int launch_label_topk(rae_engine* h, const void* const* w_shards, int world, const int32_t* indptr, const int32_t* indices,
                      int64_t n_rows, int k, int32_t* ids, float* probs, cudaStream_t st);

// ---- decoder, SIMT contraction (rae_decoder_simt.cu) ----
int simt_supported(const rae_engine* h, char* why, size_t n);
int launch_bilinear_forward_simt(rae_engine* h, const int32_t* a1, const int32_t* a2, cudaStream_t st);
int launch_score(rae_engine* h, const int32_t* a1, const int32_t* a2, const int32_t* neg1, const int32_t* neg2,
                 int64_t neg_ld, cudaStream_t st);
int launch_bilinear_backward_simt(rae_engine* h, cudaStream_t st);
int launch_grad_dense_simt(rae_engine* h, cudaStream_t st);

// ---- decoder, tcgen05 contraction (rae_decoder_tc.cu) ----
int tc_supported(const rae_engine* h);
int tc_init(rae_engine* h);
void tc_free(rae_engine* h);
int tc_prepare_c(rae_engine* h, cudaStream_t st);
int tc_prepare_p(rae_engine* h, const int32_t* a1, const int32_t* a2, cudaStream_t st);   // q^T operand + gather L, R
int tc_prepare_qt(rae_engine* h, cudaStream_t st);                                      // q^T operand only
int tc_gather_lr(rae_engine* h, const int32_t* a1, const int32_t* a2, cudaStream_t st);   // L, R only
int tc_forward(rae_engine* h, cudaStream_t st);                                         // v, w, c1, c2 -> ev
int tc_backward_recompute(rae_engine* h, cudaStream_t st);
int tc_backward_dq(rae_engine* h, cudaStream_t st);
int tc_backward_finish(rae_engine* h, cudaStream_t st);
int tc_grad_dense(rae_engine* h, cudaStream_t st);
// rae_rank_arguments: forward in chunks of B rows, query packing, one tcgen05 ranking launch per pass (rae_decoder_tc.cu)
int launch_rank_arguments(rae_engine* h, const int32_t* indptr, const int32_t* indices, const int32_t* a1, const int32_t* a2,
                          int64_t n_rows, int32_t* rank1, int32_t* rank2, cudaStream_t st);
// rae_predict_arguments: the same driver with the top-k epilogue and a merge of the partial lists (rae_decoder_tc.cu)
int launch_predict_arguments(rae_engine* h, const int32_t* indptr, const int32_t* indices, const int32_t* a1, const int32_t* a2,
                             int64_t n_rows, int k, int32_t* ids1, float* scores1, int32_t* ids2, float* scores2,
                             cudaStream_t st);

// ---- sort / segment / updates (rae_update.cu) ----
size_t segwork_temp_bytes(int64_t n);
constexpr int64_t RAE_OWN_SORT_MAX = 1 << 20;
// rae_sort.cu: one cooperative kernel, stable, ceil(key_bits / 8) passes
size_t radix_sort_temp_bytes(int64_t n, int num_sms);
int radix_sort_pairs(rae_engine* h, const uint32_t* keys, const uint32_t* vals, uint32_t* keys_s, uint32_t* vals_s, int64_t n,
                     int key_bits, cudaStream_t st, void* tmp, size_t tmp_bytes);
int radix_sort_entities(rae_engine* h, const int32_t* a1, const int32_t* a2, const int32_t* neg1, const int32_t* neg2,
                        int64_t neg_ld, uint32_t* keys_s, uint32_t* vals_s, int key_bits, cudaStream_t st, void* tmp,
                        size_t tmp_bytes);
// entity occurrences -> h->ent.keys_s / vals_s (rows ascending, equal rows in occurrence order)
int sort_entities(rae_engine* h, const int32_t* a1, const int32_t* a2, const int32_t* neg1, const int32_t* neg2, int64_t neg_ld,
                  cudaStream_t st);
int build_entity_keys(rae_engine* h, const int32_t* a1, const int32_t* a2, const int32_t* neg1, const int32_t* neg2,
                      int64_t neg_ld, cudaStream_t st);
int build_feature_keys(rae_engine* h, const int32_t* indptr, const int32_t* indices, cudaStream_t st);
int sort_pairs(rae_engine* h, SegWork& w, int64_t n, cudaStream_t st, void* tmp, size_t tmp_bytes);   // stable radix sort by row
int segment_heads(rae_engine* h, const uint32_t* keys_s, int64_t n, SegWork& w, cudaStream_t st);   // introspection
int count_unique(rae_engine* h, const uint32_t* keys_s, int64_t n, int32_t* out_dev, cudaStream_t st);
int build_feature_cache(rae_engine* h, cudaStream_t st);
int launch_entity_update(rae_engine* h, const uint32_t* keys_s, const uint32_t* vals_s, int64_t n_occ, bool emit_dense,
                         bool apply, cudaStream_t st);
int launch_w_update(rae_engine* h, const uint32_t* keys_s, const uint32_t* vals_s, int64_t nnz, bool emit_dense,
                    bool apply, cudaStream_t st);
// ---- peer-memory path (rae_peer.cu) ----
int launch_fetch_rows(rae_engine* h, const void* const* tables, int world, int64_t width, const int32_t* ids, int64_t n,
                      float* out, cudaStream_t st);
int launch_pull_apply(rae_engine* h, float* table, float* acc, int64_t width, const int32_t* rows_local, const int32_t* ent_off,
                      const int32_t* ent_src, const int32_t* ent_slot, int64_t n_rows, const void* const* grads, int world,
                      cudaStream_t st);
int launch_shard_apply(rae_engine* h, float* table, float* acc, int64_t width, const int32_t* rows_local, const int32_t* ent_off,
                       const int32_t* ent_src, const int32_t* ent_slot, int64_t n_rows, const void* const* grads, int world,
                       int64_t shard_rows, cudaStream_t st);
int launch_peer_barrier(rae_engine* h, const void* const* flag_bufs, int world, int rank, cudaStream_t st, int kind = 0);
int launch_dense_apply_peers(rae_engine* h, const void* const* dense_bufs, int world, cudaStream_t st, int part = 0);
int launch_dense_finalize(rae_engine* h, cudaStream_t st, bool fuse_apply);  // sum partials -> dense_grad, or (fused) straight into the optimiser rule
int launch_dense_apply(rae_engine* h, cudaStream_t st);     // AdaGrad/SGD on C,C1,C2,Wb (+ W when dense_w)
int stage_host_negatives(rae_engine* h, const int32_t* neg1_host, int64_t ld1, const int32_t* neg2_host, int64_t ld2,
                         cudaStream_t sc, int32_t** d1_out, int32_t** d2_out);   // host [S,B] ids -> device staging, records ev_neg
// deterministic loss reduce + regulariser.  The norms run over the handle's own W (none on an emit-only handle, whose W is
// a compact copy) or, when w_shard is given, over w_elems elements there; the decoder tensors' share is added when
// ext_reg and (not emit-only, or with_dec)
int launch_cost(rae_engine* h, cudaStream_t st, const float* w_shard = nullptr, int64_t w_elems = 0, bool with_dec = false);
int launch_zero(rae_engine* h, void* p, size_t bytes, cudaStream_t st);

}  // namespace rae
