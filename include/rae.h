/*
 * rae.h - C ABI of librae.so: the B200 (sm_100a) implementation of the relation-autoencoder training hot path.
 *
 * Drop-in boundary.  The reference touches its model only through the compiled Theano callables stored in
 * ReconstructInducer.func (learning/OieInduction.py:91):
 *     func['train'](batch_index, neg1[S,B] int32, neg2[S,B] int32) -> cost      (OieInduction.py:146-149)
 *     func['label_<split>'](batch_index) -> (labels int64[B], probs[B,K])       (OieInduction.py:151-155)
 * with the dataset bound once as device-resident "shared" copies sliced by batch_index (make_shared,
 * OieInduction.py:439-449) and the parameters living in theano.shared variables (OieModel.py:50-63).
 * Every entry point below names the reference interface it replaces.
 *
 * Conventions: plain pointers and sizes only (no torch / C++ types); all tensors are C-contiguous with the reference's
 * shapes: W[F,K] Wb[K] A[N,d] Ab[N] C[d,d,K] (= R for model A) C1[d,K] C2[d,K]; parameters and AdaGrad accumulators are
 * fp32 DEVICE buffers owned by the caller and borrowed for the lifetime of the binding; ids are int32; "stream" is a
 * cudaStream_t passed as void* (NULL = legacy default stream).  Every function returns 0 on success or a negative
 * RAE_E* code; rae_last_error() gives the message.  No C++ exception crosses this boundary.  A handle is not
 * thread-safe; work is stream-ordered.
 */
#ifndef RAE_H_
#define RAE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RAE_ABI_VERSION 4

/* decoder selection: construct_decoder(model_type, ...) learning/models/decoders/Decoder.py:84-93 */
#define RAE_MODEL_A 0  /* 'rescal'    Bilinear.py               */
#define RAE_MODEL_C 1  /* 'sp'        SelectionalPreferences.py */
#define RAE_MODEL_AC 2 /* 'rescal+sp' BilinearPlusSP.py         */

/* optimiser selection: _initialize_optimization_algorithm, OieInduction.py:261-269 */
#define RAE_OPT_ADAGRAD 0 /* Optimizers.py:6-33  */
#define RAE_OPT_SGD 1     /* Optimizers.py:36-52 */

/* parameter ids (rae_get_dense_grad) */
#define RAE_P_W 0
#define RAE_P_WB 1
#define RAE_P_A 2
#define RAE_P_AB 3
#define RAE_P_C 4
#define RAE_P_C1 5
#define RAE_P_C2 6
#define RAE_NUM_PARAMS 7

/* split ids: settings.py:26 split_labels = ['train', 'valid', 'test'] */
#define RAE_SPLIT_TRAIN 0
#define RAE_SPLIT_VALID 1
#define RAE_SPLIT_TEST 2
#define RAE_NUM_SPLITS 3

/* error codes */
#define RAE_OK 0
#define RAE_EINVAL (-1)      /* bad argument / unsupported shape */
#define RAE_ECUDA (-2)       /* CUDA runtime error (message holds cudaGetErrorString) */
#define RAE_ENOTBOUND (-3)   /* parameters / split / negatives not bound yet */
#define RAE_ENOMEM (-4)
#define RAE_ENODEVICE (-5)   /* no CUDA device: there is NO CPU fallback */

/* flags for rae_config.flags */
#define RAE_FLAG_FIX_SP_QUIRK 1u    /* use A[args2] on the right side of model C (SelectionalPreferences.py:35 uses args1) */
#define RAE_FLAG_DENSE_GRADS 2u     /* also materialise dense gradients every step (parity tests; rae_get_dense_grad) */
#define RAE_FLAG_FORCE_SIMT 4u      /* never take the tcgen05 contraction path */
#define RAE_FLAG_FORCE_TENSOR 8u    /* fail instead of falling back when the tcgen05 path does not support the shape */
#define RAE_FLAG_NO_FEATURE_CACHE 16u /* re-sort the batch's (feature, example) pairs every step instead of once at bind */
#define RAE_FLAG_CLUSTER_MULTICAST 64u /* accepted and ignored: the cluster-multicast variant of the tcgen05 path measured no gain on
                                         * B200 (the kernels are not operand-traffic bound) and was removed */
#define RAE_FLAG_NO_PDL 128u        /* launch the step's kernels in plain stream order (no programmatic dependent launch): A/B measurements */
#define RAE_FLAG_EMIT_ONLY 32u      /* row-sharded multi-GPU: W/A/Ab are per-step compact copies; emit per-row data gradients, apply
                                      * nothing (with l1/l2 != 0 the owner adds W's regulariser, rae_shard_apply) */

typedef struct rae_config {
    int32_t abi_version; /* RAE_ABI_VERSION */
    int32_t model;       /* RAE_MODEL_*                                   OieInduction.py:475 --decoder     */
    int32_t K;           /* relations  m                                  OieInduction.py:469 --relations   */
    int32_t d;           /* embed size r                                  OieInduction.py:468 --embed-size  */
    int32_t S;           /* negatives per side s                          OieInduction.py:470 --neg-samples */
    int32_t B;           /* LOCAL batch size l (rows this handle processes per step)  :467 --batch-size     */
    int64_t F;           /* feature-space dimensionality (rows of W)      OieData.py:96-98                  */
    int64_t N;           /* entity vocabulary (rows of A)                 OieData.py:92-94                  */
    int32_t optimizer;   /* RAE_OPT_*                                     OieInduction.py:473               */
    int32_t ext_reg;     /* regularise decoder weights too                OieModel.py:60-62                 */
    uint32_t flags;      /* RAE_FLAG_*                                                                      */
    int32_t device;      /* CUDA device ordinal                                                              */
    double lr;           /* learning rate                                 OieInduction.py:466               */
    double l1, l2;       /* lambda_1, lambda_2                            OieInduction.py:471-472           */
    double alpha;        /* entropy scale                                 OieModel.py:81                    */
    double adj;          /* batch_size / N_train                          OieInduction.py:131               */
    int64_t z_total;     /* denominator of the mean, 4B+2BS of the GLOBAL batch (OieModel.py:90); 0 = derive from B,S */
} rae_config;

typedef struct rae_engine rae_engine; /* opaque */

typedef struct rae_step_stats {
    int64_t nnz;            /* feature occurrences in the step's batch                     */
    int64_t unique_w_rows;  /* U_W: distinct rows of W touched                             */
    int64_t unique_e_rows;  /* U_E: distinct rows of A/Ab touched                          */
    int64_t entity_occ;     /* (2+2S)*B                                                    */
    int32_t kernel_launches;/* kernels launched by the step (ours + CUB passes)            */
    int32_t tensor_path;    /* 1 if the tcgen05 contraction ran, 0 for the SIMT contraction */
    double algorithmic_bytes; /* SURVEY 8(d) bytes model evaluated with the step's U_W / U_E */
} rae_step_stats;

/* ---- lifetime ------------------------------------------------------------------------------------------- */
/* replaces ReconstructInducer.__init__ + compile_function (OieInduction.py:28-101,118-155): sizes scratch, streams. */
int rae_create(const rae_config* cfg, rae_engine** out);
void rae_destroy(rae_engine* h);
/* message of the last failing call on this handle (h may be NULL: message of the last failing rae_create) */
const char* rae_last_error(const rae_engine* h);
int rae_abi_version(void);

/* ---- bindings ------------------------------------------------------------------------------------------- */
/* theano.shared parameters (RelationClassifier.py:24-25, Bilinear.py:15-17, SelectionalPreferences.py:16-19,
 * BilinearPlusSP.py:19-23).  Pointers a model does not use may be NULL (C for model C; C1,C2 for model A). */
int rae_bind_params(rae_engine* h, float* W, float* Wb, float* A, float* Ab, float* C, float* C1, float* C2);
/* AdaGrad accumulators, one per parameter, same shapes (Optimizers.py:12-15).  Ignored for SGD. */
int rae_bind_accumulators(rae_engine* h, float* W, float* Wb, float* A, float* Ab, float* C, float* C1, float* C2);
/* make_shared(DatasetSplit) (OieInduction.py:439-449; OieData.py:72-90): binary CSR (data implied 1.0) + args.
 * For the train split this also builds the per-batch (feature -> examples) transposed index used by the W update. */
int rae_bind_split(rae_engine* h, int32_t split_id, const int32_t* indptr, const int32_t* indices, int64_t n_rows,
                   const int32_t* args1, const int32_t* args2, void* stream);
/* the epoch's negative ids, row-major [S, n_cols] (NegativeExampleGenerator.py:24; OieInduction.py:183-184);
 * batch b uses columns [b*B, (b+1)*B) (OieInduction.py:187-188) - read strided in place, no per-batch copy. */
int rae_bind_epoch_negatives(rae_engine* h, const int32_t* neg1, const int32_t* neg2, int64_t n_cols);

/* ---- func['train'] -------------------------------------------------------------------------------------- */
/* device-resident form: rows [b*B,(b+1)*B) of the bound train split + bound epoch negatives.  cost_host may be NULL
 * (fully asynchronous); otherwise the call waits until the regularised batch cost is known and stores it.  The cost
 * depends on the forward pass only: the call may return while the backward pass and the parameter updates of this
 * step are still running - every later call on the handle (and rae_destroy) is ordered after them. */
int rae_train_step(rae_engine* h, int64_t batch_index, double* cost_host, void* stream);
/* drop-in form of func['train'](batch_index, neg1, neg2): neg1/neg2 are HOST int32[S,B] (what learn() passes,
 * OieInduction.py:187-189); copies them to the device, runs the step, returns the cost (same ordering as above; the
 * host arrays have been consumed when the call returns). */
int rae_train_step_host(rae_engine* h, int64_t batch_index, const int32_t* neg1_host, const int32_t* neg2_host,
                        double* cost_host, void* stream);
/* same with a row stride (in elements) per array: the driver passes column slices neg[:, b*B:(b+1)*B] of the epoch's
 * [S, n] arrays (OieInduction.py:187-188), which are read in place.  Page-locked host memory is copied straight to the
 * device (one strided DMA per array); pageable memory goes through the handle's pinned staging buffer. */
int rae_train_step_host_ld(rae_engine* h, int64_t batch_index, const int32_t* neg1_host, int64_t ld1,
                           const int32_t* neg2_host, int64_t ld2, double* cost_host, void* stream);
/* fully explicit form for parity tests with injected indices: all DEVICE pointers; indptr has B+1 entries and may
 * start at any offset into indices (indices is indexed by indptr values); neg_ld = row stride of neg1/neg2. */
int rae_train_step_explicit(rae_engine* h, const int32_t* indptr, const int32_t* indices, const int32_t* args1,
                            const int32_t* args2, const int32_t* neg1, const int32_t* neg2, int64_t neg_ld,
                            double* cost_host, void* stream);

/* ---- multi-GPU building blocks (SURVEY 8e): the reference has no counterpart (single process, no device) ----------
 * The row-sharded step of the peer-memory path below (relation_autoencoder_b200/dist.py) binds a rank's compact gradient
 * buffers and flat dense gradient with rae_bind_grad_buffers and runs its local step as rae_train_step_begin, then
 * rae_train_step_end around the dense-gradient all-reduce.  It copies the local cost for the cross-rank sum with
 * rae_copy_cost and labels a split's rows straight from the owners' W shards with rae_label_shards. */
/* caller-owned output buffers for the emitted gradients: gW[F,K], gA[N,d], gAb[N] (F, N = compact capacities) and the
 * flat dense gradient [C | C1 | C2 | Wb] (rae_dense_grad_size floats).  NULL keeps the internal buffer. */
int rae_bind_grad_buffers(rae_engine* h, float* gW, float* gA, float* gAb, float* dense);
int64_t rae_dense_grad_size(const rae_engine* h);
int rae_train_step_end(rae_engine* h, void* stream);
/* synchronise and read the last step's (local) cost */
int rae_read_cost(rae_engine* h, double* cost_host, void* stream);

/* ---- peer-memory data path over NVLink / NVSwitch (one process per GPU, one node) ----------------------------------
 * The sharded tables and the per-rank compact gradient buffers live in cudaMalloc'ed memory exported with CUDA IPC, so a
 * rank's kernels read its peers' rows DIRECTLY (no collective in the sparse data path): rae_fetch_rows gathers the rows a
 * batch touches from their owner shards into the rank's compact tables; after the step (RAE_FLAG_EMIT_ONLY) and the
 * dense all-reduce, rae_pull_apply lets every OWNER read the reduced gradient rows of its rows from all ranks' compact
 * gradient buffers, sum them in rank order (deterministic) and apply the optimiser once per row.  The routing (which
 * rows, which slots) depends only on the ids and is planned once per split / epoch by the host side. */
#define RAE_MAX_PEERS 16
#define RAE_FLAG_WORDS 64      /* a rank's flag buffer: RAE_MAX_PEERS barrier epochs, its local cost (double), padding to 32; a second
                                * barrier sequence (the side stream's "A, Ab and dense parameters applied") in words [32, 32 + RAE_MAX_PEERS) */
#define RAE_IPC_HANDLE_BYTES 64
/* zero-initialised device allocation + its IPC handle (handle_out: RAE_IPC_HANDLE_BYTES bytes, may be NULL) */
int rae_peer_alloc(int64_t bytes, void** ptr_out, void* handle_out);
int rae_peer_free(void* ptr);
/* map a peer process's allocation into this process (enables peer access lazily) / unmap it */
int rae_peer_open(const void* handle, void** ptr_out);
int rae_peer_close(void* ptr);
/* out[i, :] = tables[ids[i] % world][(ids[i] / world) * width ...]   (tables: HOST array of `world` device pointers, the
 * row-sharded table of every rank, own shard included; ids: device int32 global row ids) */
int rae_fetch_rows(rae_engine* h, const void* const* tables, int32_t world, int64_t width, const int32_t* ids, int64_t n,
                   float* out, void* stream);
/* owner-side update of n_rows rows of `table` (local row indices rows_local[i]): g = sum over e in
 * [ent_off[i], ent_off[i+1]) - in that order - of grads[ent_src[e]][ent_slot[e] * width ...], then the handle's optimiser
 * rule (Optimizers.py:29-32 / :51) on table / acc.  grads: HOST array of `world` device pointers (every rank's compact
 * gradient buffer of this table). */
int rae_pull_apply(rae_engine* h, float* table, float* acc, int64_t width, const int32_t* rows_local, const int32_t* ent_off,
                   const int32_t* ent_src, const int32_t* ent_slot, int64_t n_rows, const void* const* grads, int32_t world,
                   void* stream);
/* rae_pull_apply over EVERY row of a regularised table shard (shard_rows rows, local indices 0..shard_rows-1): for each
 * element, in the order of the single-GPU dense update, g = the summed contributions when the row is in rows_local
 * (ascending) else 0, then g += adj*(l1*sgn(p) + 2*l2*p) with the handle's adj / l1 / l2, then the optimiser rule - one
 * read-modify-write of table and acc per element.  Rows no rank touched move too: the regulariser reaches every row. */
int rae_shard_apply(rae_engine* h, float* table, float* acc, int64_t width, const int32_t* rows_local, const int32_t* ent_off,
                    const int32_t* ent_src, const int32_t* ent_slot, int64_t n_rows, const void* const* grads, int32_t world,
                    int64_t shard_rows, void* stream);
/* first part of a step on batch `batch_index` of the BOUND train split (cached transposed feature index) with explicit
 * device entity ids: args1/args2 [B], neg1/neg2 [S, neg_ld]: everything except the dense-parameter optimiser update, which
 * is left to rae_train_step_end (the flat dense gradient is complete when the stream reaches this point). */
int rae_train_step_begin(rae_engine* h, int64_t batch_index, const int32_t* args1, const int32_t* args2, const int32_t* neg1,
                         const int32_t* neg2, int64_t neg_ld, void* stream);
/* One row-sharded data-parallel step as TWO calls around the caller's dense-gradient all-reduce (everything the host
 * side would otherwise issue one by one; the descriptor of a batch is built once per plan and reused every epoch):
 *   rae_dist_step_begin : rae_fetch_rows for W / A / Ab into the compact tables, then rae_train_step_begin;
 *   [caller: all-reduce of the flat dense gradient]
 *   rae_dist_step_end   : rae_train_step_end, rae_pull_apply for W / A / Ab on the own shards, rae_copy_cost.
 * All pointers are device pointers except the six HOST arrays of `world` device pointers. */
typedef struct rae_dist_step {
    int32_t world;
    int32_t reserved;
    const void* const* w_shards;  const void* const* a_shards;  const void* const* ab_shards;   /* every rank's table shard   */
    const void* const* gw_bufs;   const void* const* ga_bufs;   const void* const* gab_bufs;    /* every rank's compact grads */
    float* Wc; float* Ac; float* Abc;                      /* this rank's compact tables (bound as the engine's W / A / Ab) */
    const int32_t* f_ids; int64_t n_f;                     /* distinct global feature rows of the batch, ascending          */
    const int32_t* e_ids; int64_t n_e;                     /* distinct global entity rows of the batch, ascending           */
    int64_t batch_index;
    const int32_t* a1c; const int32_t* a2c; const int32_t* n1c; const int32_t* n2c; int64_t neg_ld;   /* compact entity slots */
    float* W; float* accW; float* A; float* accA; float* Ab; float* accAb;                     /* own shards + accumulators */
    const int32_t* fr_rows; const int32_t* fr_off; int64_t n_fr; const int32_t* f_src; const int32_t* f_slot;
    const int32_t* er_rows; const int32_t* er_off; int64_t n_er; const int32_t* e_src; const int32_t* e_slot;
    double* cost_dev;                                      /* receives the local cost (device)                              */
    /* peer-memory synchronisation (optional: flag_bufs == NULL -> the caller orders the ranks with collectives) */
    const void* const* flag_bufs;                          /* every rank's flags, int32[RAE_MAX_PEERS] (RAE_FLAG_WORDS w/ cost) */
    const void* const* dense_bufs;                         /* every rank's flat dense gradient [C | C1 | C2 | Wb], or NULL:   */
    int32_t rank;                                          /*   NULL = the caller all-reduced the dense gradient itself      */
    int32_t global_cost;                                   /* 1: flag buffers are int32[RAE_FLAG_WORDS]; the ranks' costs are  */
                                                           /*    summed in rank order (cost_dev, rae_dist_read_cost)           */
    int64_t w_rows;                                        /* rows of this rank's W shard, len(range(rank, F, world)); read    */
} rae_dist_step;                                           /*    only by a regularised handle (l1 or l2 != 0)                  */
/* With flag_bufs set, rae_dist_step_end runs: barrier ("every rank has emitted") -> dense update, summing the ranks'
 * dense gradients straight from dense_bufs in rank order when given -> the three pulls -> barrier ("every owner has
 * applied").  The barrier is a one-warp kernel: release-store of the epoch into every peer's flag word, acquire-spin on the
 * own flags (bounded: a rank that never arrives sets the status word instead of hanging the GPU, see rae_peer_status).
 * Regularised handle (l1 or l2 != 0, OieModel.py:54-62): before the first barrier the local cost gets adj*(l1*L1 + l2*L2)
 * of the pre-update W shard (w_rows rows at W) and, on rank 0 with ext_reg, of C | C1 | C2; the dense update adds the
 * decoder tensors' regulariser term to the summed gradient; and W is applied by rae_shard_apply over the whole shard
 * instead of pulled row by row. */
/* Gradient push (optional, once after rae_create with RAE_FLAG_EMIT_ONLY): gw / ga / gab are HOST arrays of `world` device
 * pointers to every rank's RECEIVE buffers, float [world][f_cap][K], [world][n_cap][d], [world][n_cap].  From then on the
 * step's row-update kernels store the reduced gradient row of compact slot j (global row id = f_ids[j] / e_ids[j] of the
 * rae_dist_step) into the buffer of rank id % world at region [rank][j] instead of this rank's own compact buffer, and the
 * gw_bufs / ga_bufs / gab_bufs of rae_dist_step must then be the `world` regions of THIS rank's receive buffers (local
 * pointers): rae_dist_step_end applies from local memory.  The remote traffic becomes posted stores issued beside the
 * dense-gradient contraction instead of loads on the critical path behind the barrier. */
int rae_bind_push_targets(rae_engine* h, const void* const* gw, const void* const* ga, const void* const* gab, int32_t world,
                          int32_t rank, int64_t f_cap, int64_t n_cap);
/* dense_bufs == NULL (the caller all-reduces the dense gradient): `event` (a cudaEvent_t recorded behind that all-reduce, on
 * any stream) is waited for by the NEXT rae_dist_step_end right before its dense update - so the all-reduce may run beside
 * the barrier and the sparse-row applies instead of in front of them.  Consumed by that call. */
int rae_dist_set_dense_wait(rae_engine* h, void* event);
int rae_dist_step_begin(rae_engine* h, const rae_dist_step* d, void* stream);
int rae_dist_step_end(rae_engine* h, const rae_dist_step* d, void* stream);
/* func['train'](batch_index, neg1, neg2) form of rae_dist_step_begin: this rank's HOST negatives int32[S,B] with row strides
 * (as rae_train_step_host_ld) are copied to the device and checked against the planned compact slots
 * (e_ids[n1c[s,j]] == neg1[s,j]); a mismatch is reported by rae_dist_read_cost.  The step itself runs on the plan. */
int rae_dist_step_begin_host(rae_engine* h, const rae_dist_step* d, const int32_t* neg1_host, int64_t ld1,
                             const int32_t* neg2_host, int64_t ld2, void* stream);
/* global_cost = 1: every rank stores its local cost in words [RAE_MAX_PEERS, RAE_MAX_PEERS+2) of its flag buffer before the
 * first barrier; after it each rank sums them in rank order (no collective).  rae_dist_read_cost waits for that sum only -
 * the pulls and the second barrier of the step keep running behind it - and returns RAE_EINVAL if a host-negatives check
 * failed since the last call. */
int rae_dist_read_cost(rae_engine* h, double* cost_host);
/* stand-alone barrier over the ranks' flag buffers (same kernel as inside rae_dist_step_end) */
int rae_peer_barrier(rae_engine* h, const void* const* flag_bufs, int32_t world, int32_t rank, void* stream);
/* synchronises and returns 0 if every peer barrier of this handle completed, RAE_ECUDA if one timed out */
int rae_peer_status(rae_engine* h, void* stream);
/* copy the last step's (local) cost into a DEVICE double (no synchronisation) */
int rae_copy_cost(rae_engine* h, double* dst_device, void* stream);
/* func['label_<split>'] over n_rows rows of a split whose W is row-sharded over `world` ranks: row f of W is
 * w_shards[f % world] + (f / world) * K (w_shards: HOST array of `world` device pointers, own shard included; world = 1
 * with the handle's bound W is the single-table case).  indices are GLOBAL feature ids; indptr has n_rows+1 entries and
 * may start at any offset; n_rows is NOT bounded by B.  Wb is the handle's bound Wb.  labels int64[n_rows] (first max
 * wins); probs [n_rows, K] or NULL (not written).  The sums run in CSR order, as in rae_label: labels and probs are
 * bit-identical to those of a single-GPU handle holding the gathered W.
 * Ordering: the kernel runs on `stream`, the caller's stream of the sharded step.  There rae_dist_step_end ends with the
 * "every owner has applied" barrier, so the labels see the last step's W on every rank.  The next step cannot overtake
 * the read either: its W applies sit behind its barrier A ("every rank has emitted"), which every rank issues on its
 * caller stream behind this kernel. */
int rae_label_shards(rae_engine* h, const void* const* w_shards, int32_t world, const int32_t* indptr,
                     const int32_t* indices, int64_t n_rows, int64_t* labels, float* probs, void* stream);
/* func['label_<split>'] with the k most probable relations per row instead of the argmax (RelationClassifier.py:39-48;
 * the posteriors of OieInduction.py:240-250 without materialising [n_rows, K]).  W lookup, CSR conventions, n_rows and
 * stream ordering exactly as rae_label_shards (world = 1 with the handle's bound W is the single-table case).
 * ids int32 [n_rows, k], row-major: the k highest-scoring relations, score descending, equal scores by ascending relation
 * id (so ids[:, 0] are rae_label_shards' labels).  probs [n_rows, k] or NULL (not written): their softmax probabilities,
 * bit-identical to rae_label_shards' probs[i, ids[i, j]].  1 <= k <= min(K, RAE_MAX_TOPK); k, world or a null shard out
 * of range return RAE_EINVAL before any launch; n_rows = 0 launches nothing. */
#define RAE_MAX_TOPK 16
int rae_label_topk(rae_engine* h, const void* const* w_shards, int32_t world, const int32_t* indptr,
                   const int32_t* indices, int64_t n_rows, int32_t k, int32_t* ids, float* probs, void* stream);
/* Argument prediction: rank every row's true arguments against all N entities under the bound model (no gold relation
 * labels needed).  For row i with posterior q (RelationClassifier.py:39-48; a row without features scores Wb alone) and
 * the decoder's vectors v = M A[args2], w = M^T A[args1], M = sum_r q_r C[:,:,r], c1 = C1 q, c2 = C2 q (v = w = 0 for
 * model C, c1 = c2 = 0 for model A; Bilinear.py:33,58-59, SelectionalPreferences.py:31-32, BilinearPlusSP.py:35-37,68-72),
 * the candidate scores of the reference's negative samples (Bilinear.py:36,47 and their SP / A+SP counterparts) are
 *   slot 1 (x replaces args1): s1(x) = A[x].(v + c1) + Ab[x],   slot 2 (x replaces args2): s2(x) = A[x].(w + c2) + Ab[x]
 * up to terms that do not depend on x, and rank_s[i] = 1 + #{x in [0, N), x != true_s : s_s(x) > s_s(true_s)}.  The true
 * argument is scored by the same formula as every other entity: for model C under the args1 quirk of
 * SelectionalPreferences.py:35 the slot-2 positive term of the cost never reads A[args2], so the slot-2 threshold is not
 * the cost's u2; RAE_FLAG_FIX_SP_QUIRK changes only x-independent terms and so no rank.  Scores are fp32-accurate (FP16
 * pair split on the tensor cores); an entity whose score ties the true one within rounding may count either way.
 * indptr / indices / args1 / args2 follow rae_label_shards: device arrays, indptr has n_rows+1 entries and may start at
 * any offset, indices are feature ids into the bound W; rank1 / rank2 int32 [n_rows] (device).  n_rows is NOT bounded by
 * B; n_rows = 0 launches nothing.  Unbound parameters, an emit-only handle, null pointers or n_rows < 0 are refused
 * before any launch.  Ids are not range-checked here (Engine.rank_arguments checks them on the host).
 * The call runs the forward pass in chunks of B rows through the handle's per-batch scratch: afterwards rae_get_probs
 * returns the posteriors of the last chunk, not those of the last training step.  It allocates (stream-ordered) a
 * workspace of about 512 * N * ceil16(d) bytes for the scaled FP16 image of A plus the query images of up to 131072 rows. */
int rae_rank_arguments(rae_engine* h, const int32_t* indptr, const int32_t* indices, const int32_t* args1,
                       const int32_t* args2, int64_t n_rows, int32_t* rank1, int32_t* rank2, void* stream);
/* Argument prediction: the k most likely entities of each argument slot of every row, with the candidate scores s1 / s2 of
 * rae_rank_arguments (the fp32 value that call compares with its threshold).  ids1 / ids2 int32 [n_rows, k] and
 * scores1 / scores2 float [n_rows, k] (device, row-major): per row and slot the k entities of [0, N) with the highest
 * score, score descending, equal scores by ascending entity id.  The true argument is not excluded: its position in the
 * list, if any, shows where it landed.  The scores are the x-dependent part of the decoder's negative-sample score, so
 * they order a row's candidates exactly but are not comparable across rows.
 * A slot's list never reads the argument it predicts: slot 1 depends on the posterior and A[args2] only, slot 2 on the
 * posterior and A[args1] only (model C: on the posterior only), bit for bit, so a caller may pass any valid id (e.g. 0)
 * for an argument that is unknown and predict it.  The lists do not depend on how the candidates are split over the SMs.
 * CSR, n_rows, stream, scratch and ordering conventions as rae_rank_arguments; 1 <= k <= min(N, RAE_MAX_TOPK).
 * Unbound parameters, an emit-only handle, null pointers, n_rows < 0 or k out of range are refused before any launch;
 * n_rows = 0 launches nothing.  Workspace: that of rae_rank_arguments plus the partial top-kt lists (kt = k rounded up
 * to a power of two), 2 x kt x 8 bytes per query and candidate range: at most about 67 MB (2 x 131072 queries x 2 x
 * 16 x 8 B) on top of what ranking allocates. */
int rae_predict_arguments(rae_engine* h, const int32_t* indptr, const int32_t* indices, const int32_t* args1,
                          const int32_t* args2, int64_t n_rows, int32_t k, int32_t* ids1, float* scores1, int32_t* ids2,
                          float* scores2, void* stream);

/* ---- negative sampling on the device (replaces NegativeExampleGenerator.get_negative_samples, NegativeExampleGenerator.py:14-32)
 * out[i] = searchsorted(cum, uniform(0, cum_last)) for i in [0, n), bit-exact with the reference's host recipe on a legacy
 * numpy RandomState: mt_state is the generator state on the device (uint32 key[624] followed by pos, as from
 * rng.get_state()) and is ADVANCED in place exactly as numpy would (2 words per draw), so it can be handed back with
 * rng.set_state().  cum: device float64[n_cum] (OieData.py:57-59), cum_last = cum[n_cum-1] (host copy).
 * scratch_words: device uint32[2n].  The caller reshapes out to (S, n_examples) (NegativeExampleGenerator.py:24). */
int rae_sample_negatives(rae_engine* h, uint32_t* mt_state, const double* cum, int64_t n_cum, double cum_last, int32_t* out,
                         int64_t n, uint32_t* scratch_words, void* stream);

/* ---- func['label_<split>'] ------------------------------------------------------------------------------ */
/* labels = argmax of the scores, first max wins (RelationClassifier.py:45-47); probs = softmax.  Device outputs. */
int rae_label(rae_engine* h, int32_t split_id, int64_t batch_index, int64_t* labels, float* probs, void* stream);
/* same with HOST outputs (synchronous) */
int rae_label_host(rae_engine* h, int32_t split_id, int64_t batch_index, int64_t* labels_host, float* probs_host,
                   void* stream);

/* ---- introspection (parity tests, bench) ---------------------------------------------------------------- */
/* copy the last step's q(r|x) [B,K] into a device buffer */
int rae_get_probs(rae_engine* h, float* dst, void* stream);
/* copy the last step's dense gradient of one parameter (needs RAE_FLAG_DENSE_GRADS) into a device buffer of the
 * parameter's shape: what T.grad(cost, params) (Optimizers.py:27) would have produced */
int rae_get_dense_grad(rae_engine* h, int32_t param_id, float* dst, void* stream);
/* device copy of the last step's sorted entity occurrence keys / permutation and segment starts (bit-exact layout
 * checks against np.argsort(kind='stable') + np.unique).  Each dst may be NULL.  n_* receive the element counts. */
int rae_get_entity_segments(rae_engine* h, int32_t* sorted_rows, int32_t* sorted_occ, int32_t* seg_start,
                            int64_t* n_occ, int64_t* n_seg, void* stream);
int rae_get_step_stats(rae_engine* h, rae_step_stats* out);

/* per-phase device timing of a step (CUDA events on the step's stream; bench.py's roofline leg).  One phase = one kernel of
 * the step (plus its small helpers), in stream order:
 *  0 encoder_forward   k_encoder_forward*                      8 contract_recompute  k_tc_bilinear (M c, M^T a)
 *  1 entity_sort       k_entity_keys + CUB radix sort          9 contract_dq         k_tc_transpose_al + k_tc_dq
 *  2 feature_sort      (cached at bind time: ~0)              10 backward_finish     k_tc_bwd_finish
 *  3 operand_prep      k_tc_prep_c + k_tc_prep_qt             11 contract_dc         k_tc_dc2 (B % 4 != 0: k_tc_dc)
 *  4 contract_forward  k_tc_bilinear                          12 dense_finalize      k_dense_finalize
 *  5 score             k_score                                13 cost                k_cost (+ k_reg_norms)
 *  6 entity_update     k_rows_chunk<1> + k_entity_long2       14 dense_apply         k_dense_apply
 *  7 w_update          k_rows_chunk<0> + k_w_long2
 * (SIMT contraction path: 4 = k_bilinear_forward, 8-10 = k_bilinear_backward, 11 = k_grad_dense.)
 * Profiling serialises the side streams and adds event records between kernels: never on for a timed run. */
#define RAE_NUM_PHASES 15
int rae_set_profiling(rae_engine* h, int32_t on);
/* on == 2: timeline mode - the step keeps its normal multi-stream overlap and an event is recorded behind every kernel
 * group on the stream it ran on; rae_get_timeline writes one line per mark, "name stream microseconds-since-step-start"
 * (stream 0 = the caller's, 1 = entity side stream, 2 = W / operand side stream), NUL-terminated, into buf[len]. */
int rae_get_timeline(rae_engine* h, char* buf, int64_t len);
/* milliseconds of each phase of the last profiled step (synchronises); ms must hold RAE_NUM_PHASES floats */
int rae_get_phase_times(rae_engine* h, float* ms);
const char* rae_phase_name(int32_t phase);

#ifdef __cplusplus
}
#endif
#endif /* RAE_H_ */
