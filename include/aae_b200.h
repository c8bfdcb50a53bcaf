/*
 * aae_b200.h -- C ABI of the B200-native AAE hot path (libaae_b200.so).
 *
 * This is the drop-in boundary for the path named in BASELINE.json: the training step of
 * aaerec's AdversarialAutoEncoder (partial_fit = ae_step + disc_step + gen_step) and its
 * predict / masked top-k ranking.  The reference is pure Python on torch; a maintainer binds
 * these entry points with ctypes from aaerec/aae.py (see INTEGRATION.md).  Each function names
 * the reference code it replaces (file:line under the reference tree).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - all matrices are dense row-major float32; CSR index arrays are int32, column indices
 *     sorted and unique inside a row (what BagsWithVocab.tocsr() yields, datasets.py:459-470);
 *   - `stream` is a cudaStream_t passed as void*; calls only enqueue work, they never
 *     synchronise and never allocate (the caller owns every buffer);
 *   - return value 0 = ok, negative = error (AAE_E_*), text via aae_last_error();
 *   - the library refuses to run on anything but compute capability 10.x (no fallback path).
 *
 * Weight layout (fp32):  W1t [V,H] is enc.lin1.weight TRANSPOSED (one 4H-byte row per item, so
 * the encoder's first layer is an embedding-bag gather); Wd3 [V,H] is dec.lin3.weight as torch
 * stores it; every other layer keeps torch's [out,in] layout.
 */
#ifndef AAE_B200_H
#define AAE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AAE_OK 0
#define AAE_E_ARG (-1)      /* bad argument (null pointer, size out of the supported envelope) */
#define AAE_E_CUDA (-2)     /* a CUDA runtime call failed */
#define AAE_E_ARCH (-3)     /* device is not sm_100 */
#define AAE_E_UNSUPPORTED (-4)

/* Adam hyper-parameters and the shared step counter, resident on the device so that a captured
 * CUDA graph can be replayed: aae_step_tick() advances t and recomputes the bias corrections in
 * double precision exactly like torch/optim/adam.py (lr/(1-b1^t), sqrt(1-b2^t)).
 * The reference builds four torch.optim.Adam with default betas/eps (aae.py:798-804): enc_optim
 * and dec_optim use gen_lr, gen_optim and disc_optim use reg_lr; all four step once per
 * partial_fit, so they share t. */
typedef struct {
  int32_t t;               /* number of completed aae_step_tick calls (= Adam step index) */
  uint32_t rng_step;       /* counter mixed into the in-kernel Philox streams */
  float step_size_gen;     /* gen_lr / (1 - beta1^t) */
  float step_size_reg;     /* reg_lr / (1 - beta1^t) */
  float bc2_sqrt;          /* sqrt(1 - beta2^t) */
  float beta1, beta2, eps;
  float gen_lr, reg_lr;
  uint64_t seed;           /* Philox key for dropout / prior sampling in native RNG mode */
} aae_step_state;

/* Dropout description for one dropout layer.  mask != NULL: use the given [B,width] mask whose
 * entries are 0 or 1/(1-p) (oracle-RNG mode: draws made by torch in the reference's order, SURVEY
 * 8(a) A11).  mask == NULL and p > 0: in-kernel Philox, stream id `stream_id`.  p == 0: identity. */
typedef struct {
  const float* mask;
  float p;
  uint32_t stream_id;
} aae_drop;

int aae_version(void);
const char* aae_last_error(void);
/* 0 if device `dev` is compute capability 10.x, AAE_E_ARCH otherwise. */
int aae_device_check(int dev);

/* ---- step bookkeeping ------------------------------------------------------------------- */
int aae_step_state_init(aae_step_state* st, float gen_lr, float reg_lr, uint64_t seed, void* stream);
int aae_step_tick(aae_step_state* st, void* stream);

/* ---- K1: encoder first layer on the sparse multi-hot input ---------------------------------
 * Replaces F.normalize(inp, 1) + Encoder.lin1 (aae.py:132-135): out[b,:] = b1 + sum_{i in set_b}
 * W1t[i,:] * (normalize ? 1/|set_b| : 1).  Empty set -> b1.  Items outside [v_begin, v_end) are
 * skipped and b1 is added only when add_bias != 0 (item-sharded partial sums). */
int aae_bag_fwd(const int32_t* indptr, const int32_t* indices, int B, const float* W1t, const float* b1,
                int H, int normalize, int v_begin, int v_end, int add_bias, float* out, void* stream);




/* Dense-Adam-equivalent sweep of W1t for rows NOT in the batch: torch's Adam moves every row every
 * step even when its gradient is zero (momentum decay), once per optimizer state, enc_optim first
 * (aae.py:706) then gen_optim (aae.py:741).  Rows with slot_of >= 0 are skipped (they are updated by
 * aae_rows_adam with their gradients).  rows [r_begin, r_end) of the local shard. */
int aae_w1_sweep_untouched(const int32_t* slot_of, int r_begin, int r_end, int H, float* W, float* m1, float* v1,
                           float* m2, float* v2, const aae_step_state* st, void* stream);


/* ---- time-blocked dense Adam for W1t (the engine's default policy) ----------------------------------
 * The zero-gradient Adam update of a row that is not in the batch depends only on the row and on the step's
 * bias corrections, so it may be applied late -- bit-identically -- as long as that happens before the row is
 * read again.  last[Vloc] (int32, zero-initialised) holds the last step applied to each row, ktab
 * [AAE_KTAB_SLOTS][4] floats the constants of recent steps (slot t % AAE_KTAB_SLOTS: step_size_gen,
 * step_size_reg, 1/sqrt(1-b2^t), 0).  Each step only the rows of group t % G of G contiguous groups are swept
 * (their <= G pending steps replayed in registers, the same fp32 operations in the same order as the dense
 * sweep): 40/G bytes of HBM traffic per parameter per step instead of 40.  G = 1 is the dense sweep.
 *   aae_ktab_write      : store the constants of step st->t (after aae_step_state_init + aae_step_tick).
 *   aae_w1_catchup      : rows of the batch -> up to date through step t-1 (before the encoder gathers them);
 *                         claim[Vloc] (int32, zero-initialised) de-duplicates items shared by several sets.
 *   aae_w1_sweep_blocked: flush == 0: group t % G, rows with slot_of < 0, up to step t;  flush != 0: every row up
 *                         to step t-1 (call between steps, before predict / weight export).
 *                         ctas_per_sm > 0: slim 128-thread CTAs that run beside the step's small kernels.
 *   aae_w1_rows_update with last != NULL stamps the updated rows with step t. */
#define AAE_KTAB_SLOTS 64
int aae_ktab_write(const aae_step_state* st, float* ktab, void* stream);
int aae_w1_catchup(const int32_t* indptr, const int32_t* indices, int B, int v_begin, int v_end, int32_t* claim,
                   float* W, float* m1, float* v1, float* m2, float* v2, int32_t* last, int H,
                   const aae_step_state* st, const float* ktab, void* stream);
int aae_w1_sweep_blocked(const int32_t* slot_of, int Vloc, int H, float* W, float* m1, float* v1, float* m2,
                         float* v2, int32_t* last, const aae_step_state* st, const float* ktab, int G, int flush,
                         int ctas_per_sm, void* stream);


/* ---- K4: the small replicated layers ---------------------------------------------------------
 * All small weights of a module live in one contiguous block; the structs give their shapes.
 * enc block : [b1 (H) | We2 (H*H) | be2 (H) | We3 (C*H) | be3 (C)]        (Encoder.lin1.bias, lin2, lin3)
 * dec block : [Wd1 (H*Cp) | bd1 (H) | Wd2 (H*H) | bd2 (H)]               (Decoder.lin1, lin2)
 * disc block: [Wq1 (H*C) | bq1 (H) | Wq2 (H*H) | bq2 (H) | wq3 (H) | bq3 (1)]  (Discriminator)
 * Cp = C + D where D is the width of the concatenated condition rows (0 if none). */
typedef struct {
  int B, H, C, D;
} aae_dims;

/* ae_step backward tail: from dh2 = dL/dh2 to dL/dh1pre; writes the pre-activation gradients of
 * every small layer (g_d2, g_d1, g_z, g_e2, g_h1), consumed by aae_small_wgrad / aae_bag_bwd. */
int aae_ae_bwd(aae_dims d, const float* dh2, const float* enc, const float* dec, aae_drop e1, aae_drop e2,
               aae_drop d1, aae_drop d2, const aae_step_state* st, const float* a1, const float* a2,
               const float* dd1, const float* h2, float* g_d2, float* g_d1, float* g_z, float* g_e2,
               float* g_h1, void* stream);


/* ---- fused step (the engine's default flow): the sparse first layer inside the row-local kernels ----
 * aae_bag describes the batch's CSR rows and W1t; a kernel given a bag with indptr != NULL computes its row
 * of h1pre = b1 + sum_{i in set_b} W1t[i,:] (/|set_b|) itself (aae.py:132-135) instead of reading it from
 * memory, which removes the separate gather launch from the step's dependent chain.  indptr == NULL: the
 * kernel reads `h1pre` (item-sharded runs, where the partial sums are all-reduced first). */
typedef struct {
  const int32_t* indptr;
  const int32_t* indices;
  const float* W1t;        /* [v_end - v_begin, H] */
  int normalize;
  int v_begin, v_end;
} aae_bag;
/* aae_ae_fwd with the optional in-kernel gather; dh2_zero (may be NULL): the [B,H] accumulator of
 * aae_dec_out_train, cleared row by row here so that the step needs no separate zeroing launch. */
int aae_ae_fwd_bag(aae_dims d, aae_bag bag, const float* h1pre, const float* cond, const float* enc,
                   const float* dec, aae_drop e1, aae_drop e2, aae_drop d1, aae_drop d2, const aae_step_state* st,
                   float* a1, float* a2, float* zc, float* dd1, float* h2, float* dh2_zero, void* stream);
int aae_disc_phase_bag(aae_dims d, aae_bag bag, const float* h1pre, const float* z_real, float prior_scale,
                       const float* enc, const float* disc, aae_drop r1, aae_drop r2, aae_drop f1, aae_drop f2,
                       const aae_step_state* st, float* acts, float* grads, double* loss_sum, void* stream);
int aae_gen_phase_bag(aae_dims d, aae_bag bag, const float* h1pre, const float* enc, const float* disc, aae_drop e1,
                      aae_drop e2, aae_drop q1, aae_drop q2, const aae_step_state* st, float* a1, float* a2,
                      float* g_z, float* g_e2, float* g_h1, double* loss_sum, void* stream);
int aae_predict_tail_bag(aae_dims d, aae_bag bag, const float* h1pre, const float* cond, const float* enc,
                         const float* dec, float* h2, void* stream);

/* Batch bookkeeping in ONE launch (off the step's dependent chain): touched-row slots as aae_batch_slots
 * (slot_of / uniq / n_uniq; n_uniq is cleared here) plus the transposed view of the batch: for slot s the
 * batch rows that contain item uniq[s] are csc_row[csc_off[s] .. csc_off[s+1]).  cnt [cap] and pos [nnz] are
 * int32 scratch, csc_off has cap+1 entries, csc_row nnz entries; cap >= number of distinct local items. */
int aae_batch_prepare(const int32_t* indptr, const int32_t* indices, int B, int v_begin, int v_end,
                      int32_t* slot_of, int32_t* uniq, int32_t* n_uniq, int32_t* cnt, int32_t* pos,
                      int32_t* csc_off, int32_t* csc_row, int cap, void* stream);
/* K2 fused: gradient of the sparse first layer AND Adam on the touched rows, no intermediate buffer and no
 * atomics: for every touched item i, g = sum_{b : i in set_b} dh1[b,:] (/|set_b|) over the rows listed by
 * aae_batch_prepare, then the Adam update of W[i,:] (aae.py:703/706 with which = 0, :741 with which = 1). */
int aae_w1_rows_update(const int32_t* uniq, const int32_t* n_uniq, int cap, const int32_t* csc_off,
                       const int32_t* csc_row, const int32_t* indptr, int normalize, const float* dh1, float* W,
                       float* m, float* v, int H, const aae_step_state* st, int which, int32_t* last,
                       void* stream);
/* End of a fused step: aae_step_end, then the loss accumulators are cleared and the step state is advanced
 * (aae_step_tick) for the NEXT step -- so a step starts with its Adam constants and Philox counter in place
 * and needs no begin launch.  Call aae_step_tick once after aae_step_state_init when using this flow. */
int aae_step_finish(int32_t* slot_of, const int32_t* uniq, const int32_t* n_uniq, int cap, double* sums, int n_sums,
                    double n_total, int B, float* losses, aae_step_state* st, float* ktab /* may be NULL */,
                    void* stream);

/* Weight/bias gradients of the small layers (reductions over the batch): block-shaped outputs matching
 * the parameter blocks.  With an aae_adam_block whose p is non-NULL the optimizer step of that block
 * (enc_optim/dec_optim aae.py:706-707, disc_optim :731, gen_optim :741) is applied in the same kernel,
 * in place, right after each element's reduction; the gradient pointer may then be NULL. */
typedef struct {
  float* p;      /* packed parameter block (NULL: gradient only) */
  float* m;      /* Adam first moments, same shape */
  float* v;      /* Adam second moments */
  int which;     /* 0: step_size_gen (enc_optim, dec_optim), 1: step_size_reg (gen_optim, disc_optim) */
} aae_adam_block;
int aae_ae_wgrad(aae_dims d, const float* a1, const float* a2, const float* zc, const float* dd1,
                 const float* g_d2, const float* g_d1, const float* g_z, const float* g_e2, const float* g_h1,
                 float* g_enc, float* g_dec, aae_adam_block enc_opt, aae_adam_block dec_opt,
                 const aae_step_state* st, void* stream);
int aae_disc_wgrad(aae_dims d, const float* acts, const float* grads, float* g_disc, aae_adam_block disc_opt,
                   const aae_step_state* st, void* stream);
int aae_gen_wgrad(aae_dims d, const float* a1, const float* a2, const float* g_z, const float* g_e2, const float* g_h1,
                  float* g_enc, aae_adam_block enc_opt, const aae_step_state* st, void* stream);

/* ---- K3: the n_items-wide decoder output layer, training ------------------------------------
 * Replaces Decoder.lin3 + torch.sigmoid (aae.py:176-177), F.binary_cross_entropy(x+1e-12, t+1e-12)
 * (aae.py:693-695), its backward (aae.py:703) and dec_optim's Adam on lin3 (aae.py:707) in ONE pass
 * over Wd3: logits never reach HBM.  Targets are the batch's CSR rows.  For the local item range
 * [v_begin, v_begin+Vloc): loss_sum[0] += sum of BCE terms, dh2[B,H] += dZ.Wd3 (old weights), then
 * Wd3/bd3 and their Adam moments are updated in place.  n_total = B * V_global (the BCE mean).
 * impl: 0 = fp32 CUDA-core kernel, 1 = tcgen05 tensor-core kernel (3xTF32, fp32-accurate),
 * 2 = tcgen05 single-pass TF32; 1 and 2 run the software-pipelined kernel when the shape fits its TMEM /
 * shared-memory envelope (n_hidden 100: batch <= 104) and the one-tile-at-a-time kernel otherwise;
 * 3 / 4 force the latter (3xTF32 / TF32). */
int aae_dec_out_train(const float* h2, int B, int H, float* Wd3, float* bd3, float* mW, float* vW, float* mb,
                      float* vb, int v_begin, int Vloc, const int32_t* indptr, const int32_t* indices,
                      double n_total, const aae_step_state* st, float* dh2, double* loss_sum, int impl,
                      void* stream);
/* The same call for ANY batch size on the tensor-core path (the reference's scripts train with batches of 500, 1000
 * and 10000: main.py:76, eval/mpd/mpd.py:75-76, eval/aminer.py:62).  A batch beyond one row chunk of the pipelined
 * kernel (n_hidden 100: 104 rows) is walked chunk by chunk -- one pass over Wd3 per chunk with the forward, BCE and both
 * backward GEMMs of that chunk -- while the chunks' weight gradients are summed in `work` ([Vloc,H] + [Vloc] floats,
 * caller-owned; aae_dec_out_train_work_floats gives the size, 0 when the batch fits one chunk) and the last chunk
 * applies dec_optim's Adam once with the total gradient, as the reference's single backward does (aae.py:703-707).
 * work == NULL: batches beyond one chunk are only served by impl 0. */
int64_t aae_dec_out_train_work_floats(int B, int H, int Vloc, int impl);
int aae_dec_out_train_ws(const float* h2, int B, int H, float* Wd3, float* bd3, float* mW, float* vW, float* mb,
                         float* vb, int v_begin, int Vloc, const int32_t* indptr, const int32_t* indices,
                         double n_total, const aae_step_state* st, float* dh2, double* loss_sum, int impl, float* work,
                         int64_t work_floats, void* stream);

/* ---- predict (aae.py:840-870) --------------------------------------------------------------- */
/* out[b, v] = logit or sigmoid(logit) for local items; ldo = row pitch of out in floats.
 * impl: 0 = fp32 CUDA-core kernel, 1 = tcgen05 3xTF32 (fp32-accurate), 2 = tcgen05 single-pass TF32; 3 and 4 score as
 * 1 and 2 (the choice of kernel they make in aae_dec_out_train exists only for training); any other value: AAE_E_ARG. */
int aae_dec_out_scores(const float* h2, int B, int H, const float* Wd3, const float* bd3, int Vloc,
                       int apply_sigmoid, float* out, int64_t ldo, int impl, void* stream);
/* Ranking tail = remove_non_missing + argtopk (evaluation.py:183-199, 20-58) without the dense
 * host matrix: known items (CSR rows, global ids, offset by v_begin) are excluded, the k best
 * remaining local items per row are returned sorted by descending score (ties: lower id first).
 * scores is overwritten (known items are set to -FLT_MAX).  idx_out holds GLOBAL item ids.
 * work: caller-provided scratch of aae_topk_work_bytes(B,k) bytes. */
int aae_masked_topk(float* scores, int64_t lds, int B, int Vloc, int v_begin, const int32_t* indptr,
                    const int32_t* indices, int k, int32_t* idx_out, float* val_out, void* work, void* stream);
/* Fused predict + ranking for large vocabularies (K5): reconstruction logits and the masked top-k WITHOUT the
 * [B, Vloc] score matrix.  Replaces predict's dense lin3 (aae.py:866-868) followed by remove_non_missing + argtopk
 * (evaluation.py:183-199, 20-58).  Four launches on the stream: (1) logits of a strided sample of 64-item tiles,
 * (2) per-row threshold = the J-th largest sample score (about T = max(1024, 4(k+256)) items of the shard pass it),
 * (3) the full tcgen05 pass whose epilogue appends (logit, item) pairs above the threshold to per-row candidate
 * lists, (4) known items masked, candidates sorted, first k emitted (descending, ties by lower item id).
 * Exactness never depends on the estimate: n_bad[0] (device) counts rows whose list overflowed or held fewer than
 * k unknown items; if it is non-zero the caller must rank the batch through aae_dec_out_scores + aae_masked_topk.
 * Envelope: impl 1 (3xTF32) or 2 (TF32), Vloc >= 32641 (256 tiles of 128 items), k <= 1024; otherwise AAE_E_UNSUPPORTED.
 * work: aae_predict_topk_work_bytes(B, Vloc, k) bytes of device scratch (0 = outside the envelope). */
int64_t aae_predict_topk_work_bytes(int B, int Vloc, int k);
int aae_predict_topk(const float* h2, int B, int H, const float* Wd3, const float* bd3, int Vloc, int v_begin,
                     const int32_t* indptr, const int32_t* indices, int k, int impl, void* work, int64_t work_bytes,
                     int32_t* idx_out, float* val_out, int32_t* n_bad, void* stream);
/* k-way merge of per-shard results: cand_val/cand_idx [B, n_cand] -> top k (descending). */
int aae_topk_merge(const float* cand_val, const int32_t* cand_idx, int B, int n_cand, int k, int32_t* idx_out,
                   float* val_out, void* stream);
/* The same merge for lists an all-gather left in [world][B][kpad] order (no repacking pass): world * kpad <= 2048;
 * entries with idx < 0 are padding. */
int aae_topk_merge_seg(const float* cand_val, const int32_t* cand_idx, int world, int B, int kpad, int k,
                       int32_t* idx_out, float* val_out, void* stream);

/* ---- item-sharded exchange over NVLink peer memory (multi-GPU, SURVEY 8(e)) -------------------------------------
 * What one device does inside a single dense GEMM in the reference (aae.py:132-135 X.W1^T, aae.py:176-177/703 the
 * decoder output layer and its input gradient) becomes, for item shards, an all-reduce(sum) of [B,H] partial sums.
 * Each rank owns one exchange buffer (cudaMalloc + CUDA IPC) that its peers map; aae_peer_allreduce is ONE kernel:
 * publish the local partial, signal/wait through flags in peer memory, sum the peers' slots in rank order (bit-identical
 * result on every rank).  No host synchronisation, capturable in a CUDA graph.  See csrc/peer.cu. */
#define AAE_PEER_MAX_WORLD 8
#define AAE_PEER_EXCHANGES 4       /* independent exchange ids (each with its own flags, sequence number and slots) */
#define AAE_PEER_HANDLE_BYTES 64   /* sizeof(cudaIpcMemHandle_t) */
typedef struct {
  void* base[AAE_PEER_MAX_WORLD];  /* exchange buffer of every rank as mapped in THIS process (own buffer at [rank]) */
  int rank, world;
} aae_peers;
/* Bytes of one rank's exchange buffer for messages of up to n_max floats. */
int64_t aae_peer_buffer_bytes(int64_t n_max);
/* Allocate + clear this rank's exchange buffer, return its IPC handle (these two calls allocate and synchronise). */
int aae_peer_alloc(int64_t n_max, void** base_out, unsigned char* handle_out);
int aae_peer_open(const unsigned char* handle, void** base_out);
int aae_peer_close(void* base);
int aae_peer_free(void* base);
/* data[0..n) <- sum over ranks (in place); extra[0..n_extra) (doubles, n_extra <= 4, may be NULL) likewise.  Every rank
 * must call with the same exchange id, n and n_max, in the same order.  A wait that exceeds ~20 s poisons the result with
 * NaN and sets an error flag (aae_peer_error) instead of hanging or summing stale slots. */
int aae_peer_allreduce(aae_peers peers, int exchange, float* data, int n, double* extra, int n_extra, int64_t n_max,
                       void* stream);
int aae_peer_error(const void* base, int* err_host);
/* aae_bag_fwd of an item shard FUSED with its exchange (one launch): out[b,:] = b1 + sum over the ranks of the partial
 * sums of X.W1^T over each rank's item range (aae.py:132-135 on item shards), bit-identical on every rank.  Batches of
 * up to 256 rows, n_hidden % 4 == 0 (otherwise aae_bag_fwd + aae_peer_allreduce). */
int aae_peer_bag_allreduce(aae_peers peers, int exchange, const int32_t* indptr, const int32_t* indices, int B,
                           const float* W1t, const float* b1, int H, int normalize, int v_begin, int v_end, float* out,
                           int64_t n_max, void* stream);

/* Self-test of the tcgen05 operand views used by the tensor-core kernel (one GEMM, one CTA):
 * mode 1: D[128,32] = A[128,104].Bm[32,104]^T; mode 2: D[128,112] = A[128,32].Bm[32,112];
 * mode 3: D[128,32] = A[128,104]^T.Bm[128,32] (rows >= 104 undefined).  split = 3 (3xTF32) or 1. */
int aae_tc_selftest(int mode, const float* A, const float* Bm, float* D, int split, void* stream);

/* ---- K5 v2: TMA-fed, cluster-multicast candidate filter + exact re-scoring -------------------------
 * Same contract as aae_predict_topk (top-k of remove_non_missing(predict(X), X), evaluation.py:183-199, 20-58, exact
 * outside score ties; n_bad[0] counts rows the caller must re-rank through the dense path).  The filter pass computes
 * single-pass TF32 logits straight from a padded copy of the output layer, Wp [Vloc, 104] = [Wd3 | bd3 | 0 0 0]
 * (aae_pad_weights; rebuilt by the caller whenever the weights change), streamed by TMA tensor loads that are multicast
 * across a thread-block cluster of up to 8 row-chunk CTAs; the filter threshold is lowered by a rigorous bound of the
 * TF32 error (wmax[0] = largest row norm of Wp, written by aae_pad_weights), the survivors (~1.4 k per row) are
 * re-scored exactly in fp32 from Wd3/bd3 and ranked.  n_hidden % 4 == 0, n_hidden <= 100. */
int64_t aae_pad_weights_floats(int Vloc, int H);
int aae_pad_weights(const float* Wd3, const float* bd3, int Vloc, int H, float* Wp, float* wmax, void* stream);
int64_t aae_predict_topk2_work_bytes(int B, int Vloc, int k, int H);
int aae_predict_topk2(const float* h2, int B, int H, const float* Wd3, const float* bd3, const float* Wp,
                      const float* wmax, int Vloc, int v_begin, const int32_t* indptr, const int32_t* indices, int k,
                      void* work, int64_t work_bytes, int32_t* idx_out, float* val_out, int32_t* n_bad, void* stream);

/* ---- candidate-restricted ranking (predict_topk(..., items=, exclude=)) -----------------------------------------
 * Replaces ranking every item and filtering the list afterwards (which leaves rows short): the eligible items of a shard
 * are gathered into a compact output layer [A, H] / [A] (aae_gather_item_rows) and the ranking entry points run on it
 * with v_begin = 0, so that the GEMM work, the weight bytes and the TF32 error bound (aae_pad_weights on the compact
 * copy) all follow the eligible set.  The filter tells the ranking which global id each compact column stands for and
 * which (row, item) pairs must never be returned:
 *   item_ids     [n_cols] global id of each column, strictly ascending; NULL: column c is item v_begin + c (with a table,
 *                v_begin must be 0)
 *   excl_indptr  [B+1] / excl_indices: per-row exclusions (global ids, sorted within each row); NULL: none
 * Known items (indptr/indices, global ids) that are columns rank below every other item (-FLT_MAX) as in the unfiltered
 * calls; excluded items and the padding of rows with fewer than k returnable items come out as (-1, -INFINITY).  Ties
 * go to the lower item id.  A NULL filter, or one with both tables NULL, is exactly the unfiltered call.  The fused
 * calls count rows with fewer than k returnable candidates in n_bad, like overflowing rows: the dense pair
 * aae_dec_out_scores + aae_masked_topk_filtered then gives the exact, padded answer. */
typedef struct {
  const int32_t* item_ids;
  const int32_t* excl_indptr;
  const int32_t* excl_indices;
} aae_rank_filter;
/* Wd3c[j,:] = Wd3[item_ids[j] - v_begin, :], bd3c[j] = bd3[item_ids[j] - v_begin] for j < A (one warp per row; float4
 * when H % 4 == 0, then Wd3 and Wd3c 16-byte aligned).  Checks the table: n_bad[0] (device) receives the number of
 * ids that lie outside [v_begin, v_begin + Vloc) or are not above their predecessor; it must be 0 before the copy is
 * used (a bad id's row is not read and is written as zeros with bias -INFINITY).  Replaces indexing the shard's
 * output layer on the host. */
int aae_gather_item_rows(const float* Wd3, const float* bd3, int H, int Vloc, int v_begin, const int32_t* item_ids,
                         int A, float* Wd3c, float* bd3c, int32_t* n_bad, void* stream);
/* aae_masked_topk / aae_predict_topk / aae_predict_topk2 on a filtered column set (Vloc = number of columns). */
int aae_masked_topk_filtered(float* scores, int64_t lds, int B, int Vloc, int v_begin, const int32_t* indptr,
                             const int32_t* indices, int k, int32_t* idx_out, float* val_out, void* work, void* stream,
                             const aae_rank_filter* filt);
int aae_predict_topk_filtered(const float* h2, int B, int H, const float* Wd3, const float* bd3, int Vloc, int v_begin,
                              const int32_t* indptr, const int32_t* indices, int k, int impl, void* work,
                              int64_t work_bytes, int32_t* idx_out, float* val_out, int32_t* n_bad, void* stream,
                              const aae_rank_filter* filt);
int aae_predict_topk2_filtered(const float* h2, int B, int H, const float* Wd3, const float* bd3, const float* Wp,
                               const float* wmax, int Vloc, int v_begin, const int32_t* indptr, const int32_t* indices,
                               int k, void* work, int64_t work_bytes, int32_t* idx_out, float* val_out, int32_t* n_bad,
                               void* stream, const aae_rank_filter* filt);

/* ---- GPU-side ranking metrics (SURVEY 8(f)-2) -----------------------------------------------------
 * Replaces the dense D2H + host argsort behind the harness' metrics (evaluation.py:70-164 RankingMetric / MRR /
 * MAP / P, evaluate 202-240 on remove_non_missing(predict(X), X)): for every held-out ("gold") item of every
 * query row, counts[p] = number of items of the local shard that rank before it -- unknown items with a strictly
 * higher score, or an equal score and a lower id (the tie order of the top-k kernels); known items of the row
 * (CSR indptr/indices, may be NULL) are pushed to the bottom first, as the reference's zeroing after min-max
 * scaling does.  rank = 1 + counts (summed over item shards).  scores [B, >=Vloc] (row pitch lds) are the logits
 * from aae_dec_out_scores and are modified (known entries := -FLT_MAX).  gold_indptr [B+1] / gold_indices [n_gold]:
 * CSR of the gold items (global ids); gold_scores [n_gold]: gold_scores_given == 0: receives their logits (NaN when
 * the item lies in another shard -- item-sharded callers replace NaN by 0, sum over the shards and call again with
 * gold_scores_given != 0, then sum the counts). */
int aae_rank_counts(float* scores, int64_t lds, int B, int Vloc, int v_begin, const int32_t* indptr,
                    const int32_t* indices, const int32_t* gold_indptr, const int32_t* gold_indices, int n_gold,
                    float* gold_scores, int gold_scores_given, int32_t* counts, void* stream);
/* aae_rank_counts on a filtered column set (evaluate_topk(..., items=, exclude=)): the gold ranks in the list that
 * aae_predict_topk*_filtered / aae_masked_topk_filtered return in full.  scores [B, >=Vloc] are the logits of the
 * filter's columns: the compact copy of aae_gather_item_rows when filt->item_ids is set (then v_begin must be 0), else
 * the shard's own columns v_begin + c.  Known items that are columns become -FLT_MAX, excluded (row, item) pairs
 * -INFINITY, so an excluded item never ranks before a gold.  The caller passes only returnable gold: items that are
 * eligible and not excluded for their row (on some shard); their rank in the filtered list is 1 + the counts summed
 * over item shards.  Gold items stay global ids.  With a column table a gold's tie position is the number of columns
 * with a lower id (a lower bound in item_ids), so the lower-id tie rule holds for a gold of another shard as well;
 * its score is that of its column, or NaN when it is not a column of this shard (the two-pass protocol of
 * aae_rank_counts then applies unchanged: NaN -> 0, sum over shards, call again with gold_scores_given != 0).  A NULL
 * filter, or one with both tables NULL, is exactly aae_rank_counts. */
int aae_rank_counts_filtered(float* scores, int64_t lds, int B, int Vloc, int v_begin, const int32_t* indptr,
                             const int32_t* indices, const int32_t* gold_indptr, const int32_t* gold_indices,
                             int n_gold, float* gold_scores, int gold_scores_given, int32_t* counts, void* stream,
                             const aae_rank_filter* filt);

/* ---- device-side epoch feed --------------------------------------------------------------------
 * Replaces sklearn.utils.shuffle(X, *condition_data) + X_shuf[start:end].toarray() (aae.py:815-823) and the
 * condition slices c[start:end] (aae.py:828): the training matrix (CSR: int64 indptr_all, int32 indices_all, sorted
 * unique columns) and the float32 condition matrix cond_all [n,D] stay resident in HBM; the host uploads one
 * permutation per epoch (the same np.random permutation the reference draws) and this call builds the packed CSR rows
 * (and condition rows) of the batch perm[row0 .. row0+B) in the step's fixed batch buffers.  perm == NULL: identity
 * (predict).  cond_all may be NULL.  out_indices must hold the batch's nnz (the caller knows the row lengths). */
int aae_batch_gather(const int64_t* indptr_all, const int32_t* indices_all, const int32_t* perm, int64_t row0, int B,
                     int32_t* out_indptr, int32_t* out_indices, const float* cond_all, int D, float* out_cond,
                     void* stream);

/* ---- denoising autoencoder input corruption (SURVEY 8(f)-3) ------------------------------------------
 * Replaces zeros_noise (dae.py:48-52: `mask = torch.rand(batch.size()) < noise_factor; batch[mask] = 0`, in place,
 * so the BCE target of dae.py:198-200 is the corrupted batch as well): every entry of the batch's CSR rows is dropped
 * with probability p.  noise != NULL: the reference's own [B,V] uniform draws (oracle-RNG mode); NULL: in-kernel Philox
 * keyed by (seed, step, row, item).  Column order is preserved; the output must not alias the input. */
int aae_batch_corrupt(const int32_t* in_indptr, const int32_t* in_indices, int B, int V, float p, const float* noise,
                      const aae_step_state* st, int32_t* out_indptr, int32_t* out_indices, void* stream);

/* ---- sibling recommenders on the same decoder output layer (SURVEY 8(f)-3) -------------------------------
 * DecodingRecommender (aae.py:461-584): "only the decoder part of the AAE" -- the reference's Decoder (aae.py:149-178)
 * fed with the concatenated condition encodings inp [B,D] (aae.py:499-507), BCE against the item sets, one Adam
 * (aae.py:522-523).  d.C must be 0, d.D = input width.  dec block: [Wd1 (H*D) | bd1 (H) | Wd2 (H*H) | bd2 (H)];
 * lin3 + sigmoid + BCE + its backward + Adam is aae_dec_out_train, predict ranks h2 through the K5 entry points.
 *   aae_decoder_fwd  : h2 = relu(drop(lin2(relu(drop(lin1(inp))))))  (train == 0: eval mode, dd1 may be NULL)
 *   aae_decoder_bwd  : dh2 -> g_d2, g_d1 (pre-activation gradients)
 *   aae_decoder_wgrad: weight / bias gradients of lin1, lin2 (+ Adam in place, as aae_ae_wgrad) */
int aae_decoder_fwd(aae_dims d, const float* inp, const float* dec, aae_drop d1, aae_drop d2, const aae_step_state* st,
                    float* dd1, float* h2, float* dh2_zero, int train, void* stream);
int aae_decoder_bwd(aae_dims d, const float* dh2, const float* dec, aae_drop d1, aae_drop d2, const aae_step_state* st,
                    const float* dd1, const float* h2, float* g_d2, float* g_d1, void* stream);
int aae_decoder_wgrad(aae_dims d, const float* inp, const float* dd1, const float* g_d2, const float* g_d1,
                      float* g_dec, aae_adam_block dec_opt, const aae_step_state* st, void* stream);
/* VAE (vae.py:47-266): fc1 (the sparse first layer: W1t gather, as aae_bag) -> relu -> fc21 | fc22 -> z = eps *
 * exp(logvar/2) + mu (vae.py:107-110) -> [z | cond] -> fc3 -> relu -> fc4 (= Wd3/bd3: aae_dec_out_train / K5); loss =
 * BCE + KLD (vae.py:132-145), ONE Adam over all parameters (vae.py:90-91).  No dropout.
 * enc block: [b1 (H) | Wml (2C*H) | bml (2C)] (rows 0..C-1 of Wml = fc21.weight, C..2C-1 = fc22.weight),
 * dec block: [W3 (H*(C+D)) | b3 (H)].
 *   aae_vae_fwd : eps [B,C] != NULL: the reference's randn draws (oracle-RNG mode), NULL: in-kernel Philox.  Writes
 *                 a1 = relu(fc1), mulv = (mu | logvar) [B,2C], eps_used, zc, h3 (any of the first four may be NULL in
 *                 predict) and adds KLD = -0.5 sum(1 + logvar - mu^2 - exp(logvar)) to kld_sum[0] (may be NULL).
 *   aae_vae_bwd : dh3 -> g_3 (fc3 pre-activation), g_ml = (dmu | dlogvar) incl. the KLD gradient, g_h1 (fc1
 *                 pre-activation; aae_w1_rows_update applies it to the touched rows of W1t)
 *   aae_vae_wgrad: gradients of b1, fc21/fc22, fc3 (+ Adam in place) */
int aae_vae_fwd(aae_dims d, aae_bag bag, const float* h1pre, const float* cond, const float* eps, const float* enc,
                const float* dec, const aae_step_state* st, float* a1, float* mulv, float* eps_used, float* zc,
                float* h3, float* dh3_zero, double* kld_sum, void* stream);
int aae_vae_bwd(aae_dims d, const float* dh3, const float* enc, const float* dec, const float* eps_used, const float* a1,
                const float* mulv, const float* h3, float* g_3, float* g_ml, float* g_h1, void* stream);
int aae_vae_wgrad(aae_dims d, const float* a1, const float* zc, const float* g_3, const float* g_ml, const float* g_h1,
                  float* g_enc, float* g_dec, aae_adam_block enc_opt, aae_adam_block dec_opt,
                  const aae_step_state* st, void* stream);

/* ---- host-buffer convenience (the end-to-end call): copies a CSR batch from pinned host memory. */
int aae_upload_batch(const int32_t* indptr_host, const int32_t* indices_host, int B, int nnz, int32_t* indptr,
                     int32_t* indices, void* stream);

/* The same with two source / destination candidates, chosen on the device: index (st->t + bias) & 1.  One captured
 * graph then alternates between two pinned slots (batch in: bias -1 before the step; losses out: bias 0 after it). */
int aae_copy_words_sel(const void* src0, const void* src1, void* dst0, void* dst1, int64_t n_words,
                       const aae_step_state* st, int bias, void* stream);

/* ---- step timeline (profiling aid) ---------------------------------------------------------------
 * With a device buffer of aae_trace_slots() uint64 installed, block 0 of every kernel of the step writes
 * %globaltimer (ns) at its start (slot 2*id) and end (slot 2*id+1); ids in the order: batch_prepare,
 * w1_sweep_untouched, ae_fwd, dec_out_train, ae_bwd, ae_wgrad, w1_rows_update(enc_optim), disc_phase,
 * disc_wgrad, gen_phase, gen_wgrad, w1_rows_update(gen_optim), step_finish, bag_fwd, w1_catchup.  buf == NULL: off.
 * Synchronises the device. */
int aae_trace_set(uint64_t* buf);
int aae_trace_slots(void);


#ifdef __cplusplus
}
#endif
#endif /* AAE_B200_H */
