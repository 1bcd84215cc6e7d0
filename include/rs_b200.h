/*
 * rs_b200.h — C-ABI of the B200-native CTR training hot path.
 *
 * Boundary that replaces, for the hot path of yueshifeng/recommendSystem
 * (SURVEY.md §8), the arithmetic that the reference reaches through Keras
 * layers + the `tensornet` sparse runtime.  The reference has no FFI of its
 * own (it is pure Python over TensorFlow); every entry point below cites the
 * reference call site whose arithmetic it replaces (paths relative to the
 * reference repo root).
 *
 * Conventions
 *   - extern "C"; plain pointers and sizes only.  No torch / STL types.
 *   - every pointer is CALLER-OWNED DEVICE memory unless the name ends in
 *     `_host`; the library never allocates behind the caller's back
 *     (workspaces are sized with rs_*_workspace_bytes and passed in).
 *   - every call is asynchronous on the `stream` passed (a cudaStream_t cast
 *     to void*; NULL = legacy default stream) and is CUDA-graph capturable.
 *   - return value: 0 = ok, otherwise an rs_status / cudaError_t code; the
 *     text is available from rs_last_error().  Never aborts the process.
 *   - matrices are row-major.  Keras `Dense.kernel` layout is kept: [in, out],
 *     y = x @ kernel + bias.
 *   - dtype codes: RS_F32 = 0, RS_BF16 = 1.
 */
#ifndef RS_B200_H_
#define RS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RS_ABI_VERSION 6   /* 4: + rs_interacting_path; saved buffer grows by the per-head softmax statistics.
                              5: + deferred parameter-gradient reductions (rs_logit_head_reduce, rs_interacting_bwd_reduce),
                                 a peer-store all-to-all of the routed ids, rs_embed_keys_from_rows;
                                 + rs_idmap_insert / _lookup / _rebuild, rs_idmap_count / _evict
                                 (additions only, same version)
                              6: the peer-store all-to-all of the routed ids is removed (they reach their owners by a
                                 NCCL all-to-all) */

enum rs_dtype { RS_F32 = 0, RS_BF16 = 1 };

enum rs_status {
  RS_OK = 0,
  RS_ERR_INVALID = 10001,     /* bad argument (shape / dtype / alignment) */
  RS_ERR_UNSUPPORTED = 10002, /* combination not built */
  RS_ERR_WORKSPACE = 10003    /* workspace too small */
};

/* GEMM epilogues (rs_gemm).  `aux` is an [M,N] tensor with leading dim ldaux. */
enum rs_epilogue {
  RS_EPI_NONE = 0,         /* C = A·B                               */
  RS_EPI_BIAS = 1,         /* C = A·B + bias[n]                      */
  RS_EPI_BIAS_RELU = 2,    /* C = relu(A·B + bias)      Dense(relu)  */
  RS_EPI_BIAS_SIGMOID = 3, /* C = sigmoid(A·B + bias)   Dense(sigmoid) */
  RS_EPI_MUL_RELU_MASK = 4,/* C = (A·B) * (aux > 0)     dgrad through relu */
  RS_EPI_MUL_DSIGMOID = 5, /* C = (A·B) * aux*(1-aux)   dgrad through sigmoid */
  RS_EPI_ACCUM = 6         /* C += A·B                               */
};

/* DIN attention-unit variants. */
enum rs_din_mode {
  RS_DIN_A = 0, /* din.py:18-47           [q,k,q*k] relu/relu, zero mask, sum pool   */
  RS_DIN_B = 1  /* staytime/layer.py:16-41 [q,f,q-f,q*f] sigmoid/linear, softmax pool */
};

/* ------------------------------------------------------------------ misc -- */
int rs_abi_version(void);
const char* rs_last_error(void);
/* Number of kernels this library has launched since load (bench.py's
 * `gpu_launches` claim is read from here). */
uint64_t rs_launch_count(void);
/* 1 if the library was compiled for sm_100a (it never is anything else). */
int rs_built_for_sm100a(void);
/* Measurement aid (tools/step_timeline.py): a one-thread kernel that stores %globaltimer (ns) into *dst when the stream
 * reaches it — inside a captured CUDA graph it timestamps the phase boundaries of a replay.  Not counted by
 * rs_launch_count; never launched by the product path unless a trainer's `stamps` buffer is set. */
int rs_debug_timestamp(unsigned long long* dst, void* stream);

/* ------------------------------------------------- K1/K2 embedding gather --
 * Replaces tn.layers.EmbeddingFeatures(...)(inputs) for single-valued slots
 * (bag = 1, `combiner='mean'` degenerates to a gather):
 *   staytime/VideoDnn.py:224-226,237   rough_rank/model.py:96-107
 *   rank/ctr/base_model.py:210-216     rank/finish/videodnn.py:60-66
 *
 * Tables of all fields live in one fp32 arena `table[total_rows, d]`.
 * Lookup i (i in [0,n)) belongs to field f = i % F and reads arena row
 *   row = row_base[f] + (ids[i] mod rows[f])       (ids[i] >= 0)
 * ids[i] < 0 is a padding id: the output row is zeros and row = -1.
 * `sort_keys` (nullable) receives (uint64(row) << 32) | i  — the key the
 * sparse-gradient path sorts (padding rows get row = 0xFFFFFFFF).
 * `rows_out` (nullable) receives the int32 arena row.
 * Integer addressing and the fp32 payload copy are bit-exact.
 */
int rs_embed_gather_fwd(const float* table, const int64_t* ids,
                        const int64_t* row_base, const int64_t* rows,
                        int64_t n, int F, int d,
                        void* out, int out_dtype,
                        uint64_t* sort_keys, int32_t* rows_out, void* stream);

/* Same with an explicit row stride `table_ld` (floats, >= d, multiple of 4; 0 = d): the trainer keeps each
 * row's weights and its Adam moments in ONE 3d-float record [w | m | v] (table_ld = 3d) so that the sparse
 * update touches one contiguous 12d-byte block per row instead of three scattered ones. */
int rs_embed_gather_fwd_ld(const float* table, int64_t table_ld, const int64_t* ids,
                           const int64_t* row_base, const int64_t* rows,
                           int64_t n, int F, int d,
                           void* out, int out_dtype,
                           uint64_t* sort_keys, int32_t* rows_out, void* stream);

/* Gather by precomputed arena rows (used by the row-sharded multi-GPU path
 * after id routing, and for sequence slots: staytime/VideoDnn.py:228-231
 * `combiner=None, seq_max_len=N` -> ([B,T,d], mask[B,T])).
 * rowidx[i] < 0 -> zeros and mask 0.  `mask_out` nullable (uint8).  out == NULL: no rows are
 * read, only `sort_keys` / `mask_out` are produced (the owner side of the peer-gather path). */
int rs_embed_gather_rows(const float* table, const int32_t* rowidx, int64_t n,
                         int d, void* out, int out_dtype, uint8_t* mask_out,
                         uint64_t* sort_keys, void* stream);

int rs_embed_gather_rows_ld(const float* table, int64_t table_ld, const int32_t* rowidx, int64_t n,
                            int d, void* out, int out_dtype, uint8_t* mask_out,
                            uint64_t* sort_keys, void* stream);

/* Row-sharded tables read IN PLACE over NVLink (one process per GPU; replaces the id all-to-all +
 * owner gather + row all-to-all of the sharded path — the only trace of sharding in the reference is
 * tn.core.shard_num() / self_shard_id(), staytime/parse.py:78-79).  peer_tables[r] (HOST array of
 * `world` DEVICE pointers) is rank r's shard, mapped into this process with rs_ipc_import; lookup i reads
 *   r = ids[i] mod rows[f] ; owner = r mod world ; peer_tables[owner] + (local_base[f] + r div world) * table_ld
 * (ids[i] < 0 -> zeros).  Bit-exact with rs_embed_gather_fwd on the unsharded arena.  The caller orders
 * the owners' sparse update of the previous step before this call (cross-rank barrier). */
#define RS_MAX_PEERS 8
int rs_embed_gather_peer_fwd(const float* const* peer_tables, int64_t table_ld, int world, const int64_t* ids,
                             const int64_t* local_base, const int64_t* rows, int64_t n, int F, int d,
                             void* out, int out_dtype, void* stream);
/* The backward half of the same exchange: row i of `src` (this rank's gradient rows, `row_bytes` each) is stored
 * into peer_recv[owner] (HOST array of `world` DEVICE pointers to every rank's receive buffer, rs_ipc_import) at
 * slot my_rank * cap + k, where index[i] = owner * cap + k is the lookup's slot in the send order produced by
 * rs_route_ids_padded (index[i] < 0: skipped).  Replaces permute + all-to-all; the caller separates it from the
 * owners' reads by a cross-rank barrier. */
int rs_scatter_rows_peer(const void* src, void* const* peer_recv, int world, int my_rank,
                         const int32_t* index, int64_t n, int cap, int row_bytes, void* stream);
/* Cross-rank barrier over peer memory for the two calls above (every rank launches it, in the same order, on its
 * own GPU): peer_flags[r] (HOST array of `world` DEVICE pointers, rs_ipc_import) is rank r's flag array of
 * RS_MAX_PEERS + 1 zero-initialised uint32; rank `rank` release-stores its next epoch into slot `rank` of every
 * array and spins (acquire loads) until all `world` slots of its own array have reached it.  Everything the rank
 * wrote before (peer stores included) is visible to a peer once that peer leaves the barrier. */
int rs_peer_barrier(unsigned int* const* peer_flags, int world, int rank, void* stream);
/* sort_keys[i] = (rowidx[i] << 32 | i) for rs_embed_sort_keys: the keys rs_embed_gather_rows writes as a by-product,
 * without the gather (the owners of a sharded step only need the keys: the rows were read through peer memory). */
int rs_embed_keys_from_rows(const int32_t* rowidx, int64_t n, uint64_t* sort_keys, void* stream);
/* CUDA-IPC plumbing for the above: export the allocation containing `ptr` (64-byte handle + byte offset
 * of ptr inside it); import maps a peer's allocation (peer access enabled lazily) and returns
 * base + offset. */
int rs_ipc_export(const void* ptr, unsigned char* handle64, unsigned long long* offset);
int rs_ipc_import(const unsigned char* handle64, unsigned long long offset, void** mapped);

/* Multi-valued slots: `combiner='mean'` over a CSR bag
 * (staytime/VideoDnn.py:224-226 with VarLenFeature ids, staytime/parse.py:22-23).
 * bag b of field f covers ids[offsets[b*F+f] .. offsets[b*F+f+1]). Empty bag -> zeros. */
int rs_embed_gather_bag_mean(const float* table, const int64_t* ids,
                             const int64_t* offsets, const int64_t* row_base,
                             const int64_t* rows, int64_t n_bags, int F, int d,
                             void* out, int out_dtype, void* stream);
/* The same lookup for TRAINING: table with an explicit row stride (0 = d; 3d for [w|m|v] records), and the two
 * by-products the backward needs: sort_keys[p] = (arena row << 32 | p) for every occurrence p (padding id < 0 ->
 * all-ones key, skipped by the segment sum) and inv_cnt[b] = 1 / #valid ids of bag b (0 if empty).  Either may be NULL.
 * rs_embed_bag_grad is the mean combiner's backward: g_occ[p, :] = dout[b(p), :] * inv_cnt[b(p)] (fp32 [nnz, d]), the
 * per-occurrence gradient rows that rs_embed_sort_keys + rs_embed_segsum_* consume. */
int rs_embed_bag_fwd_ld(const float* table, int64_t table_ld, const int64_t* ids,
                        const int64_t* offsets, const int64_t* row_base, const int64_t* rows,
                        int64_t n_bags, int F, int d, void* out, int out_dtype,
                        uint64_t* sort_keys, float* inv_cnt, void* stream);
int rs_embed_bag_grad(const void* dout, int dtype, const int64_t* offsets, const float* inv_cnt,
                      int64_t n_bags, int d, float* g_occ, void* stream);

/* --------------------------------- K3 sparse gradient + fused optimizer --
 * Replaces the backward of EmbeddingFeatures + the server-side sparse
 * optimizers tn.core.Adam(learning_rate, beta1, beta2, epsilon)
 *   (rank/multi_head/multidnn.py:235, rank/ctr/base_model.py:163,
 *    rough_rank/model.py:106)
 * and tn.core.AdaGrad(learning_rate, initial_g2sum, initial_scale)
 *   (staytime/VideoDnn.py:233,259).
 * Deterministic: keys are radix-sorted (stable) by row; each run of equal
 * rows is summed left-to-right in lookup order by one thread group, then the
 * optimizer is applied once per touched row.  No atomics.
 */
size_t rs_embed_sort_workspace_bytes(int64_t n);
/* Sorts `keys` by their high 32 bits restricted to `row_bits` significant
 * bits (row_bits = ceil(log2(total_rows+1)), or 32 to be safe). */
int rs_embed_sort_keys(const uint64_t* keys, uint64_t* keys_sorted, int64_t n,
                       int row_bits, void* ws, size_t ws_bytes, void* stream);

/* opt_scalars: device float[4] = {step, beta1^t, beta2^t, corr} maintained by
 * rs_adam_advance; the effective rate is lr * corr with
 * corr = sqrt(1-beta2^t)/(1-beta1^t) (Keras/TF Adam form):
 *   m = b1*m + (1-b1)*g ; v = b2*v + (1-b2)*g*g ; w -= lr*corr * m/(sqrt(v)+eps)
 * grad is [n, d] in lookup order (row i = gradient of lookup i), scaled by
 * grad_scale before use. */
int rs_embed_segsum_adam(float* w, float* m, float* v,
                         const void* grad, int grad_dtype,
                         const uint64_t* keys_sorted, int64_t n, int d,
                         float lr, float beta1, float beta2, float eps,
                         const float* opt_scalars, float grad_scale, void* stream);
/* Same with a common row stride `state_ld` (floats) of w, m, v — see rs_embed_gather_fwd_ld. */
int rs_embed_segsum_adam_ld(float* w, float* m, float* v, int64_t state_ld,
                            const void* grad, int grad_dtype,
                            const uint64_t* keys_sorted, int64_t n, int d,
                            float lr, float beta1, float beta2, float eps,
                            const float* opt_scalars, float grad_scale, void* stream);

/* TensorNet AdaGrad: g2sum is ONE scalar per row:
 *   g2sum += mean_d(g*g) ; w -= lr * g / (sqrt(g2sum) + eps)
 * per_element != 0 switches to the classic per-element accumulator
 * (g2sum then has shape [rows, d]). */
int rs_embed_segsum_adagrad(float* w, float* g2sum,
                            const void* grad, int grad_dtype,
                            const uint64_t* keys_sorted, int64_t n, int d,
                            float lr, float eps, int per_element,
                            float grad_scale, void* stream);

/* Deterministic sorted-segment sum only (no optimizer).  Output is indexed by
 * SORTED position p in [0,n): seg_rows[p] = arena row if p is the first
 * position of its run (a segment head) else -1; seg_sum[p, :] = the run's
 * summed gradient at heads (unspecified elsewhere).  Used by the parity tests
 * and by the multi-GPU path's checks. */
int rs_embed_segsum(const void* grad, int grad_dtype, const uint64_t* keys_sorted,
                    int64_t n, int d, int32_t* seg_rows, float* seg_sum,
                    void* stream);

/* step += 1; beta powers and corr refreshed (device-side so that a captured
 * CUDA graph advances the optimizer on every replay). */
int rs_adam_advance(float* opt_scalars, float beta1, float beta2, void* stream);

/* Dense Adam over a flat fp32 parameter buffer (tn.optimizer.Optimizer(
 * tn.core.Adam(...)), rank/multi_head/model.py:53, staytime/model.py:72).
 * Optionally refreshes a bf16 shadow copy used by the tensor-core GEMMs. */
int rs_dense_adam(float* w, float* m, float* v, const float* g, int64_t n,
                  float lr, float beta1, float beta2, float eps,
                  const float* opt_scalars, void* w_bf16_shadow, void* stream);

/* ------------------------------------------------ K7 id routing (sharded) --
 * Row-sharded tables: owner(i) = (ids[i] mod rows[f]) mod world,
 * local arena row = local_base[f] + (ids[i] mod rows[f]) / world.
 * Stable bucket-by-owner: send_rows[ send_offsets[o] + k ] is the k-th lookup
 * (in lookup order) owned by rank o; inverse[i] = its slot. Bit-exact vs the
 * CPU oracle.  Replaces TensorNet's sign->shard routing (only trace in the
 * reference: tn.core.shard_num()/self_shard_id(), staytime/parse.py:78-79).
 * counts/offsets are int32[world] / int32[world+1] device arrays. */
size_t rs_route_workspace_bytes(int64_t n, int world);
int rs_route_ids(const int64_t* ids, int64_t n, int F, const int64_t* rows,
                 const int64_t* local_base, int world,
                 int32_t* send_rows, int32_t* inverse,
                 int32_t* send_counts, int32_t* send_offsets,
                 void* ws, size_t ws_bytes, void* stream);
/* Fixed-capacity variant (no host round trip for the counts, so the whole sharded
 * step, all-to-alls included, is CUDA-graph capturable): bucket o owns the slots
 * [o*capacity, (o+1)*capacity) of send_rows[world*capacity]; unused slots hold row
 * -1 (gathers as zeros, contributes no gradient).  inverse[i] = slot of lookup i.
 * If a bucket would exceed `capacity`, *overflow is set to 1 (never cleared here)
 * and the surplus lookups get inverse = -1: the caller must treat that as an error.
 * ws >= rs_route_workspace_bytes(n, world) + (world+1)*4. */
int rs_route_ids_padded(const int64_t* ids, int64_t n, int F, const int64_t* rows,
                        const int64_t* local_base, int world, int capacity,
                        int32_t* send_rows, int32_t* inverse, int32_t* send_counts,
                        int32_t* overflow, void* ws, size_t ws_bytes, void* stream);
/* The same with padding ids (< 0) spread over the owners (owner = ((uint32(i) * 0x9E3779B1) >> 16) mod world, row -1)
 * instead of all in owner 0's bucket: inputs that are mostly padding (sequence / bag columns) keep the buckets balanced. */
int rs_route_ids_padded_spread(const int64_t* ids, int64_t n, int F, const int64_t* rows,
                        const int64_t* local_base, int world, int capacity,
                        int32_t* send_rows, int32_t* inverse, int32_t* send_counts,
                        int32_t* overflow, void* ws, size_t ws_bytes, void* stream);
/* out[i, :] = src[index[i], :] (un-permute received rows; index < 0 -> zeros) and
 * its adjoint out[index[i], :] = src[i, :] (index < 0 skipped). */
int rs_permute_rows(const void* src, void* out, const int32_t* index, int64_t n,
                    int d, int dtype, int scatter, void* stream);

/* ------------------------------------------ K9 collision-free id map ----
 * Replaces TensorNet's per-shard sign -> row hash tables, which the reference
 * reaches through tn.feature_column.category_column + tn.layers.EmbeddingFeatures
 * (rank/ctr/base_model.py:203-217, staytime/VideoDnn.py:217-244,
 * rough_rank/model.py:89-115): every distinct (field, id) gets its own arena row
 * the first time a training step sees it, instead of row_base + id mod rows.
 *
 * Map of `n_fields` fields (field f: capacity R_f rows starting at arena row
 * row_base_f):
 *   slots       16-byte {int64 key; int32 row; int32 pad} slots, field f owns
 *               S_f = next_pow2(2 R_f) of them from slot_base_f; key -1 = empty,
 *               row -1 = the key got no row (its field was full).  16-B aligned.
 *   key_of_row  int64[total rows]: the id that owns each arena row (-1 = unused).
 *   counters    int64[2][n_fields]: rows used per field, then overflowed lookups.
 *   geom        int64[n_fields][4] = {row_base_f, R_f, slot_base_f, S_f - 1}, 16-B aligned.
 * Lookup i reads ids[i] of field field_of_col[i % F] (int32[F]); ids < 0 are padding.
 * The slot of an id is splitmix64(id) & (S_f - 1), probed linearly (at most S_f
 * probes; no thread ever waits for another).
 *
 * rs_idmap_insert gives every new key a row (row_base_f + the counter's next value)
 * and writes that row's whole optimizer record: w[0:d] (row stride w_ld) from the
 * init rule below, s0 / s1 (nullable; s_width floats at row stride s_ld) set to
 * s*_init.  Once R_f rows are used, new keys of the field get no row.
 * Init rule: pair p = k/2 of w draws r = mix64(base + G (p+1)), base =
 * mix64(mix64(seed + G (f+1)) ^ id), G = 0x9E3779B97F4A7C15; u1 = ((r >> 40) + 1) 2^-24,
 * u2 = ((r mod 2^32) >> 8) 2^-24; w[2p] = scale (sqrt(-2 ln u1) cos(2 pi u2)),
 * w[2p+1] = scale (sqrt(-2 ln u1) sin(2 pi u2)) in fp32 (logf, sincospif).
 * A row's initial value depends on (seed, field, id) only.
 *
 * rs_idmap_lookup writes rows_out[i] (int64 arena row, -1 for padding, unseen or
 * overflowed keys).  after_insert = 1 (the call follows rs_idmap_insert on the same
 * ids): lookups of keys without a row are counted in counters[1][f], and the row
 * counters are clamped to R_f.  after_insert = 0 (inference): the map is not changed.
 *
 * rs_idmap_rebuild clears all `n_slots` slots (cudaMemsetAsync) and re-inserts
 * key_of_row[row_base_f + j] for j < counters[0][f] with its row; key_of_row past
 * the counters is set to -1.  Used to restore a map from a checkpoint or to roll it
 * back to earlier counters.  max_rows = max R_f.
 *
 * Eviction (TensorNet's feature_drop_show; the rules are this library's choice):
 *   show        fp32[total rows]: the show count of each row.  A row no key owns has
 *               show 0 at all times, so a newly inserted key starts from 0.
 * rs_idmap_count adds 1.0f to show[rows[i]] for every rows[i] >= 0 (atomicAdd; every
 * increment adds the same value, so the sum is independent of their order; it stops
 * growing at 2^24).  Callers pass the rows of training lookups only.
 * rs_idmap_evict, for 0 < decay <= 1 and a finite threshold (else RS_ERR_INVALID):
 *   1. show = fp32(show * decay) for every live row (row_base_f + j, j < counters[0][f]);
 *   2. drops every key whose decayed show is < threshold and compacts each field's
 *      live rows back into [row_base_f, row_base_f + live_f): the k-th dropped row
 *      below live_f receives the record of the k-th kept row at or above live_f
 *      (both ascending) — w (d floats, stride w_ld), s0 / s1 (nullable, s*_width
 *      floats at stride s*_ld; the arguments of rs_idmap_insert), show and key_of_row;
 *   3. vacated rows get show 0 and key_of_row -1; counters[0][f] = live_f and
 *      evicted[f] (int64[n_fields], caller-owned) grows by the keys dropped;
 *   4. rebuilds the slots as rs_idmap_rebuild.
 * Asynchronous on `stream` (no host synchronisation); `ws` (256-B aligned) holds
 * rs_idmap_evict_workspace_bytes(total_rows) bytes.  The layout after it is a pure
 * function of the layout before; an evicted key is like a key never seen. */
int rs_idmap_insert(void* slots, int64_t* key_of_row, int64_t* counters, const int64_t* geom, int n_fields,
                    const int64_t* ids, int64_t n, int F, const int32_t* field_of_col, uint64_t seed, float scale,
                    float* w, int64_t w_ld, int d, float* s0, int64_t s0_ld, int s0_width, float s0_init,
                    float* s1, int64_t s1_ld, int s1_width, float s1_init, void* stream);
int rs_idmap_lookup(const void* slots, int64_t* counters, const int64_t* geom, int n_fields, const int64_t* ids,
                    int64_t n, int F, const int32_t* field_of_col, int64_t* rows_out, int after_insert, void* stream);
int rs_idmap_rebuild(void* slots, int64_t n_slots, int64_t* key_of_row, const int64_t* counters, const int64_t* geom,
                     int n_fields, int64_t max_rows, void* stream);
int rs_idmap_count(float* show, const int64_t* rows, int64_t n, void* stream);
size_t rs_idmap_evict_workspace_bytes(int64_t total_rows);
int rs_idmap_evict(void* slots, int64_t n_slots, int64_t* key_of_row, int64_t* counters, const int64_t* geom,
                   int n_fields, int64_t total_rows, float* show, float threshold, float decay, float* w, int64_t w_ld,
                   int d, float* s0, int64_t s0_ld, int s0_width, float* s1, int64_t s1_ld, int s1_width,
                   int64_t* evicted, void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------- K4 InteractingLayer ----
 * InteractingLayer.call (InteractingLayer.py:37-61; duplicate at
 * rank/multi_head/interacting_layer.py): L iterations with SHARED weights of
 *   Q,K,V,R = relu(X·W{q,k,v,r} + b)         (:42-46)
 *   per head: P = softmax(Q_h K_hᵀ / sqrt(U/H))  (:47-52)
 *   X <- LayerNorm(relu(P V_h [+ R]))         (:55-60)
 * Wqkvr is [D, 4U] = [Wq | Wk | Wv | Wr] (Keras [in,out] kernels side by
 * side), bqkvr [4U].  D must equal U when L > 1.  x, y are [B, F, D|U]:
 * element (b,f,c) lives at ptr[b*bs + f*ld + c] (ld = field stride, bs = sample
 * stride in elements; bs = 0 means F*ld), so the layer can read / write the
 * Flatten()ed [B, F*U] columns of a wider concat buffer in place (autoint:36,45).
 * `saved` (training): rs_interacting_saved_bytes(B,F,U,L) bytes = fp32 [L, B*F, U] (then
 * fp32 [L, B*F, 4], tensor-core kernels only: the per-head softmax statistics
 * lse = max_j(s c) + log2 sum_j exp2(s c - max) of every row, first H of the 4 slots),
 * written by the forward and handed unchanged to the backward of the SAME
 * compute_bf16 mode; its content is private to that pair (kept in fp32 whatever
 * `dtype` is, so a bf16 run rounds only at the layer's input and output):
 *   FFMA kernels       : slots 0..L-2 = the input of every iteration after the first;
 *   tensor-core kernels: slots 0..L-1 = the pre-LayerNorm activations relu(o + r) of
 *                        every iteration (the backward differentiates ReLU/LayerNorm at
 *                        them and re-derives iteration inputs as LayerNorm(slot)).
 * The backward recomputes everything else.  NULL = inference (forward only; the FFMA
 * backward also accepts NULL when L == 1).  dtype applies to x, y (and dy, dx).
 * Parameters are fp32.
 * compute_bf16 != 0 runs every contraction of the layer on tcgen05 tensor cores (tf32
 * projections / QK^T, bf16 P.V and gradient products, fp32 TMEM accumulators) for the
 * shapes built (D = U = 16, H = 2, F <= 48, bf16 activations, no dropout) and uses the
 * FFMA kernels for the others; 0 = fp32 FFMA everywhere (parity mode).
 * rs_interacting_path tells which kernels a call with these arguments runs:
 * RS_PATH_TCGEN05, RS_PATH_FFMA, or RS_PATH_NONE (shape not built: the call would fail
 * with RS_ERR_UNSUPPORTED) — tests assert the path instead of inferring it.
 */
#define RS_PATH_NONE 0
#define RS_PATH_FFMA 1
#define RS_PATH_TCGEN05 2
int rs_interacting_path(int F, int D, int U, int H, int dtype, int compute_bf16, float dropout_rate);
size_t rs_interacting_workspace_bytes(int B, int F, int D, int U);
size_t rs_interacting_saved_bytes(int B, int F, int U, int L);
int rs_interacting_fwd(const void* x, int64_t x_ld, int64_t x_bs, int dtype,
                       const float* Wqkvr, const float* bqkvr,
                       const float* ln_gamma, const float* ln_beta, float ln_eps,
                       void* y, int64_t y_ld, int64_t y_bs, void* saved,
                       int B, int F, int D, int U, int H, int L, int use_res,
                       int compute_bf16, void* stream);
/* K1 fused into K4 (tensor-core path only; rs_interacting_path(...) == RS_PATH_TCGEN05, no dropout): the forward's
 * tile loader performs the embedding lookup itself (tn.layers.EmbeddingFeatures call sites, rank/ctr/base_model.py:216)
 * — ids [B, F] int64 (id < 0 = padding -> zero row), row = id mod rows[f], owner = row mod world, local row =
 * local_base[f] + row div world, read from peer_tables[owner] (fp32, row stride table_ld floats, 64-byte aligned rows;
 * world == 1: the local table) — and writes, as by-products, x_out = RNE(dtype) of the rows ([B,F,D], what
 * rs_embed_gather_fwd would have written: the MLP tower and the backward read it) and, if not NULL,
 * sort_keys[i] = (local row << 32 | i) for rs_embed_sort_keys.  Bit-identical to rs_embed_gather_* + rs_interacting_fwd. */
int rs_interacting_fwd_gather(const float* const* peer_tables, int64_t table_ld, int world,
                              const int64_t* ids, const int64_t* local_base, const int64_t* rows,
                              void* x_out, int64_t x_ld, int64_t x_bs, unsigned long long* sort_keys,
                              int dtype, const float* Wqkvr, const float* bqkvr,
                              const float* ln_gamma, const float* ln_beta, float ln_eps,
                              void* y, int64_t y_ld, int64_t y_bs, void* saved,
                              int B, int F, int D, int U, int H, int L, int use_res, void* stream);
/* Bags in the fused lookup (one GPU, the local table): ids [B, S] int64, field f owning the slots
 * [slot_off[f], slot_off[f+1]) of every sample (slot_off: F + 1 device int64, slot_off[F] = S, B * S < 2^31); id < 0 =
 * padding.  x_out[b, f] = RNE(dtype) of the mean of the rows of the bag's valid ids (fp32 sum in slot order times
 * 1 / count; an empty bag is zeros), inv_cnt[b * F + f] = 1 / count (0 for an empty bag) and, if not NULL,
 * sort_keys[p] = (row << 32 | p) for slot p = b * S + slot_off[f] + k (all-ones for padding): bit-identical to
 * rs_embed_bag_fwd_ld with offsets[b * F + f] = b * S + slot_off[f] followed by rs_interacting_fwd. */
int rs_interacting_fwd_gather_bag(const float* table, int64_t table_ld, const int64_t* ids, const int64_t* slot_off,
                                  const int64_t* row_base, const int64_t* rows, void* x_out, int64_t x_ld, int64_t x_bs,
                                  unsigned long long* sort_keys, float* inv_cnt, int dtype, const float* Wqkvr,
                                  const float* bqkvr, const float* ln_gamma, const float* ln_beta, float ln_eps,
                                  void* y, int64_t y_ld, int64_t y_bs, void* saved,
                                  int B, int F, int S, int D, int U, int H, int L, int use_res, void* stream);
/* The backward with the embedding-gradient exchange fused in (tensor-core path only): dx_add (may be NULL) is added
 * to the layer's input gradient row by row (the MLP tower's dX, same strides as dx; dx_add == dx is allowed), and when
 * `inverse` is not NULL the finished row of lookup i is stored straight into slot (rank * cap + inverse[i] mod cap) of
 * peer_recv[inverse[i] / cap] (peer stores over NVLink; inverse / cap from rs_route_ids_padded) instead of dx —
 * rs_scatter_rows_peer without the extra pass over dX.  inverse == NULL: dx = gradient (+ dx_add). */
int rs_interacting_bwd_scatter(const void* x, int64_t x_ld, int64_t x_bs, const void* saved, int dtype,
                               const float* Wqkvr, const float* bqkvr,
                               const float* ln_gamma, const float* ln_beta, float ln_eps,
                               const void* dy, int64_t dy_ld, int64_t dy_bs,
                               void* dx, int64_t dx_ld, int64_t dx_bs, const void* dx_add,
                               void* const* peer_recv, int world, int rank, const int* inverse, int cap,
                               float* dparams, int B, int F, int D, int U, int H, int L, int use_res,
                               void* ws, size_t ws_bytes, void* stream);
/* Deferred tail of rs_interacting_bwd_scatter: called with dparams == NULL it leaves the per-CTA partial sums of
 * [dW | db | dgamma | dbeta] in `ws`; this sums them in CTA order into dparams (same values as the undeferred call).
 * May run on another stream (ordered after the backward by the caller): the embedding update that follows the backward
 * does not read dparams, only the dense optimizer does.  B, F, D, U, H as passed to the backward. */
int rs_interacting_bwd_reduce(const void* ws, size_t ws_bytes, float* dparams, int B, int F, int D, int U, int H,
                              void* stream);
/* Training-mode attention-weight dropout (InteractingLayer.py:53-54; use_dropout=True at
 * rank/multi_head/multidnn.py:54 and rank/ctr/model_init.py:54-59): the softmax weights are multiplied by an
 * inverted-dropout mask before P.V.  The mask is a pure function of (dropout_seed, iteration, sample, head,
 * query, key) — a splitmix64 hash of the element's linear index, kept iff its top 24 bits >= rate * 2^24 — so
 * the backward regenerates it; pass the SAME rate and seed to both, and a fresh seed every step.
 * dropout_step (device pointer, may be NULL): the mask seed becomes dropout_seed + 0x9E3779B97F4A7C15 * (*dropout_step),
 * read by the kernel at launch — a step whose scalar arguments are frozen in a CUDA graph still gets a fresh
 * mask on every replay when the caller bumps the counter inside the graph.
 * dropout_rate == 0 is exactly rs_interacting_fwd / _bwd.  Built into the FFMA kernels (any shape). */
int rs_interacting_fwd_dropout(const void* x, int64_t x_ld, int64_t x_bs, int dtype,
                               const float* Wqkvr, const float* bqkvr,
                               const float* ln_gamma, const float* ln_beta, float ln_eps,
                               void* y, int64_t y_ld, int64_t y_bs, void* saved,
                               int B, int F, int D, int U, int H, int L, int use_res,
                               int compute_bf16, float dropout_rate, unsigned long long dropout_seed,
                               const unsigned long long* dropout_step, void* stream);
int rs_interacting_bwd_dropout(const void* x, int64_t x_ld, int64_t x_bs, const void* saved, int dtype,
                               const float* Wqkvr, const float* bqkvr,
                               const float* ln_gamma, const float* ln_beta, float ln_eps,
                               const void* dy, int64_t dy_ld, int64_t dy_bs,
                               void* dx, int64_t dx_ld, int64_t dx_bs, float* dparams,
                               int B, int F, int D, int U, int H, int L, int use_res,
                               int compute_bf16, float dropout_rate, unsigned long long dropout_seed,
                               const unsigned long long* dropout_step,
                               void* ws, size_t ws_bytes, void* stream);
/* dx [B,F,D] (ld dx_ld), dparams: fp32 [D*4U + 4U + U + U] = dW | db | dgamma |
 * dbeta, OVERWRITTEN.  ws >= rs_interacting_workspace_bytes. */
int rs_interacting_bwd(const void* x, int64_t x_ld, int64_t x_bs, const void* saved, int dtype,
                       const float* Wqkvr, const float* bqkvr,
                       const float* ln_gamma, const float* ln_beta, float ln_eps,
                       const void* dy, int64_t dy_ld, int64_t dy_bs,
                       void* dx, int64_t dx_ld, int64_t dx_bs,
                       float* dparams, int B, int F, int D, int U, int H, int L,
                       int use_res, int compute_bf16, void* ws, size_t ws_bytes,
                       void* stream);

/* --------------------------------------------------------- K6 DIN unit ----
 * mode RS_DIN_A  din.py:18-47:
 *   s_t = relu(relu([q,k_t,q*k_t]·W1+b1)·W2+b2); s_t = t < seq_len[b] ? s_t : 0
 *   out = Σ_t s_t · values_t
 * mode RS_DIN_B  staytime/layer.py:16-41:
 *   s_t = sigmoid([q,f_t,q-f_t,q*f_t]·W1+b1)·W2+b2; s_t = mask ? s_t : -2^32+1
 *   out = Σ_t softmax(s)_t · f_t        (values == keys == facts)
 * q [B,H]; keys/values [B,T,H] (element (b,t,c) at ptr[(b*T+t)*kv_ld + c], so
 * the first 16 columns of a wider [B,T,32] tensor can be used in place,
 * staytime/VideoDnn.py:68); seq_len int32 [B] (mode A) or mask uint8 [B,T]
 * (mode B; NULL = all valid).  W1 [3H|4H, Hd], b1 [Hd], W2 [Hd,1], b2 [1]
 * with Hd = 16 in both reference variants.  out [B,H] fp32|bf16.
 */
int rs_din_fwd(int mode, const void* q, const void* keys, const void* values,
               int64_t kv_ld, int dtype, const int32_t* seq_len,
               const uint8_t* mask, const float* W1, const float* b1,
               const float* W2, const float* b2, void* out,
               int B, int T, int H, int Hd, void* stream);
size_t rs_din_workspace_bytes(int mode, int B, int T, int H, int Hd);
/* dq [B,H], dkeys/dvalues [B,T,H] (ld dkv_ld; in mode B dvalues is ignored and
 * dkeys holds the full facts gradient), dparams fp32 = dW1|db1|dW2|db2
 * OVERWRITTEN. */
int rs_din_bwd(int mode, const void* q, const void* keys, const void* values,
               int64_t kv_ld, int dtype, const int32_t* seq_len,
               const uint8_t* mask, const float* W1, const float* b1,
               const float* W2, const float* b2, const void* dout,
               void* dq, void* dkeys, void* dvalues, int64_t dkv_ld,
               float* dparams, int B, int T, int H, int Hd,
               void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------- K5 MLP tower ----
 * One Dense layer and its gradients as a GEMM with a fused epilogue:
 *   C[M,N] = epi( op(A)[M,K] · op(B)[K,N] )
 * (`DNN.call` rough_rank/layer.py:100-109; MultiLayerDense autoint:40-41,49-50;
 *  expert/gate Dense staytime/VideoDnn.py:135-147, multidnn.py:62-63,83-85.)
 * transA: A is stored [K,M] (ld lda); transB: B is stored [N,K] (ld ldb).
 * dtype_ab RS_F32  -> any transA/transB.  Problems with 16-byte aligned bases / leading dims (ld % 4 == 0),
 *   fp32 C, M, N, K >= 8 and M*N*K >= 2^20 run on the tensor cores as 3xTF32 (hi/lo split inside the kernel, three
 *   tcgen05.mma.kind::tf32 products, ~2^-20 relative error per product: inside the 1e-5 fp32 bar);
 *   everything else, or everything after rs_set_fp32_gemm_mode(1), runs the fp32 FFMA kernel.
 * dtype_ab RS_BF16 -> tcgen05 tensor-core kernel (TMA-fed, fp32 accumulation in
 *   TMEM).  It consumes K-major operands only: transA = 0 and transB = 1 (weights
 *   are kept as bf16 [out,in] shadows; activations feeding a weight gradient are
 *   transposed with rs_transpose2d), lda/ldb multiples of 8, 16-byte aligned
 *   bases.  Deep-K, small-output problems (weight gradients) are split along K
 *   into fp32 partials in `ws` and summed in split order (deterministic).
 * dtype_c is the dtype of C / aux.  ws >= rs_gemm_workspace_bytes() (may be
 * NULL for RS_F32). */
size_t rs_gemm_workspace_bytes(void);
int rs_set_fp32_gemm_mode(int mode);   /* 0 = 3xTF32 tensor cores when eligible (default), 1 = FFMA only; returns the previous mode */
int rs_gemm(const void* A, int64_t lda, int transA,
            const void* B, int64_t ldb, int transB,
            void* C, int64_t ldc, const float* bias,
            const void* aux, int64_t ldaux, int epilogue,
            int M, int N, int K, int dtype_ab, int dtype_c,
            void* ws, size_t ws_bytes, void* stream);
/* out[n] = Σ_m x[m, n]  (bias gradient); deterministic two-level reduce
 * (fixed row-block order, no atomics). ws >= rs_colsum_workspace_bytes. */
size_t rs_colsum_workspace_bytes(int M, int N);
int rs_colsum(const void* x, int64_t ldx, int dtype, float* out, int M, int N,
              void* ws, size_t ws_bytes, void* stream);
/* y = x * (ref > 0) or x * ref*(1-ref) elementwise (activation backward on a
 * [M,N] tile with leading dims). kind: 0 relu-mask, 1 dsigmoid. */
int rs_act_bwd(const void* x, int64_t ldx, const void* ref, int64_t ldref,
               void* y, int64_t ldy, int M, int N, int dtype, int kind,
               void* stream);
/* dst[m, 0:N] = src[m, 0:N] with dtype conversion and leading dims
 * (concat / slice / cast glue). */
int rs_copy2d(const void* src, int64_t lds, int src_dtype, void* dst,
              int64_t ldd, int dst_dtype, int M, int N, void* stream);
/* y[m, n] = a[m, n] + b[m, n] with leading dims. */
int rs_add2d(const void* a, int64_t lda, const void* b, int64_t ldb, void* y,
             int64_t ldy, int M, int N, int dtype, void* stream);

/* ----------------------------------------------------------- K8 losses ----
 * p = clip(p_raw, 1e-6, 1)                                  (autoint:52)
 * loss = mean_b Σ_k ( -y log(p+1e-6) - (a-y) log(1-p+1e-6) )
 *                                  (rank/ctr/base_model.py:7-12; a = 1)
 * p_raw is the output of the final Dense(·, sigmoid); dz is the gradient wrt
 * that layer's PRE-activation (sigmoid' and the clip's pass-through folded in).
 * loss_out: device float[1], overwritten (deterministic block-ordered sum).
 */
int rs_bce_sigmoid_fwd_bwd(const void* p_raw, int dtype, const float* y,
                           float a, float* loss_out, void* dz, int B, int k,
                           void* stream);

/* Fused logits head for k = 1 (AutoInt): final Dense(1, sigmoid) + clip + the
 * loss above + the head's backward in ONE pass over Z:
 *   p_out[b] = sigmoid(Z[b,:]·w + bias)            (autoint:49-50)
 *   loss     = as rs_bce_sigmoid_fwd_bwd            (autoint:52, base_model.py:7-12)
 *   dZ[b,:]  = dz_b * w ;  dw = Z^T dz ;  db = Σ dz
 * Z, dZ are [B, zw] with leading dims ldz / lddz (zw % 4 == 0, zw <= 2048);
 * w, bias, dw, db, loss_out, y are fp32.  Deterministic (ordered partial sums). */
size_t rs_logit_head_workspace_bytes(int B, int zw);
int rs_logit_head_fwd_bwd(const void* Z, int64_t ldz, int dtype, const float* w,
                          const float* bias, const float* y, float a, void* p_out,
                          float* loss_out, void* dZ, int64_t lddz, float* dw, float* db,
                          int B, int zw, void* ws, size_t ws_bytes, void* stream);
/* Same, and columns [0, relu_cols) of dZ come out already multiplied by relu'(Z) (those columns of Z are the
 * output of the tower's last Dense(relu), autoint:39-45): the MLP backward starts from dZ[:, :relu_cols] as is. */
int rs_logit_head_fwd_bwd_relu(const void* Z, int64_t ldz, int dtype, const float* w,
                          const float* bias, const float* y, float a, void* p_out,
                          float* loss_out, void* dZ, int64_t lddz, float* dw, float* db,
                          int B, int zw, int relu_cols, void* ws, size_t ws_bytes, void* stream);
/* Deferred tail of the two calls above.  With dw == NULL they leave the per-CTA partial sums of dw / db / loss in
 * `ws` (dZ and p_out are complete); this sums them in fixed order.  It may run on another stream than the head (ordered
 * after it by the caller): only the dense optimizer (dense_feature_optimizer, rank/ctr/dnn_optimizer.py) reads
 * dw / db, so the tower's backward does not have to wait for the reduction. */
int rs_logit_head_reduce(const void* ws, size_t ws_bytes, float* dw, float* db, float* loss_out, int B, int zw,
                         void* stream);

/* The head's parameter gradients and loss from a p_out computed elsewhere (rs_tower_step): the per-CTA partials of
 * dw = Z^T dz, db = sum dz and the loss, dz derived from the stored p_out and y exactly as the two calls above derive
 * it, are left in `ws` for rs_logit_head_reduce. */
int rs_logit_head_grad(const void* Z, int64_t ldz, int dtype, const void* p, const float* y, float a, int B, int zw,
                       void* ws, size_t ws_bytes, void* stream);

/* The AutoInt tower's part of the bf16 train step in one launch (Dense(relu) N0 -> Dense(relu) N1 -> the logit head
 * -> their backward down to the tower's input gradient), all activations bf16 and row-major:
 *   H0 = relu(X W0 + b0) [B, N0];  Z[:, :N1] = relu(H0 W1 + b1);  p_out = sigmoid(Z w + ob) [B];
 *   dz = d BCE(clip(p_out, 1e-6, 1), y; a) / d logit (mean over B, as rs_logit_head_fwd_bwd_relu);
 *   dZ = dz w with dZ[:, :N1] multiplied by relu'(Z[:, :N1]);  dH0 = (dZ[:, :N1] W1^T) relu'(H0);  dX = dH0 W0^T.
 * X [B, K0]; Z, dZ [B, N1 + Ki] (Z[:, N1:] is read); W0T [N0, K0] and W1T [N1, N0] are the transposed bf16 weights,
 * W0 [K0, N0] and W1 [N0, N1] the weights as they lie; b0, b1, w [N1 + Ki], ob [1], y [B] fp32.  dX is stored, not
 * accumulated.  The head's dw / db / loss are not computed (rs_logit_head_grad).  rs_tower_supported says whether the
 * kernel exists for these widths (N0 = 256, N1 = 128, K0 and Ki multiples of 16, Ki <= 700). */
int rs_tower_supported(int K0, int N0, int N1, int Ki);
int rs_tower_step(const void* X, const void* W0T, const void* W1T, const void* W0, const void* W1, const float* b0,
                  const float* b1, const float* w, const float* ob, const float* y, float a, void* Z, void* p_out,
                  void* dZ, void* H0, void* dH0, void* dX, int B, int K0, int N0, int N1, int Ki, void* stream);
/* The forward half of rs_tower_step, for evaluation: H0 and H1 stay on chip, only p_out = sigmoid(Z w + ob) is written
 * (rows >= B are masked), bit-identical to the p_out rs_tower_step writes for the same X, Z[:, N1:] and weights (the
 * same kernel code: the bf16 rounding of H0 and H1, the order of the H1 w dot, the tensor-core dot of the interacting
 * half, expf).  Z[:, :N1] is neither read nor written; no label, gradient or loss is computed.  W0 and W1 are not read
 * (the backward's operands, in the argument order of rs_tower_step).  Same widths as rs_tower_supported. */
int rs_tower_fwd(const void* X, const void* W0T, const void* W1T, const void* W0, const void* W1, const float* b0,
                 const float* b1, const float* w, const float* ob, const void* Z, void* p_out, int B, int K0, int N0,
                 int N1, int Ki, void* stream);

/* dst[n, m] = src[m, n] (2-D transpose with leading dims; bf16 or fp32).  Used to
 * present activations K-major to the tensor-core weight-gradient GEMMs. */
int rs_transpose2d(const void* src, int64_t lds, void* dst, int64_t ldd, int M, int N,
                   int dtype, void* stream);

/* ---- DCN-v1 cross network ------------------------------------------------------------------
 * CrossNet.call (rough_rank/layer.py:256-264) and DeepCrossLayer.call (staytime/layer.py:66-72):
 *   x_{l+1} = x0 * (x_l . w_l) + b_l + x_l ,  l = 0..L-1 ,  x_0 = x0 ;  out = x_L.
 * x, out, dout, dx are [B, dim] with leading dims (elements); W, b are fp32 [L, dim] (the
 * reference's [dim,1] kernels / [dim] or [dim,1] biases laid side by side); dW, db fp32 [L, dim],
 * OVERWRITTEN.  One pass over the rows forward, two backward (HBM bound: dim * (in + out) bytes per
 * sample forward); weight gradients are reduced over fixed batch chunks in a fixed order
 * (deterministic).  dim % 4 == 0, L <= 8.  ws >= rs_cross_workspace_bytes(B, dim, L). */
size_t rs_cross_workspace_bytes(int B, int dim, int L);
int rs_cross_fwd(const void* x, int64_t x_ld, int dtype, const float* W, const float* b,
                 void* out, int64_t out_ld, int B, int dim, int L,
                 void* ws, size_t ws_bytes, void* stream);
int rs_cross_bwd(const void* x, int64_t x_ld, const void* dout, int64_t dout_ld, int dtype,
                 const float* W, const float* b, void* dx, int64_t dx_ld, float* dW, float* db,
                 int B, int dim, int L, void* ws, size_t ws_bytes, void* stream);

/* ---- input labels and metrics: the steps either side of the train step ------------------
 * rs_staytime_labels replaces the label half of `parse_input_func` (staytime/parse.py:30-68):
 *   wt        = min(watch_ms / 1000, cap_s)                                  (:41-43, cap 160)
 *   label[b,j]= exp((bins[j] - wt)^2 / (-2 sigma^2)) / (sqrt(2 pi) sigma) * (right-left)/(nbins-1)
 *               for j < nbins, label[b,nbins] = wt                           (:45-64)
 *   short/long= watch_ms > short_ms / long_ms  (int64 0/1)                   (:30-39, 7000 / 18000)
 *   weight    = landing[b] ? landing_weight : 1                              (:66, 5.0; the regex on
 *               `extra_info` is host string work, its result comes in as a byte per sample)
 * staytime_label is [B, nbins+1] fp32, dense; short_label, long_label,
 * sample_weight and landing may be NULL.  fp32 arithmetic in the reference's operation order. */
int rs_staytime_labels(const int64_t* watch_ms, const uint8_t* landing, const float* bins, int nbins,
                       int B, float* staytime_label, int64_t* short_label, int64_t* long_label,
                       float* sample_weight, int64_t short_ms, int64_t long_ms, float cap_s, float sigma,
                       float left, float right, float landing_weight, void* stream);

/* Streaming binary metrics of `compile(metrics=[BinaryAccuracy(), AUC(), tn.metric.CTR(), tn.metric.COPC()])`
 * (rough_rank/model.py:215-219, staytime/model.py:78-82).  `state` is rs_binary_metrics_state_bytes(T)
 * of zero-initialised device memory that accumulates over calls: exact integer confusion histograms
 * for the T ascending thresholds (Keras: pred > threshold, label cast to bool), sample and correct
 * counts, and ordered (deterministic) double sums of labels and predictions.
 * rs_binary_metrics_result writes 6 doubles: AUC (ROC, 'interpolation' summation as keras AUC.result()),
 * accuracy at acc_threshold, CTR = sum(label)/n, COPC = sum(label)/sum(pred), n, mean prediction. */
size_t rs_binary_metrics_state_bytes(int num_thresholds);
size_t rs_binary_metrics_workspace_bytes(int64_t n);
int rs_binary_metrics_update(const void* pred, int pred_dtype, const float* label, int64_t n,
                             const float* thresholds, int num_thresholds, float acc_threshold,
                             void* state, void* ws, size_t ws_bytes, void* stream);
int rs_binary_metrics_result(const void* state, int num_thresholds, double* out6, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RS_B200_H_ */
