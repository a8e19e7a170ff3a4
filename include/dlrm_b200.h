/*
 * dlrm_b200.h -- C ABI of libdlrm_b200.so: DLRM.jl's embedding + dot-interaction hot path
 * as hand-written sm_100a CUDA kernels with device-resident (HBM) embedding tables.
 *
 * Every entry point is what a `ccall((:sym, libdlrm_b200), Int32, ...)` in DLRM.jl would
 * bind in place of the Julia/EmbeddingTables.jl code cited next to it (paths relative to
 * the DLRM.jl checkout).  No torch / C++ types cross this boundary: opaque handles, plain
 * pointers, sizes.  All functions return a dlrmb_status (0 = ok); the message of the last
 * failure on the calling thread is available from dlrmb_last_error().
 *
 * Conventions
 *   - Arrays are C order.  A Julia `D x N` column-major matrix is the C array [N][D], so
 *     Julia buffers can be passed unchanged.
 *   - `idx`: table-major [ntab][B][P] (sample b of table k owns the P consecutive entries at
 *     (k*B + b)*P); this is DACLoader's `sparse[B x ntab]` matrix (src/data/criteo.jl:320-326)
 *     for P = 1 and load_inputs' `reshape(vec, :, B)` (src/data/criteo.jl:551-557) for P > 1.
 *     `idx_bytes` is 4 (UInt32/Int32) or 8 (Int64); `idx_base` is 1 for Julia callers, 0 for
 *     PyTorch-style callers.  Like the reference's `@inbounds` loops, the kernels do not
 *     range-check indices; dlrmb_check_indices does, on request.
 *   - Activations: `T` / `out` of the lookup is the PreallocationStrategy buffer
 *     [B][slots][D] with the first `slot0` slots reserved for the bottom-MLP output
 *     (slot0 = 1 in DLRM: src/model/model.jl:161, src/model/interact.jl:264-281).
 *   - `stream` is a cudaStream_t (NULL = the legacy default stream).  Device-pointer entry
 *     points are asynchronous on it; `_host` entry points take host buffers, copy in and out
 *     on the tables' own stream and return after completion.
 *   - Ownership: the library owns table storage and all workspaces (sized at
 *     dlrmb_tables_create for `max_lookups` = max B*P per table; no per-call allocation);
 *     activation buffers belong to the caller.  One host thread per handle at a time.
 */
#ifndef DLRM_B200_H
#define DLRM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dlrmb_tables dlrmb_tables;
typedef void* dlrmb_stream;

typedef enum dlrmb_status {
    DLRMB_OK = 0,
    DLRMB_EINVAL = 1, /* bad argument (the reference raises AssertionError / BoundsError) */
    DLRMB_ECUDA = 2,  /* CUDA runtime failure; message carries cudaGetErrorString */
    DLRMB_ENOMEM = 3, /* device allocation failed */
    DLRMB_EOOB = 4,   /* dlrmb_check_indices found an index outside [base, rows+base) */
    DLRMB_ESTATE = 5, /* call order violated (e.g. update_sorted without a sort) */
    DLRMB_ENCCL = 6   /* NCCL failure, or libnccl.so.2 could not be loaded (dlrmb_comm_* only) */
} dlrmb_status;

#define DLRMB_ABI_VERSION 1

int32_t dlrmb_abi_version(void);
const char* dlrmb_last_error(void);
/* Number of kernel launches issued by this library in this process (bench bookkeeping). */
int64_t dlrmb_launch_count(void);
/* Process-wide tuning / test switches, read by the launchers (never from the environment):
 *   "interact_general" 1 = run the general tiled interaction kernels even for the specialised shapes
 *   "update_two_launches" 1 = separate fix-up launch of the sparse update at every batch size
 *   "update_tile" 4, 8, .. 32 = entries per lane group of the sparse update (0 = chosen per batch)
 *   "bwd_variant" 0 = by batch size (default); 1 | 2 | 3 = one-sample-per-warp interaction backward (d = 128) holding all of T in
 *                     registers: FFMA2 with duplicated S at 144 registers / the same at 128 registers (one wave of CTAs up
 *                     to 2368 samples) / S stored once (FFMA2 with a scalar operand); 5 | 6 = streaming kernels (half of the
 *                     output rows per pass, T rows through a cp.async ring): duplicated S / S stored once, row-paired FFMA2
 *   "fwd_tb" 3|6|9, "fwd_ks" 0..3 = register block / k-split of the general tiled forward
 *   "fwd_ksplit" 0|1|2 = tensor-core forward with one warp per sample always / two warps per sample for one-wave
 *                        batches (default) / two warps per sample always
 * Defaults are the measured-fastest configuration; unknown names return DLRMB_EINVAL. */
int32_t dlrmb_set_option(const char* name, int64_t value);
int32_t dlrmb_get_option(const char* name, int64_t* value);
/* Device-side kernel stamps for measurement: with a buffer of dlrmb_clock_buffer_bytes() registered,
 * thread 0 of every CTA of every launch of the main kernels folds %globaltimer (nanoseconds, 32 ns steps)
 * at entry (atomic min) and exit (atomic max) into buffer[kernel][cta % 4096][2] (uint64; kernel order:
 * lookup, sort, update, update fix-up, interaction forward, interaction backward, sigmoid + BCE;
 * dlrmb_clock_kernels() of them).
 * The caller pre-fills entries with UINT64_MAX/2 and exits with 0 and reads min(entry) / max(exit) after
 * the launches have completed: the duration of a kernel where it really runs (e.g. inside a multi-stream
 * CUDA graph of a training step) without the microseconds a CUDA-event pair adds.  The pointer is read when a
 * launch is ISSUED (or captured); pass NULL to switch the stamps off (the default). */
int64_t dlrmb_clock_buffer_bytes(void);
int32_t dlrmb_clock_kernels(void);
int32_t dlrmb_clock_enable(void* device_buffer);

/* ---- table storage: replaces SimpleEmbedding{Static{D}}(data) on an `embedding_allocator`
 * array (src/model/model.jl:185-206, src/data/criteo.jl:413,490) and the CachedArrays-backed
 * storage of src/cachedarrays.jl with HBM-resident tables. ------------------------------- */
int32_t dlrmb_tables_create(int32_t device, int32_t ntab, const int64_t* rows, int32_t D,
                            int64_t max_lookups, dlrmb_tables** out);
/* Same with a storage element size: 4 = Float32 rows, 2 = BFloat16 rows (the reference's
 * `embedding_eltype` option, src/model/model.jl:187; src/cachedarrays.jl:5-19).  With bf16 storage
 * every kernel still accumulates in fp32; rows are rounded to nearest even when written.  Host
 * buffers of upload/download stay Float32.  (SURVEY.md section 8(f) row 3.) */
int32_t dlrmb_tables_create_ex(int32_t device, int32_t ntab, const int64_t* rows, int32_t D,
                               int64_t max_lookups, int32_t elem_bytes, dlrmb_tables** out);
int32_t dlrmb_tables_elem_bytes(const dlrmb_tables* t);
/* Grow the sort / update workspaces to serve batches of up to `max_lookups` = B*P lookups per table
 * (no-op when already large enough).  The tables themselves are untouched.  Synchronises the device;
 * meant for the first batch of a run, when a host that builds its tables before it knows the batch
 * size (DLRM.jl's `dlrm(...)` constructor) learns it. */
int32_t dlrmb_tables_reserve(dlrmb_tables* t, int64_t max_lookups);
int32_t dlrmb_tables_destroy(dlrmb_tables* t);
int32_t dlrmb_tables_info(const dlrmb_tables* t, int32_t* ntab, int32_t* D, int64_t* max_lookups,
                          int64_t* total_rows);
/* host [rows_k][D] f32 <-> device; `Array(table)` / `table.data` read-back
 * (src/validation.jl:138) and load_embeddings (src/data/criteo.jl:484-492). */
int32_t dlrmb_tables_upload(dlrmb_tables* t, int32_t k, const float* host);
int32_t dlrmb_tables_download(dlrmb_tables* t, int32_t k, float* host);
/* Device base pointer of table k ([rows_k][D] f32), for zero-copy views. */
int32_t dlrmb_tables_device_ptr(dlrmb_tables* t, int32_t k, float** dev);
/* ScaledUniform init, U(-1/sqrt(rows_k), 1/sqrt(rows_k)) (src/model/model.jl:61-65), from a
 * counter-based generator so the result depends only on (seed, k, row, col). */
int32_t dlrmb_tables_init_uniform(dlrmb_tables* t, uint64_t seed, dlrmb_stream stream);
int32_t dlrmb_tables_sync(dlrmb_tables* t);

/* ---- lookup: maplookup(PreallocationStrategy(slot0*D), tables, sparse)
 * (call site src/model/model.jl:161).  out[b][slot0+k][:] = sum_p table_k[idx[k][b][p]][:],
 * p ascending.  One launch covers every table. ------------------------------------------- */
int32_t dlrmb_embedding_fwd(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                            int32_t B, int32_t P, float* out, int32_t slots, int32_t slot0,
                            dlrmb_stream stream);

/* Training-step form of the lookup: the same pooled output plus, in the same launch, the index
 * sort / dedup that the sparse update of this batch needs (what dlrmb_embedding_sort computes; it
 * depends on the indices only).  The reference builds its SparseIndexer dictionaries inside
 * update! (src/train/train.jl:276-290); here that work rides in extra CTAs of the gather launch, so
 * dlrmb_embedding_update_sorted can follow the backward pass directly. */
int32_t dlrmb_embedding_fwd_sort(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                                 int32_t B, int32_t P, float* out, int32_t slots, int32_t slot0,
                                 dlrmb_stream stream);

/* ---- dot interaction: (dot::DotInteraction)(x, ys) and its rrule
 * (src/model/interact.jl:394-411, 438-447).  T is [B][F][d] with slot 0 = x.  If `x` is
 * non-NULL ([B][d]) it is used for slot 0 and also stored into T[b][0] (the fast_vcat of
 * :271-281, fused).  out is [B][d + F(F-1)/2 + pad], pad = padding to `pad_to_mul`
 * (POST_INTERACTION_PAD_TO_MUL, src/model/model.jl:32). ---------------------------------- */
int32_t dlrmb_interaction_fwd(int32_t device, float* T, const float* x, int32_t B, int32_t F,
                              int32_t d, int32_t pad_to_mul, float* out, dlrmb_stream stream);
/* dot_back (src/model/interact.jl:424-436): dT [B][F][d] (slot 0 included, as the reference
 * returns the whole (d*F) x B matrix) and dx [B][d] = dOut[:, :d] + dT[:, 0]. */
int32_t dlrmb_interaction_bwd(int32_t device, const float* dOut, const float* T, int32_t B,
                              int32_t F, int32_t d, int32_t pad_to_mul, float* dT, float* dx,
                              dlrmb_stream stream);
/* 1 if (F, d) has a compiled warp-per-sample specialisation (the Criteo / golden geometries; every
 * other shape runs the general tiled kernels), else 0.  Introspection for tests and benchmarks: the
 * reference picks its interaction implementation per type the same way (src/model/interact.jl:390-411
 * vs :503-513). */
int32_t dlrmb_interaction_has_warp_path(int32_t F, int32_t d);

/* ---- sparse SGD: lookup pullback -> SparseEmbeddingUpdate(delta = dT[:, slot0+k, :],
 * indices) (src/train/train.jl:144) followed by EmbeddingTables.update!(Flux.Descent(lr), ...)
 * (src/train/train.jl:283-290): table_k[r] -= lr * sum_{(b,p): idx=r} dT[b][slot0+k],
 * duplicates summed in ascending flat position, one read-modify-write per touched row.
 *
 * dlrmb_embedding_sort depends on the indices only (it may run on a side stream while the
 * forward/backward passes execute); dlrmb_embedding_update_sorted consumes its result.
 * dlrmb_embedding_bwd_sgd = both, on one stream. ----------------------------------------- */
int32_t dlrmb_embedding_sort(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                             int32_t B, int32_t P, dlrmb_stream stream);
int32_t dlrmb_embedding_update_sorted(dlrmb_tables* t, const float* dT, int32_t slots,
                                      int32_t slot0, float lr, dlrmb_stream stream);
int32_t dlrmb_embedding_bwd_sgd(dlrmb_tables* t, const void* idx, int32_t idx_bytes,
                                int32_t idx_base, int32_t B, int32_t P, const float* dT,
                                int32_t slots, int32_t slot0, float lr, dlrmb_stream stream);

/* Parity/debug export of the last sort for table k (host outputs; the SparseIndexer role,
 * src/train/train.jl:107-115,276-281): uniq[n_uniq] ascending 0-based row ids,
 * seg_offsets[n_uniq+1] exclusive prefix of multiplicities, perm[B*P] stable argsort of the
 * flat [B][P] index list.  Buffers must hold B*P (+1) entries.  Synchronises. */
int32_t dlrmb_sort_dedup_export(dlrmb_tables* t, int32_t k, int64_t* uniq, int32_t* seg_offsets,
                                int32_t* perm, int32_t* n_uniq);
/* Range check of a device or host index batch; DLRMB_EOOB + message on the first offender. */
int32_t dlrmb_check_indices(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                            int32_t B, int32_t P, int32_t idx_on_host);

/* ---- per-table pooling factors (multi-hot with mixed hotness): the index container of the reference's
 * load_inputs, "a vector mixing per-table vectors and P x B matrices" with each table's P = length / B
 * (src/data/criteo.jl:551-557).  `P` is a host array [ntab] of pooling factors, each >= 1; table k's
 * indices are the [B][P_k] block starting at element B * (P_0 + .. + P_{k-1}) of `idx` (Julia:
 * reduce(vcat, vec.(sparse))).  Per table the semantics are those of the uniform entry points above
 * (pooling in ascending p, dedup ties by flat position b*P_k + p, Flux.Descent with duplicates summed),
 * and with every P_k equal the results are bit-identical to them.  Limits: B * max_k P_k <= max_lookups
 * (grow with dlrmb_tables_reserve) and ntab <= dlrmb_mp_max_tables() (256: the per-table geometry reaches
 * the kernels as one kernel-parameter struct); anything else returns DLRMB_EINVAL.  Device-pointer calls
 * do not allocate, synchronise or copy from host memory, so they can be captured into a CUDA graph.
 * dlrmb_embedding_update_sorted and dlrmb_sort_dedup_export consume the last sort, uniform or _mp: after
 * an _mp sort, the export of table k returns its B * P_k entries.  The table-sharded multi-GPU entry
 * points have `_mp` forms too (dlrmb_shard_plan_mp, dlrmb_comm_a2a_indices_mp, dlrmb_indices_scatter_p2p_mp,
 * dlrmb_embedding_fwd_p2p_mp / _sort_mp below). */
int32_t dlrmb_mp_max_tables(void);
int32_t dlrmb_embedding_fwd_mp(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base, int32_t B,
                               const int32_t* P, float* out, int32_t slots, int32_t slot0, dlrmb_stream stream);
/* lookup + the sort for the coming update (tables with B * P_k <= 4096 sort inside the lookup launch) */
int32_t dlrmb_embedding_fwd_sort_mp(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base, int32_t B,
                                    const int32_t* P, float* out, int32_t slots, int32_t slot0, dlrmb_stream stream);
int32_t dlrmb_embedding_sort_mp(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base, int32_t B,
                                const int32_t* P, dlrmb_stream stream);
int32_t dlrmb_embedding_bwd_sgd_mp(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base, int32_t B,
                                   const int32_t* P, const float* dT, int32_t slots, int32_t slot0, float lr,
                                   dlrmb_stream stream);
int32_t dlrmb_check_indices_mp(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base, int32_t B,
                               const int32_t* P, int32_t idx_on_host);
/* host-buffer forms (every pointer host memory), as dlrmb_embedding_fwd_host / dlrmb_embedding_bwd_sgd_host */
int32_t dlrmb_embedding_fwd_mp_host(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base, int32_t B,
                                    const int32_t* P, float* out, int32_t slots, int32_t slot0);
int32_t dlrmb_embedding_bwd_sgd_mp_host(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                                        int32_t B, const int32_t* P, const float* dT, int32_t slots, int32_t slot0,
                                        float lr);

/* ---- jagged (variable-length) bags: the input of torch.nn.EmbeddingBag(input, offsets) and of the PyTorch DLRM's
 * (lS_o offsets, lS_i indices), in TorchRec's key-major KeyedJaggedTensor layout.  Single GPU, every table of the
 * handle, ntab <= dlrmb_mp_max_tables().
 *   values   all tables' indices, one flat array, table-major; `idx_base` (0 or 1) applies to values only.
 *   offsets  [ntab * B + 1] element offsets into values, non-decreasing, offsets[0] = 0, the same width as the
 *            indices (idx_bytes 4 or 8): bag b of table k is values[offsets[k*B + b] .. offsets[k*B + b + 1]).
 *   L        host [ntab], L[k] = offsets[(k+1)*B] - offsets[k*B]: table k's lookups in the batch.  0 <= L[k] <=
 *            max_lookups (grow with dlrmb_tables_reserve); L[k] = 0 is a table with no lookup.  The launchers size
 *            their grids and choose sort regimes from L, so a device-pointer call allocates nothing, does not
 *            synchronise or copy from the host, and can be captured into a CUDA graph.  The kernels trust that
 *            offsets agree with L (and that the indices are in range); dlrmb_check_indices_jagged verifies both.
 *   pooling  0 = sum, 1 = mean, for every table of the call.
 * Sum: out[b][slot0 + k] = sum of table_k[values[j]] over the bag, j ascending, in fp32 from +0.0f.  Mean: with n
 * the bag's length and w = 1.0f / n rounded to fp32, out = fl(S * w) for the sum S.  An empty bag gives +0.0f in
 * both modes and no gradient.  Update (dlrmb_embedding_update_sorted, Flux.Descent): sorted entry j of table k
 * contributes dT[b(j)][slot0 + k], times w(b(j)) in mean mode; duplicates are summed as for the other entry points
 * and row -= lr * sum.  When every bag of table k has P_k lookups, sum pooling gives the bits of the _mp (and
 * uniform) entry points: pooled rows, dedup export and tables after the update.
 * Anything else returns DLRMB_EINVAL.  dlrmb_embedding_update_sorted consumes the last sort, uniform, _mp or jagged;
 * after a jagged sort dlrmb_sort_dedup_export(k) returns table k's L[k] entries, perm holding positions inside table
 * k's block of values. */
int32_t dlrmb_embedding_fwd_jagged(dlrmb_tables* t, const void* values, const void* offsets, int32_t idx_bytes,
                                   int32_t idx_base, int32_t B, const int64_t* L, int32_t pooling, float* out,
                                   int32_t slots, int32_t slot0, dlrmb_stream stream);
/* training form: the lookup, then the sort for the coming update */
int32_t dlrmb_embedding_fwd_sort_jagged(dlrmb_tables* t, const void* values, const void* offsets, int32_t idx_bytes,
                                        int32_t idx_base, int32_t B, const int64_t* L, int32_t pooling, float* out,
                                        int32_t slots, int32_t slot0, dlrmb_stream stream);
int32_t dlrmb_embedding_sort_jagged(dlrmb_tables* t, const void* values, const void* offsets, int32_t idx_bytes,
                                    int32_t idx_base, int32_t B, const int64_t* L, int32_t pooling, dlrmb_stream stream);
/* DLRMB_EINVAL when offsets[0] != 0, offsets decrease or a table's total disagrees with L; DLRMB_EOOB for an index
 * outside its table.  The message names the first offender.  values / offsets on the host when on_host != 0.
 * Synchronises. */
int32_t dlrmb_check_indices_jagged(dlrmb_tables* t, const void* values, const void* offsets, int32_t idx_bytes,
                                   int32_t idx_base, int32_t B, const int64_t* L, int32_t on_host);

/* ---- weighted jagged bags: torch.nn.EmbeddingBag(input, offsets, per_sample_weights=w) in mode 'sum', TorchRec's
 * weighted KeyedJaggedTensor.  The jagged layout and rules above, plus
 *   weights  device f32 [sum(L)], one weight per entry of values, in the same order, whatever the table storage.
 *            Null only when the batch has no lookup.  Weights go with sum pooling only (these calls take no pooling
 *            argument), as torch refuses per_sample_weights outside mode 'sum'.
 * Forward: the pooled row of a bag starts at +0.0f; for j ascending over the bag, acc = fl(acc + fl(w_j * row_j)),
 * the product and the sum rounded separately (never a fused multiply-add).  An empty bag gives +0.0f.  With every
 * w_j = 1.0f the pooled rows are those of the unweighted sum, bit for bit.
 * Update (dlrmb_embedding_update_sorted after the weighted sort, Flux.Descent): sorted entry j of table k contributes
 * fl(dT[b(j)][slot0 + k] * w_j); the contributions of one row are added in ascending position, then
 * row -= fl(lr * sum).  With every w_j = 1.0f the tables after the update are those of the unweighted sum.  The
 * update and dlrmb_sort_dedup_export consume a weighted sort like any other; a later sort of any kind replaces it.
 * dlrmb_check_indices_jagged checks a weighted batch as it is (it does not read the weights). */
int32_t dlrmb_embedding_fwd_jagged_weighted(dlrmb_tables* t, const void* values, const void* offsets,
                                            const float* weights, int32_t idx_bytes, int32_t idx_base, int32_t B,
                                            const int64_t* L, float* out, int32_t slots, int32_t slot0,
                                            dlrmb_stream stream);
/* training form: the lookup, then the weighted sort for the coming update */
int32_t dlrmb_embedding_fwd_sort_jagged_weighted(dlrmb_tables* t, const void* values, const void* offsets,
                                                 const float* weights, int32_t idx_bytes, int32_t idx_base, int32_t B,
                                                 const int64_t* L, float* out, int32_t slots, int32_t slot0,
                                                 dlrmb_stream stream);
int32_t dlrmb_embedding_sort_jagged_weighted(dlrmb_tables* t, const void* values, const void* offsets,
                                             const float* weights, int32_t idx_bytes, int32_t idx_base, int32_t B,
                                             const int64_t* L, dlrmb_stream stream);
/* Gradient of the pooled rows with respect to the weights (per_sample_weights.grad):
 *   dw[j] = sum over d of dT[b][slot0 + k][d] * table_k[values[j]][d]   for entry j of bag b of table k,
 * dw device f32 [sum(L)] in the order of values (null only when the batch has no lookup), dT [B][slots][D] as for the
 * update (16-byte aligned when D % 4 == 0).  The rows are read as they are now, so call it before
 * dlrmb_embedding_update_sorted of the same batch to get the gradient of the forward's rows.  A bag with no entries
 * writes nothing.  Order of the sum, fixed by D alone: with V = 4 if D % 4 == 0 else 1, C = D / V chunks of V
 * floats and G = min(32, C rounded up to a power of two), partial l (0 <= l < G) adds the products of chunks
 * c = l, l + G, l + 2G, .. in ascending d, p_l = fl(p_l + fl(dT[d] * row[d])) from +0.0f; then for s = G/2, G/4,
 * .., 1: p_l = fl(p_l + p_(l xor s)) for every l; dw[j] = p_0.  Bit-identical from call to call.  It does not
 * read the weights.  Allocates nothing, does not synchronise, can be captured into a CUDA graph. */
int32_t dlrmb_embedding_weight_grad_jagged(dlrmb_tables* t, const void* values, const void* offsets, int32_t idx_bytes,
                                           int32_t idx_base, int32_t B, const int64_t* L, const float* dT, int32_t slots,
                                           int32_t slot0, float* dw, dlrmb_stream stream);

/* ---- loss: the top MLP's final sigmoid (src/model/model.jl:87-90) fused with bce_loss and its
 * pullback (src/train/train.jl:33-41, 45-71).  logits/labels [B] device f32.  Writes the mean loss
 * (one float), d(loss)/d(logit) [B] (sensitivity 1 folded in) and, if `prob` is non-NULL, the
 * sigmoid outputs [B].  `scratch` is a caller-provided, zero-initialised device buffer of at least
 * 65 floats that must not be shared between concurrent calls (SURVEY.md section 8(f) row 1). ---- */
int32_t dlrmb_bce_sigmoid_fwd_bwd(int32_t device, const float* logits, const float* labels, int32_t B,
                                  float* prob, float* dlogits, float* loss, float* scratch,
                                  dlrmb_stream stream);

/* ---- dense-layer backward glue: the pullback of OneDNN.Dense(Flux.Dense(in, out, relu))
 * (src/model/model.jl:72-93) minus its GEMMs: dZ = dY .* (Y > 0) (no mask when `y` is NULL) and the
 * bias gradient db[n] = sum_b dZ[b][n], one launch.  dy, y, dz are [B][N] device arrays (dz may be
 * dy), db is [N].  `scratch` is a caller-provided device buffer of at least
 * dlrmb_dense_bwd_scratch_floats(N) floats, zero-initialised once and not shared between concurrent
 * calls; the call leaves it ready for the next one. ---------------------------------------------- */
/* Forward epilogue of the same layer: z[b][n] = act(z[b][n] + bias[n]) in place on the GEMM output
 * (act = relu when `relu` != 0, identity otherwise). */
int32_t dlrmb_dense_fwd_bias_act(int32_t device, float* z, const float* bias, int32_t B, int32_t N, int32_t relu,
                                 dlrmb_stream stream);
int64_t dlrmb_dense_bwd_scratch_floats(int32_t N);
int32_t dlrmb_dense_bwd_act_bias(int32_t device, const float* dy, const float* y, int32_t B, int32_t N,
                                 float* dz, float* db, float* scratch, dlrmb_stream stream);

/* ---- batch marshalling: `load!(labels, dense, sparse, records)` (src/data/criteo.jl:284-310) on
 * the device.  `records` is a DEVICE copy of B packed DACRecord structs (160 bytes each: Int32
 * label, 13 Float32, 26 UInt32; src/data/criteo.jl:91-95).  Outputs: labels [B] as Float32,
 * dense [B][13], sparse [26][B] (table-major, the layout dlrmb_embedding_fwd takes).
 * (SURVEY.md section 8(f) row 2.) ------------------------------------------------------------- */
int32_t dlrmb_dac_unpack(int32_t device, const void* records, int32_t B, float* labels, float* dense,
                         uint32_t* sparse, dlrmb_stream stream);

/* ---- multi-GPU, table-wise sharded embeddings (new functionality: DLRM.jl is single-process).
 * Exchange buffers are library-owned device allocations that other ranks (one process per GPU)
 * map through CUDA IPC; dlrmb_embedding_fwd_p2p pools this rank's tables for the GLOBAL batch
 * (B_global = B_local * world, sample b belongs to rank b / B_local) and stores each pooled row
 * directly into peer_T[owner of the sample][b_local][slot_map[k]][:] over NVLink -- the lookup and
 * the forward all-to-all in one kernel.  peer_T is a host array of `world` device pointers (this
 * rank's own buffer at index `rank`).  The caller orders the launch against the peers' use of the
 * buffers (a stream-ordered collective after it, see dlrm_jl_b200/sharded.py). ---------------- */
typedef struct dlrmb_xbuf dlrmb_xbuf;
int32_t dlrmb_xbuf_create(int32_t device, int64_t bytes, dlrmb_xbuf** out);
int32_t dlrmb_xbuf_destroy(dlrmb_xbuf* x);
int32_t dlrmb_xbuf_ptr(dlrmb_xbuf* x, void** dev);
int32_t dlrmb_xbuf_ipc_handle(dlrmb_xbuf* x, uint8_t* handle64);
int32_t dlrmb_xbuf_open(int32_t device, const uint8_t* handle64, void** peer_ptr);
int32_t dlrmb_xbuf_close(int32_t device, void* peer_ptr);
int32_t dlrmb_tables_set_slot_map(dlrmb_tables* t, const int32_t* slots);
/* Destination map of the p2p lookups for column-wise sharded tables (dlrmb_shard_plan_cw): local table k's pooled
 * row of sample b lands at columns [col0[k], col0[k] + D) of slot slots[k] in destination rows of `D_dest` floats
 * per slot, i.e. at peer_T[h] + b_local * slots_arg * D_dest + slots[k] * D_dest + col0[k] (slots_arg: the `slots`
 * argument of the lookup call).  col0[k] + D <= D_dest.  dlrmb_tables_set_slot_map(t, s) is the map with col0 = 0
 * and D_dest = D; a later call of either replaces the map.  The 16-byte store path needs D, D_dest and every
 * col0 to be multiples of 4 (and 16-byte aligned peer_T); otherwise the lookups store one float at a time. */
int32_t dlrmb_tables_set_dest_map(dlrmb_tables* t, const int32_t* slots, const int32_t* col0, int32_t D_dest);
int32_t dlrmb_embedding_fwd_p2p(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                                int32_t B_global, int32_t P, float* const* peer_T, int32_t world,
                                int32_t B_local, int32_t slots, dlrmb_stream stream);

/* Training-step form of dlrmb_embedding_fwd_p2p: also sorts / dedups the owned indices for the coming
 * dlrmb_embedding_update_sorted (in extra CTAs of the same launch when B_global * P <= 4096, by the
 * stand-alone sort kernel on the same stream above that). */
int32_t dlrmb_embedding_fwd_p2p_sort(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                                     int32_t B_global, int32_t P, float* const* peer_T, int32_t world,
                                     int32_t B_local, int32_t slots, dlrmb_stream stream);
/* Per-table pooling factors: `P` is a host array of the handle's ntab pooling factors and `idx` the `_mp`
 * layout at B = B_global (table k's [B_global][P_k] block at element B_global * (P_0 + .. + P_{k-1}), the
 * owner layout that dlrmb_comm_a2a_indices_mp / dlrmb_indices_scatter_p2p_mp fill).  The pooled rows are
 * bit-identical to dlrmb_embedding_fwd_mp's.  The _sort_mp form sorts every table for the coming
 * dlrmb_embedding_update_sorted as dlrmb_embedding_fwd_sort_mp does (B_global * P_k <= 4096 inside the
 * lookup launch, larger tables by the stand-alone sorts on the same stream).  Arguments are checked as for
 * the `_mp` and p2p entry points (B_global * max P_k <= max_lookups; DLRMB_ESTATE without a slot map).
 * No allocation, synchronisation or host copy: graph-capturable. */
int32_t dlrmb_embedding_fwd_p2p_mp(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                                   int32_t B_global, const int32_t* P, float* const* peer_T, int32_t world,
                                   int32_t B_local, int32_t slots, dlrmb_stream stream);
int32_t dlrmb_embedding_fwd_p2p_sort_mp(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                                        int32_t B_global, const int32_t* P, float* const* peer_T, int32_t world,
                                        int32_t B_local, int32_t slots, dlrmb_stream stream);

/* Jagged bags (variable length, the layout of dlrmb_embedding_fwd_jagged): `values` / `offsets` / `weights` are the
 * owner's jagged batch of its tables at B = B_global (dlrmb_indices_scatter_p2p_jagged below fills it: bag
 * j * B_global + h * B_local + b is rank h's bag b of the owner's table j) and `L` its host [ntab] lookup counts.  The
 * pooled rows are bit-identical to dlrmb_embedding_fwd_jagged's (pooling 0 sum, 1 mean) or, with `weights` non-null,
 * to dlrmb_embedding_fwd_jagged_weighted's (then pooling must be 0).  They land as for dlrmb_embedding_fwd_p2p_mp.
 * Arguments are checked as for dlrmb_embedding_fwd_jagged and the p2p entry points (L[k] <= max_lookups, B_global =
 * B_local * world; DLRMB_ESTATE without a slot map).  The _sort_ form then sorts the batch for the coming
 * dlrmb_embedding_update_sorted as dlrmb_embedding_sort_jagged / _weighted do (dlrmb_sort_dedup_export works after
 * it).  No allocation, synchronisation or host copy: graph-capturable.  The weights' gradient of a sharded batch
 * (dlrmb_embedding_weight_grad_jagged returned to the samples' ranks) is not provided. */
int32_t dlrmb_embedding_fwd_p2p_jagged(dlrmb_tables* t, const void* values, const void* offsets, const float* weights,
                                       int32_t idx_bytes, int32_t idx_base, int32_t B_global, const int64_t* L,
                                       int32_t pooling, float* const* peer_T, int32_t world, int32_t B_local,
                                       int32_t slots, dlrmb_stream stream);
int32_t dlrmb_embedding_fwd_p2p_sort_jagged(dlrmb_tables* t, const void* values, const void* offsets,
                                            const float* weights, int32_t idx_bytes, int32_t idx_base,
                                            int32_t B_global, const int64_t* L, int32_t pooling, float* const* peer_T,
                                            int32_t world, int32_t B_local, int32_t slots, dlrmb_stream stream);

/* Ordering point of the fused exchanges without NCCL: a flag barrier over IPC-mapped memory, one tiny
 * kernel per call.  Every rank allocates a zero-initialised dlrmb_xbuf of dlrmb_peer_barrier_flag_bytes()
 * (its flag array, mapped by all peers) and a zero-initialised private device buffer of
 * dlrmb_peer_barrier_state_bytes() (epochs; the last word counts waits that timed out after 4 s).
 * dlrmb_peer_barrier(stream): everything this rank stored into peers' buffers earlier on `stream` is
 * visible to a peer once that peer's own barrier call of the same `channel` (0..7) has passed, and
 * vice versa.  `peer_flags` is a host array of `world` device pointers (rank r's flag array at r).
 * Graph-capturable (the epoch lives in device memory).  Every rank must have its own GPU. */
int32_t dlrmb_peer_barrier(int32_t device, uint32_t* const* peer_flags, int32_t world, int32_t rank, int32_t channel,
                           uint32_t* state, dlrmb_stream stream);
int64_t dlrmb_peer_barrier_flag_bytes(void);
int64_t dlrmb_peer_barrier_state_bytes(void);
/* One-shot all-reduce (sum, in place) of a SMALL float buffer over IPC-mapped memory: the bottom MLP's
 * gradients at the end of the data-parallel step, which sit on the critical path and are latency-bound.
 * Every rank allocates a zero-initialised dlrmb_xbuf of 2 * world * n floats (mapped by all peers;
 * `peer_bufs` = host array of the `world` device pointers) and shares the flag arrays / state of
 * dlrmb_peer_barrier (a channel of its own).  push (each rank stores its n floats into its slot of every
 * rank's buffer) -> flag barrier -> every rank sums the slots in rank order: bit-identical sums on all
 * ranks.  n % 4 == 0, data 16-byte aligned.  (world - 1) * n * 4 bytes leave each GPU, so this is for
 * buffers up to about 1 MB; larger ones stay with dlrmb_comm_allreduce_f32 / NCCL. */
int32_t dlrmb_peer_allreduce_f32(int32_t device, float* const* peer_bufs, uint32_t* const* peer_flags, int32_t world,
                                 int32_t rank, int32_t channel, uint32_t* state, float* data, int64_t n,
                                 dlrmb_stream stream);
/* Index exchange by peer stores: idx_local [ntab][B_local][P] (this rank's samples, every table) goes to
 * the owners' index buffers: `dests_dev` is a DEVICE array of ntab pointers, entry k = the owner's buffer
 * [B_global][P] of table k (inside its idx_owned [t_owner][B_global][P]); this rank fills rows
 * [rank * B_local, (rank + 1) * B_local).  Follow with dlrmb_peer_barrier. */
int32_t dlrmb_indices_scatter_p2p(int32_t device, const void* idx_local, int32_t idx_bytes, int32_t ntab,
                                  int32_t B_local, int32_t P, const void* const* dests_dev, int32_t rank,
                                  dlrmb_stream stream);
/* Per-table pooling factors: idx_local is the `_mp` layout at B_local (table k's [B_local][P_k] block at
 * element B_local * (P_0 + .. + P_{k-1})), `P` a host array [ntab] (ntab <= dlrmb_mp_max_tables()), and
 * dests_dev[k] the owner's [B_global][P_k] block of global table k; this rank fills rows
 * [rank * B_local, (rank + 1) * B_local) of it.  No allocation; graph-capturable. */
int32_t dlrmb_indices_scatter_p2p_mp(int32_t device, const void* idx_local, int32_t idx_bytes, int32_t ntab,
                                     int32_t B_local, const int32_t* P, const void* const* dests_dev, int32_t rank,
                                     dlrmb_stream stream);
/* Column-wise sharding: a split table's block goes to every rank holding one of its slices.  Destination i
 * (0 <= i < ndest <= 1024) receives global table dest_table[i]'s block (`dest_table` a host array) at
 * dests_dev[i] + rank * B_local * P_k indices, i.e. rows [rank * B_local, (rank + 1) * B_local) of that holder's
 * [B_global][P_k] block; idx_local and P as for dlrmb_indices_scatter_p2p_mp.  One launch for every destination;
 * no allocation; graph-capturable. */
int32_t dlrmb_indices_scatter_p2p_mp_list(int32_t device, const void* idx_local, int32_t idx_bytes, int32_t ntab,
                                          int32_t B_local, const int32_t* P, int32_t ndest, const int32_t* dest_table,
                                          const void* const* dests_dev, int32_t rank, dlrmb_stream stream);

/* Jagged bags: this rank's jagged batch of B_local bags per table (values, offsets [ntab * B_local + 1] of width
 * idx_bytes, and per-sample `weights` or null) goes into the owners' jagged batches over the global batch.  Host
 * arrays: owner[ntab] (the plan), L_all[world][ntab] (every rank's lookup counts of this step), cap_values[world]
 * (entries each owner's values buffer holds) and peer_values / peer_offsets / peer_weights[world] (device pointers of
 * the owners' mapped buffers; peer_weights null exactly when weights is null).  For owner o with tables j = 0..t-1
 * in ascending global id k_j, L_own[j] = sum over h of L_all[h][k_j]: table j's block of values starts at
 * L_own[0] + .. + L_own[j-1], rank h's entries inside it after those of ranks h' < h, in their own order; offsets has
 * t * B_global + 1 entries, bag j * B_global + h * B_local + b being rank h's bag b of k_j, rebased; weights sit in the
 * positions of their values.  One launch stores this rank's values (and weights) and B_local offsets of every table;
 * rank world - 1 also writes each table's closing entry (j + 1) * B_global.  DLRMB_EINVAL, before any launch, when an
 * owner's total exceeds cap_values[o], a 4-byte total reaches 2^31, or weights and peer_weights disagree.  Follow with
 * dlrmb_peer_barrier.  No allocation; graph-capturable.  (NCCL exchanges of jagged batches and column-wise splits of
 * jagged tables are not provided: dlrmb_comm_a2a_indices* and the _list scatter stay fixed-width.) */
int32_t dlrmb_indices_scatter_p2p_jagged(int32_t device, const void* values, const void* offsets, const float* weights,
                                         int32_t idx_bytes, int32_t ntab, int32_t B_local, const int32_t* owner,
                                         const int64_t* L_all, int32_t world, int32_t rank, void* const* peer_values,
                                         void* const* peer_offsets, float* const* peer_weights,
                                         const int64_t* cap_values, dlrmb_stream stream);

/* Interaction backward fused with the gradient exchange: as dlrmb_interaction_bwd, but the gradient
 * row of feature slot f >= 1 of local sample b is stored at
 *   dests[f].base + (sample_offset + b) * dests[f].sample_stride + dests[f].offset   (floats)
 * i.e. straight into the gradient buffer [B_global][tables of that rank][D] of the rank that owns
 * table f-1 (a dlrmb_xbuf mapped over NVLink); slot 0 only contributes to dx.  `dests` is a DEVICE
 * array of F entries (entry 0 unused). */
typedef struct dlrmb_slot_dest {
    float* base;
    int64_t sample_stride;
    int64_t offset;
} dlrmb_slot_dest;
int32_t dlrmb_interaction_bwd_scatter(int32_t device, const float* dOut, const float* T, int32_t B,
                                      int32_t F, int32_t d, int32_t pad_to_mul,
                                      const dlrmb_slot_dest* dests, int64_t sample_offset, float* dx,
                                      dlrmb_stream stream);
/* Column pieces (column-wise sharded tables): `dests` is a DEVICE array [F][Q] and entry (f, q) receives columns
 * [q * d / Q, (q + 1) * d / Q) of slot f's gradient row, at
 *   dests[f * Q + q].base + (sample_offset + b) * dests[f * Q + q].sample_stride + dests[f * Q + q].offset
 * (floats; the offset addresses the piece's first column).  A slot held whole gets Q entries pointing at
 * consecutive column ranges of one row.  Q a power of two in 1..32, d / Q a multiple of 4; Q = 1 is
 * dlrmb_interaction_bwd_scatter.  Same products in the same order: the pieces carry the bits of dT. */
int32_t dlrmb_interaction_bwd_scatter_cols(int32_t device, const float* dOut, const float* T, int32_t B,
                                           int32_t F, int32_t d, int32_t pad_to_mul, const dlrmb_slot_dest* dests,
                                           int32_t Q, int64_t sample_offset, float* dx, dlrmb_stream stream);

/* ---- collectives of the sharded path (new functionality; one process per GPU, NCCL over NVLink).
 * A non-Python host runs BASELINE config 4 with these: rank 0 calls dlrmb_comm_unique_id, carries the 128
 * bytes to the other ranks (file, socket, MPI ...), every rank calls dlrmb_comm_create.  Calls are
 * stream-ordered and must be issued in the same order on every rank.  NCCL is bound at run time
 * (libnccl.so.2 via dlopen), so single-GPU users do not need it.  `owner` is the host array [ntab] of
 * dlrmb_shard_plan (rank owning each table: table count balanced first, bytes second, the big tables
 * on different GPUs); B_global = B_local * world, sample b of the global batch belongs to rank
 * b / B_local.
 *   dlrmb_comm_a2a_indices   idx_local [ntab][B_local][P]  ->  idx_owned [t_mine][B_global][P]
 *   dlrmb_comm_a2a_fwd       pooled [B_global][t_mine][D] (dlrmb_embedding_fwd with slot0 = 0 on the owner)
 *                            ->  T [B_local][1 + ntab][D], slot 1 + k for table k (slot 0 is left for x)
 *   dlrmb_comm_a2a_bwd       dT [B_local][1 + ntab][D]  ->  grads [B_global][t_mine][D] on each owner
 *                            (then dlrmb_embedding_bwd_sgd with slot0 = 0)
 *   dlrmb_comm_allreduce_f32 in-place sum of the data-parallel dense gradients
 *   dlrmb_comm_allgather     nbytes per rank, device buffers (e.g. the 64-byte dlrmb_xbuf IPC handles that
 *                            set up the fused peer-store exchanges above)
 * The first a2a call sizes a staging buffer (cudaMalloc); later calls with the same geometry do not
 * allocate and can be captured into a CUDA graph.
 * Per-table pooling factors (`P` = host array [ntab] of P_k >= 1):
 *   dlrmb_shard_plan_mp      equal P_k: exactly dlrmb_shard_plan.  Mixed: tables dealt longest first
 *                            (descending P_k, then rows, then id), each to the rank with the smallest sum
 *                            of P_k so far (ties: fewer rows, then the lower rank)
 *   dlrmb_comm_a2a_indices_mp  idx_local (`_mp` layout at B_local) -> idx_owned, the `_mp` layout of this
 *                            rank's tables (ascending global id) at B_global: table j's [B_global][P_j] block
 *                            starts at B_global * (sum of P_i of the owned tables before it), rank h's samples
 *                            are its rows [h * B_local, (h + 1) * B_local).  dlrmb_embedding_fwd_mp /
 *                            _sort_mp / _bwd_sgd_mp read it with the owned tables' P as is.
 * The a2a calls take one owner per table, so they serve table-wise plans only; a column-wise plan
 * (dlrmb_shard_plan_cw below) goes through the peer-store exchanges.
 * Column-wise sharding of hot tables (S = max_col_shards, a power of two; D / S a multiple of 4 when S > 1):
 *   dlrmb_shard_plan_cw      shards[k] = c_k, the number of column slices of table k (a power of two <= min(S,
 *                            world)); owner[k * S + j] = rank holding slice j, columns [j * D / c_k, (j + 1) * D / c_k),
 *                            -1 for j >= c_k.  Rule: start with every c_k = 1; repeatedly take the table with the
 *                            largest P_k / c_k (ties: more rows, then lower id) and double its c_k, until
 *                            P_k * world <= c_k * sum(P) or 2 * c_k > min(S, world).  Nothing split: exactly
 *                            dlrmb_shard_plan_mp's owners in owner[k * S].  Otherwise the slices are dealt longest
 *                            first (descending P_k / c_k, then rows, then k, then j), each to the rank with the
 *                            smallest sum of P_k / c_k so far among those holding no slice of k (ties: fewer
 *                            rows * D / c_k, then the lower rank).  Column j of a pooled row is an ordered sum of
 *                            column j of the rows it gathers, so a slice's holder produces exactly the columns the
 *                            whole-table lookup would. */
typedef struct dlrmb_comm dlrmb_comm;
int32_t dlrmb_shard_plan(int32_t ntab, const int64_t* rows, int32_t world, int32_t* owner);
int32_t dlrmb_shard_plan_mp(int32_t ntab, const int64_t* rows, const int32_t* P, int32_t world, int32_t* owner);
int32_t dlrmb_shard_plan_cw(int32_t ntab, const int64_t* rows, const int32_t* P, int32_t world, int32_t D, int32_t S,
                            int32_t* shards, int32_t* owner);
int32_t dlrmb_comm_unique_id(uint8_t* id128);
int32_t dlrmb_comm_create(int32_t device, const uint8_t* id128, int32_t rank, int32_t world, dlrmb_comm** out);
int32_t dlrmb_comm_destroy(dlrmb_comm* c);
int32_t dlrmb_comm_info(const dlrmb_comm* c, int32_t* rank, int32_t* world);
int32_t dlrmb_comm_a2a_indices(dlrmb_comm* c, const int32_t* owner, int32_t ntab, const void* idx_local,
                               int32_t idx_bytes, int32_t B_local, int32_t P, void* idx_owned, dlrmb_stream stream);
int32_t dlrmb_comm_a2a_indices_mp(dlrmb_comm* c, const int32_t* owner, int32_t ntab, const void* idx_local,
                                  int32_t idx_bytes, int32_t B_local, const int32_t* P, void* idx_owned,
                                  dlrmb_stream stream);
int32_t dlrmb_comm_a2a_fwd(dlrmb_comm* c, const int32_t* owner, int32_t ntab, const float* pooled, int32_t B_local,
                           int32_t D, float* T, dlrmb_stream stream);
int32_t dlrmb_comm_a2a_bwd(dlrmb_comm* c, const int32_t* owner, int32_t ntab, const float* dT, int32_t B_local,
                           int32_t D, float* grads, dlrmb_stream stream);
int32_t dlrmb_comm_allreduce_f32(dlrmb_comm* c, float* buf, int64_t n, dlrmb_stream stream);
int32_t dlrmb_comm_allgather(dlrmb_comm* c, const void* send, void* recv, int64_t nbytes, dlrmb_stream stream);

/* dx of dot_back alone (src/model/interact.jl:434: dx = dOut[1:d, :] + dT[1:d, :]) without the rest of dT:
 * what the bottom MLP's backward waits for.  The sharded step launches it in front of
 * dlrmb_interaction_bwd_scatter (on another stream), so the bottom MLP's backward overlaps the gradient
 * exchange.  Same bits as the dx of the full kernels for the specialised shapes.  Needs d % 4 == 0. */
int32_t dlrmb_interaction_bwd_dx(int32_t device, const float* dOut, const float* T, int32_t B, int32_t F, int32_t d,
                                 int32_t pad_to_mul, float* dx, dlrmb_stream stream);

/* ---- host-buffer entry points: every pointer is host memory (pageable or pinned); this is
 * the form a CPU-resident DLRM.jl model calls.  Copies run inside the call. -------------- */
int32_t dlrmb_embedding_fwd_host(dlrmb_tables* t, const void* idx, int32_t idx_bytes,
                                 int32_t idx_base, int32_t B, int32_t P, float* out,
                                 int32_t slots, int32_t slot0);
int32_t dlrmb_interaction_fwd_host(dlrmb_tables* t, float* T, const float* x, int32_t B, int32_t F,
                                   int32_t d, int32_t pad_to_mul, float* out);
int32_t dlrmb_interaction_bwd_host(dlrmb_tables* t, const float* dOut, const float* T, int32_t B,
                                   int32_t F, int32_t d, int32_t pad_to_mul, float* dT, float* dx);
int32_t dlrmb_embedding_bwd_sgd_host(dlrmb_tables* t, const void* idx, int32_t idx_bytes,
                                     int32_t idx_base, int32_t B, int32_t P, const float* dT,
                                     int32_t slots, int32_t slot0, float lr);

#ifdef __cplusplus
}
#endif
#endif /* DLRM_B200_H */
