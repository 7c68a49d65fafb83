/*
 * locator_b200 -- C ABI of the B200-native Locator hot path.
 *
 * The reference (kr-colab/locator) is pure Python with no FFI of its own; its
 * stable interface is the `locator` CLI, its output files and the function
 * surface of locator/locator.py.  This header is the boundary a maintainer
 * binds (ctypes stub in INTEGRATION.md) to replace, one for one:
 *
 *   reference (locator/locator.py)                 entry points here
 *   ---------------------------------------------  -----------------------------------
 *   filter_snps            :265-281  (allel count_  loc_site_stats, loc_pack_sites,
 *     alleles / is_biallelic / to_allele_counts)      loc_patch_calls
 *   split_train_test       :295-308  (ac[:, idx])   loc_gather_rows
 *   bootstrap column gather :648-653                loc_gather_cols
 *   jacknife column replace :721-727                loc_replace_cols
 *   uint8 [n, K] matrices in/out of the API         loc_pack_counts, loc_unpack_counts
 *   load_network           :311-327                 loc_model_create / _init / _set_weight / _get_weight
 *   load_callbacks         :330-362                 loc_model_set_schedule (device-side callback state)
 *   train_network / fit    :365-376                 loc_train_epochs, loc_train_step
 *   load_weights(best)     :380,386                 loc_restore_best
 *   model.predict          :414,441                 loc_predict
 *   validation pass of fit :374                     loc_eval
 *   history                :468-469                 loc_model_history, loc_model_state
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; loc_last_error()
 *     gives the message for the calling thread.
 *   - pointers prefixed d_ are CUDA device pointers owned by the caller (torch
 *     tensors); h_ are host pointers.  No torch types cross this boundary.
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *     is asynchronous unless the function returns host data (documented below).
 *   - a loc_model is bound to the device current at creation and is not
 *     thread-safe: one host thread / process per GPU.
 *   - packed genotype matrix: sample-major, 2 bits per genotype (alt-allele count
 *     0/1/2), 16 genotypes per little-endian uint32 (SNP k of a row lives in word
 *     k/16, bits 2*(k%16)..+1), row pitch `row_words` uint32 (>= ceil(K/16),
 *     multiple of 4 so rows are 16-byte aligned); pad bits are zero.
 *   - there is NO CPU fallback: every entry point fails if CUDA is unavailable.
 */
#ifndef LOCATOR_B200_H
#define LOCATOR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LOC_ABI_VERSION 1
#define LOC_MAX_BATCH 32        /* rows of one batch tile: steps of up to 32 rows run on the fused tensor-core kernels */
#define LOC_MAX_BATCH_SIZE 256  /* largest --batch_size: steps of 33..256 rows go through the stack in 32-row chunks   */

typedef struct loc_model loc_model;

/* Snapshot of the device-side training/callback state (loc_model_state). */
typedef struct loc_state {
  int32_t t;            /* optimizer iterations done                         */
  int32_t epoch;        /* epochs completed                                  */
  int32_t stopped;      /* EarlyStopping fired (or max_epochs reached)       */
  int32_t improved;     /* last finished epoch improved val_loss             */
  int32_t best_epoch;   /* epoch index of the checkpointed weights, -1 none  */
  int32_t es_wait;
  int32_t rlr_wait;
  int32_t nonfinite;    /* a non-finite loss was seen                        */
  float lr;             /* current learning rate                             */
  float ckpt_best;      /* best val_loss so far (+inf before the first)      */
  float last_loss;
  float last_val_loss;
} loc_state;

int loc_abi_version(void);
const char* loc_last_error(void);
/* Name of the first-layer kernel family a width-256 model runs on the sm_100a device the library is
 * built for: "tcgen05".  loc_model_impl gives the family a particular model uses. */
const char* loc_l1_impl(void);

/* ---------------- genotype ingest (K1/K2) ---------------- */

/* Per-site allele statistics over d_gt int8 [nvar][nsamp][2] (-1 = missing).
 * d_n_alleles[v] = number of distinct allele indices observed (allel allelism),
 * d_alt_count[v] = copies of allele index 1, d_n_missing[v] = calls with any
 * negative allele.  d_keep[v] = 1 iff n_alleles == 2 and (min_mac == 1 or
 * alt_count >= min_mac)  -- locator.py:267-273.  Any output pointer may be NULL. */
int loc_site_stats(const int8_t* d_gt, int64_t nvar, int64_t nsamp, int32_t min_mac,
                   int32_t* d_n_alleles, int32_t* d_alt_count, int32_t* d_n_missing,
                   uint8_t* d_keep, void* stream);

/* The kept sites in ascending order, on the device: d_site_idx[0 .. *d_count) = { v : d_keep[v] != 0 },
 * *d_count (device int64) = their number.  d_site_idx needs room for nvar entries.  The reference builds the
 * same list on the host (boolean-mask indexing of the genotype array, locator.py:269,273).  Async. */
int loc_compact_sites(const uint8_t* d_keep, int64_t nvar, int64_t* d_site_idx, int64_t* d_count, void* stream);

/* Missing calls of the kept sites in row-major (site, sample) order -- np.nonzero(is_missing), the order in which
 * replace_md draws its imputed values (locator.py:255-261).  Two phases:
 *   d_k == NULL: d_offsets[0 .. K] = exclusive prefix sums of d_n_missing[d_site_idx[k]] (d_offsets[K] = total);
 *   otherwise  : d_k[i] = kept-site index k, d_samp[i] = sample of missing call i, i < d_offsets[K].
 * d_n_missing is loc_site_stats' output over all nvar sites.  Async. */
int loc_missing_calls(const int8_t* d_gt, int64_t nvar, int64_t nsamp, const int64_t* d_site_idx, int64_t K,
                      const int32_t* d_n_missing, int64_t* d_offsets, int64_t* d_k, int64_t* d_samp, void* stream);

/* d_sums[k] = sum over the n rows of the packed matrix of SNP k's allele count (int64; jacknife allele
 * frequencies over ALL samples, locator.py:714-717).  Async. */
int loc_site_sums(const uint32_t* d_packed, int64_t n, int64_t K, int64_t row_words, int64_t* d_sums, void* stream);

/* Pack the K sites d_site_idx[0..K) of d_gt into the 2-bit sample-major matrix:
 * genotype = number of index-1 alleles of the call (missing/other alleles count 0)
 * -- GenotypeArray.to_allele_counts()[:, :, 1], locator.py:277. */
int loc_pack_sites(const int8_t* d_gt, int64_t nvar, int64_t nsamp, const int64_t* d_site_idx,
                   int64_t K, uint32_t* d_packed, int64_t row_words, void* stream);

/* Overwrite individual genotypes (imputation results of replace_md, :258-261):
 * packed[d_samp[i]][d_k[i]] = d_val[i], i < n.  (k indexes packed columns.) */
int loc_patch_calls(uint32_t* d_packed, int64_t row_words, const int64_t* d_k,
                    const int64_t* d_samp, const uint8_t* d_val, int64_t n, void* stream);

/* uint8 allele-count matrix [n][K] (row-major, values 0/1/2) <-> packed. */
int loc_pack_counts(const uint8_t* d_counts, int64_t n, int64_t K, uint32_t* d_packed,
                    int64_t row_words, void* stream);
int loc_unpack_counts(const uint32_t* d_packed, int64_t n, int64_t K, int64_t row_words,
                      uint8_t* d_counts, void* stream);
/* The same from a HOST matrix (the uint8 [n, K] traingen / testgen / predgen arrays the reference hands to
 * model.fit / model.predict, :367-376, :414): row blocks staged through two pinned buffers by LOC_UPLOAD_THREADS
 * host threads (default 4), copied and packed on `stream` while the next block is staged.  Returns once the
 * last block is packed. */
int loc_upload_pack_counts(const uint8_t* h_counts, int64_t n, int64_t K, uint32_t* d_packed,
                           int64_t row_words, void* stream);

/* out[r] = in[d_rows[r]] for r < n_out (sample split, :303-307). */
int loc_gather_rows(const uint32_t* d_in, int64_t row_words, const int64_t* d_rows, int64_t n_out,
                    uint32_t* d_out, void* stream);

/* out[r][k] = in[r][d_cols[k]], k < K_out (bootstrap site_order, :651-653;
 * max_SNPs subsample, :279). */
int loc_gather_cols(const uint32_t* d_in, int64_t n, int64_t row_words_in, const int64_t* d_cols,
                    int64_t K_out, uint32_t* d_out, int64_t row_words_out, void* stream);

/* packed[r][d_sites[i]] = d_vals[i*n + r] (jacknife, :726-727; sites distinct). */
int loc_replace_cols(uint32_t* d_packed, int64_t n, int64_t row_words, const int64_t* d_sites,
                     int64_t nsites, const uint8_t* d_vals, void* stream);

/* Host helper for load_genotypes' zarr branch (locator.py:187-194): decompress one Blosc-1 frame
 * (LZ4 codec, byte shuffle or none -- zarr's default compressor, what allel.vcf_to_zarr writes)
 * from host memory into host memory.  Returns the decompressed size or < 0 on error. */
int64_t loc_blosc_decompress(const uint8_t* h_src, int64_t src_len, uint8_t* h_dst, int64_t dst_len);
/* One plain Zstandard frame (zarr compressor id "zstd"; also the streams of Blosc frames with cname "zstd"):
 * the system's libzstd.so.1 is bound at first use.  Returns the decompressed size or < 0. */
int64_t loc_zstd_decompress(const uint8_t* h_src, int64_t src_len, uint8_t* h_dst, int64_t dst_len);

/* Host helpers for load_genotypes' VCF branch (allel.read_vcf, locator.py:195-199): data lines of an
 * uncompressed VCF text buffer -> GT int8 [n_variants][n_samples][2] (missing allele -1, haploid call ->
 * second allele -1, first two alleles of a polyploid call) and POS.  loc_vcf_count gives n_variants;
 * loc_vcf_parse_gt parses with n_threads host threads and fails (return 1) on a line it cannot parse. */
int64_t loc_vcf_count(const char* h_buf, int64_t len);
int loc_vcf_parse_gt(const char* h_buf, int64_t len, int64_t n_samples, int64_t n_variants, int8_t* h_gt, int64_t* h_pos,
                     int32_t n_threads);

/* Host helper for the index draws that bound the jacknife sweep and replace_md (locator.py:722-727,
 * :258-261): consecutive numpy RandomState.binomial(n, p[i]) draws -- `reps` per p[i], sites in order --
 * taken from the MT19937 state of np.random.get_state() (key[624], position), which is advanced in place
 * exactly as numpy would advance it.  out uint8 [n_p][reps].  Returns 0; 1 if some (n, p[i]) needs numpy's
 * BTPE branch (min(p, 1-p) * n > 30) or n > 255 -- nothing is drawn then; 2 for p outside [0, 1]. */
int loc_np_legacy_binomial(uint32_t* mt_key, int32_t* mt_pos, int64_t n, const double* h_p, int64_t n_p, int64_t reps,
                           uint8_t* h_out);

/* RandomState.permutation(n) from the same state (numpy's legacy Fisher-Yates over arange(n)); the first
 * `size` entries are np.random.choice(n, size, replace=False) (split :299, max_SNPs :279, jacknife :722). */
int loc_np_legacy_permutation(uint32_t* mt_key, int32_t* mt_pos, int64_t n, int64_t* h_out);

/* ---------------- model (K3-K7) ---------------- */

/* BN(K) -> Dense(width, elu) x nlayers (Dropout after the floor(nlayers/2)-th)
 * -> Dense(2) -> Dense(2); Adam(1e-3, .9, .999, 1e-7).  batch_size <= LOC_MAX_BATCH_SIZE
 * (locator.py:69,371; steps of more than LOC_MAX_BATCH rows: batch statistics over the whole step,
 * 32-row chunks through the hidden stack, one pass over W1 | m | v -- csrc/bigbatch.cu; such models
 * cannot be sharded), nlayers >= 2.  Allocates parameters, Adam state, best-weights snapshot and
 * workspaces on the current device. */
int loc_model_create(loc_model** out, int64_t K, int32_t width, int32_t nlayers, int32_t batch_size,
                     float dropout_prop, int32_t max_epochs);
/* Replicate runs (--bootstrap / --windows: locator.py:519-583, :609-681 build one model per replicate and call
 * keras.backend.clear_session() after each, :681) create and drop models all the time; destroyed handles are kept
 * in a small pool (LOC_MODEL_POOL handles, default 8, 0 = off) and loc_model_create re-uses one whose buffers
 * fit (same width / nlayers, K within [0.6, 1] of its capacity), zeroed exactly like a fresh handle, instead
 * of ~35 cudaMalloc / cudaFree calls per replicate.  loc_model_pool_clear() releases the pool's device memory. */
int loc_model_destroy(loc_model* m);
int loc_model_pool_clear(void);
/* Diagnostics (LOC_TIMELINE=1 in the environment before the first model is created): the step kernels log
 * (globaltimer ns, tag << 32 | model number) at the start and end of their first and last blocks; this copies up
 * to max_records pairs to h_out, clears the log and returns the number of records. */
int64_t loc_debug_timeline(uint64_t* h_out, int64_t max_records);
/* First-layer kernel family this model actually runs: "tcgen05" or "simt". */
const char* loc_model_impl(const loc_model* m);
/* Hidden-stack kernel family this model actually runs: "tcgen05" (width 256, nlayers up to 14) or "simt" (the
 * CUDA-core stack: other widths, deeper width-256 stacks -- behind the tcgen05 first layer there). */
const char* loc_model_hidden_impl(const loc_model* m);
/* Deepest nlayers in [2, 64] that loc_model_create can build at this width: the CUDA-core hidden stack's layout
 * (needed by every model) has at least one weight slot in shared memory at some admissible cluster size.  0: no
 * nlayers fits (the widths above 320 except 384), or the width is not a multiple of 32 in [32, 1024].  Host arithmetic, no
 * device needed; an upper bound -- loc_model_create also needs the device to schedule the cluster. */
int32_t loc_hidden_max_nlayers(int32_t width);

/* Philox glorot-uniform kernels, zero biases, gamma 1 / beta 0 / moving mean 0 /
 * moving var 1, zero Adam state, reset optimizer + callback state. `seed` also
 * keys the dropout masks. */
int loc_model_init(loc_model* m, uint64_t seed, void* stream);

/* Keras weight order: [gamma, beta, moving_mean, moving_var, W1, b1, ..., Wo1, bo1, Wo2, bo2],
 * kernels [in, out] row-major fp32.  set/get copy between HOST memory and the model
 * and synchronise the stream. */
int loc_model_num_weights(const loc_model* m);
int64_t loc_model_weight_size(const loc_model* m, int32_t idx);
int loc_model_set_weight(loc_model* m, int32_t idx, const float* h_src, int64_t n, void* stream);
int loc_model_get_weight(loc_model* m, int32_t idx, float* h_dst, int64_t n, void* stream);
/* Adam moments of trainable weight idx (idx 2,3 are not trainable -> error). */
int loc_model_get_adam(loc_model* m, int32_t idx, float* h_m, float* h_v, int64_t n, void* stream);

/* ---- one model sharded over SNPs (tensor parallelism; SURVEY.md section 8(f)2) ----
 * A shard is a model created with K = its own number of SNP columns.  It owns those rows of W1 (+ Adam
 * state) and their BatchNorm vectors; the hidden stack is replicated.  The only exchange per forward pass
 * is the sum over shards of the [32][width] first-layer pre-activation tile.
 *
 * loc_model_set_shard (before loc_model_init): this model's columns are [k_offset, k_offset + K) of a
 * K_global-column model -- glorot limit and random stream of W1 are those of the whole layer, so the
 * shards together initialise exactly as the unsharded model with the same seed.
 *
 * loc_model_set_exchange: `fn(ctx, d_tile, n, stream)` is called on the host while kernels are being
 * enqueued, every time a tile is complete; it must enqueue on `stream` an in-place sum of d_tile
 * (n = 32 * width floats, device memory owned by the caller) over all shards, leaving bitwise identical
 * results on every shard (e.g. ncclAllReduce / torch.distributed.all_reduce); returns 0 on success.
 * fn = NULL removes the hook.  Needs the tcgen05 kernels (width 256); not combined with replicate groups. */
typedef int (*loc_exchange_fn)(void* ctx, float* d_tile, int64_t n, void* stream);
int loc_model_set_shard(loc_model* m, int64_t k_offset, int64_t K_global);
int loc_model_set_exchange(loc_model* m, loc_exchange_fn fn, void* ctx, float* d_tile);

/* Peer-memory exchange for sharded models on one NVLink / NVSwitch box (replaces the host hook: no library
 * collective, no host call per step).  Every shard process: loc_tp_create -> loc_tp_handle (64-byte
 * cudaIpc handle of its buffer) -> exchange the handles by any host means -> loc_tp_connect with all
 * `world` handles in rank order -> loc_model_set_tp.  Per forward pass a shard then reduces its partial
 * tiles, stores the result into its slot of every peer's buffer over NVLink and raises flags there; the
 * hidden-stack kernel sums the slots in rank order.  loc_tp_error != 0: a peer never arrived (2 s timeout). */
typedef struct loc_tp loc_tp;
int loc_tp_create(loc_tp** out, int32_t rank, int32_t world, int32_t width);
int loc_tp_handle(loc_tp* tp, uint8_t* h_handle64);
int loc_tp_connect(loc_tp* tp, const uint8_t* h_handles /* [world][64] */);
int loc_tp_error(loc_tp* tp);
int loc_tp_destroy(loc_tp* tp);
int loc_model_set_tp(loc_model* m, loc_tp* tp);

/* Number of CTAs (= SMs used, = split-K partial tiles) of the tcgen05 first-layer kernels; default: all SMs.
 * The plain backward + Adam kernel is memory-bound and as fast on SMs - 16 as on all of them (B200: 113 vs
 * 114 us at K = 100k), the variant with the fused next forward loses 3 %.  The value fixes the fp32
 * summation order of the layer: set it the same way for runs that must agree bit for bit.  SMs - 16 is what
 * the ring schedule of loc_group_train_epochs needs (one cluster of the hidden stack fits next to the kernel). */
int loc_model_set_l1_ctas(loc_model* m, int32_t n_ctas);

/* lr, EarlyStopping patience (ReduceLROnPlateau patience = patience/6), and
 * reset of the callback state machine (best = +inf, waits = 0, epoch = 0). */
int loc_model_set_schedule(loc_model* m, float lr, int32_t patience);

/* Data the epochs run on (device memory owned by the caller, must outlive use).
 * d_locs: float32 [n][2] normalised targets. */
int loc_model_bind_train(loc_model* m, const uint32_t* d_packed, int64_t n, int64_t row_words,
                         const float* d_locs);
int loc_model_bind_val(loc_model* m, const uint32_t* d_packed, int64_t n, int64_t row_words,
                       const float* d_locs);

/* Test hook: use d_keep[step][32 * ceil(batch_size / 32)][width] (uint8 0/1) as the dropout keep
 * mask of optimizer step `step` instead of Philox; NULL restores Philox. */
int loc_model_set_dropout_masks(loc_model* m, const uint8_t* d_keep, int64_t nsteps);

/* One optimizer step on training rows d_rows[0..nb) (indices into the bound
 * training matrix).  Async.  Batch loss is added to the running epoch mean. */
int loc_train_step(loc_model* m, const int32_t* d_rows, int32_t nb, void* stream);

/* n_epochs epochs: epoch e visits rows d_perms[e*n_train .. +n_train) in slices
 * of batch_size (last partial), then the validation pass at batch 32, then the
 * callback state machine (checkpoint-best / early-stop / reduce-LR) and the
 * device-side snapshot, all on the GPU.  Async; epochs after the stop epoch are
 * no-ops.  History rows are appended per epoch.
 * Scheduling (width 256, unsharded): inside an epoch the step's kernels -- hidden stack, small-layer update,
 * first-layer backward + Adam + next step's forward -- are queued on `stream` as programmatic dependent launches
 * that hand over through device-side flags instead of kernel boundaries (DESIGN.md section 4, "Chained step");
 * results are bit-identical to plain launches (environment LOC_NO_CHAIN=1).  Do not enqueue unrelated work that
 * reads this model's buffers on another stream without synchronising with `stream` first. */
int loc_train_epochs(loc_model* m, const int32_t* d_perms, int32_t n_epochs, void* stream);

/* Part of an epoch on the same schedule as loc_train_epochs (the production path: every first-layer backward
 * also runs the next step's forward): optimizer steps [step0, step0 + n_steps) of the epoch whose batch order
 * is d_perm[0 .. n_train) -- step s trains on rows d_perm[s*batch_size ..).  The span must lie inside the
 * epoch.  When it ends the epoch, the validation pass, callbacks and checkpoint follow exactly as in
 * loc_train_epochs (validation data must be bound); consecutive calls that continue the same d_perm keep the
 * fused forward across the call boundary.  Callers that want model.fit semantics use loc_train_epochs; this
 * entry exists for partial epochs (bench.py --steps K, progress reporting inside long epochs).  Async. */
int loc_train_steps(loc_model* m, const int32_t* d_perm, int32_t step0, int32_t n_steps, void* stream);

/* Replicate group (bootstrap / window models trained side by side on one GPU, locator.py:519-583 and
 * :609-681 run them one after the other): the same as loc_train_epochs for n_models <= 8 independent models.
 * Models must share width, nlayers, batch size and training-set size (true for the replicates of one run)
 * and one kernel family: all tcgen05 (width 256, nlayers <= 14) or all CUDA-core (other widths).  Width 256
 * with 15..21 layers (tcgen05 first layer, CUDA-core hidden stack) and groups mixing families are refused:
 * such models train one at a time.  d_perms[g] is model g's batch order.  Every model ends bit-identical to
 * the same model trained alone.  Two schedules:
 *   ring     (tcgen05 models of >= 32768 SNPs whose first-layer kernels leave 16 SMs free,
 *            loc_model_set_l1_ctas): the hidden stack of one model runs concurrently with the first-layer
 *            backward + Adam of the previous model of its ring (programmatic dependent launch inside one stream);
 *   lockstep (otherwise, and always for CUDA-core models): the hidden stacks of all models share one launch
 *            (one cluster per model), the first-layer kernels run back to back.
 * Environment LOC_GROUP_SCHEDULE=ring|lockstep overrides the choice by size for tcgen05 models.
 * Models of batch_size > 32 have a third schedule, whatever LOC_GROUP_SCHEDULE says: per step, the batch
 * statistics of all models in one launch; on tcgen05 each model's wide first-layer forward, the 32-row chunks
 * of whole models packed into shared hidden-stack launches (floor(8 / chunks) models per launch) and one step
 * end for all models; on CUDA cores, chunk by chunk, every model's first-layer forward and then that chunk of
 * every model in one hidden-stack launch; then the first-layer backwards back to back while the small-layer
 * updates run on side streams. */
int loc_group_train_epochs(loc_model** models, int32_t n_models, const int32_t* const* d_perms, int32_t n_epochs,
                           void* stream);

/* Mean Euclidean loss (Keras evaluate semantics, batch 32) in inference mode.
 * Synchronises; result in *h_loss. */
int loc_eval(loc_model* m, const uint32_t* d_packed, int64_t n, int64_t row_words, const float* d_locs,
             float* h_loss, void* stream);

/* Inference-mode forward of n rows -> d_out float32 [n][2] (normalised units). Async. */
int loc_predict(loc_model* m, const uint32_t* d_packed, int64_t n, int64_t row_words, float* d_out,
                void* stream);

/* Copy the best-val_loss snapshot back into the live weights (load_weights). Async. */
int loc_restore_best(loc_model* m, void* stream);
/* Force a snapshot of the live weights (used by tests). Async. */
int loc_snapshot(loc_model* m, void* stream);

/* Synchronising reads of device-side state / history ([epoch][3] = loss, val_loss, lr).  loc_model_state fails
 * (non-zero, loc_last_error) if a kernel of a chained step gave up waiting for its producer (2 s): an internal
 * error that invalidates the model's results instead of hanging the GPU. */
int loc_model_state(loc_model* m, loc_state* h_out, void* stream);
int loc_model_history(loc_model* m, float* h_out, int32_t max_rows, void* stream);

/* Profiling / test hook: launch ONE stage of an optimizer step on rows d_rows[0..nb):
 * 0 = first-layer forward, 1 = hidden stack (fwd + loss + bwd), 2 = first-layer backward + Adam,
 * 3 = small-layer update, 4 = first-layer backward + Adam with the next step's forward fused in (tcgen05 path).
 * Stages read the scratch the previous ones left.  Async. */
int loc_debug_stage(loc_model* m, int32_t stage, const int32_t* d_rows, int32_t nb, void* stream);

/* Test hook: copy a scratch buffer to the host (synchronises).  which: 0 = split-K partial tiles of
 * Z1 [n_partials][32][width], 1 = dz of every Dense(width) layer [nlayers][32][width] (slot 0 = dZ1),
 * 2 = activations [nlayers][32][width].  Returns the number of floats (written: min(count, max_n)), < 0 on error. */
int64_t loc_debug_read(loc_model* m, int32_t which, float* h_dst, int64_t max_n, void* stream);

/* Number of kernel launches this library has issued in this process (bench.py's gpu_launches). */
int64_t loc_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* LOCATOR_B200_H */
