// Internal layout of a loc_model and the launch interfaces between the translation units.
//
// One optimizer step of the reference (Keras fit on BN -> Dense(H,elu) x L -> Dense(2) -> Dense(2),
// locator/locator.py:311-327,367-376) is four launches here:
//
//   L1 forward   (l1_simt.cu / l1_tc.cu)  batch BN statistics + folded-BN first Dense, split over SNPs;
//                                         every CTA leaves a partial [32][H] tile of Z1
//   hidden       (hidden.cu)              one thread-block cluster: reduce the partials, layers 1..L-1,
//                                         Dense(2), Dense(2), loss, and the whole backward chain down to dZ1
//   L1 backward  (l1_simt.cu / l1_tc.cu)  streams W1, m, v once: dW1 + Adam fused, BN gamma/beta Adam
//   hidden update(hidden.cu)              dW + Adam of the small layers (off the critical path)
#pragma once
#include "common.cuh"

namespace loc {

constexpr int kMaxB = LOC_MAX_BATCH;  // batch rows per step (MMA N / K extent)
constexpr int kF1Chunk = 64;          // SNPs per inner chunk of the SIMT first-layer kernels

// Offsets (in floats) of the small parameters inside loc_model::small / m_small / v_small / best_small.
struct SmallLayout {
  int H, L;
  __host__ __device__ int64_t b1() const { return 0; }
  __host__ __device__ int64_t Wh(int i) const { return (int64_t)H + (int64_t)(i - 1) * H * H; }  // layer i in 1..L-1
  __host__ __device__ int64_t bh(int i) const { return (int64_t)H + (int64_t)(L - 1) * H * H + (int64_t)(i - 1) * H; }
  __host__ __device__ int64_t Wo1() const { return (int64_t)H + (int64_t)(L - 1) * H * H + (int64_t)(L - 1) * H; }
  __host__ __device__ int64_t bo1() const { return Wo1() + 2 * H; }
  __host__ __device__ int64_t Wo2() const { return bo1() + 2; }
  __host__ __device__ int64_t bo2() const { return Wo2() + 4; }
  __host__ __device__ int64_t total() const { return bo2() + 2; }
};

// Where a step takes its rows from. rows == nullptr: rows row0 .. row0+nb-1 (validation / predict).
// Otherwise rows[(epoch - epoch0) * epoch_stride + offset + b] with epoch read from DevState on the
// device, so the same launch sequence (or CUDA graph) serves every epoch.
struct RowSrc {
  const int32_t* rows;
  int64_t epoch_stride;
  int64_t offset;
  int32_t row0;
  int32_t nb;
};

__device__ __forceinline__ int64_t row_of(const RowSrc& r, const DevState* st, int b) {
  if (r.rows == nullptr) return (int64_t)r.row0 + b;
  const int64_t e = r.epoch_stride ? (int64_t)(st->epoch - st->epoch0) : 0;
  return (int64_t)r.rows[e * r.epoch_stride + r.offset + b];
}

// HBM layout of W1 / m / v when the tcgen05 first layer is in use (width 256): blocks of 8 SNPs
// (8 KB), inside a block [8 chunks of 32 columns][8 SNP rows][128 B] with 32-byte atoms XOR (row & 3)
// -- the canonical MN-major tf32 UMMA operand image, so both first-layer kernels move it with plain
// contiguous bulk copies.  Rows are padded to a multiple of 64 with zeros.
__host__ __device__ inline int64_t w1_tiled_index(int64_t k, int j) {
  return ((k >> 3) << 11) + ((int64_t)(j >> 5) << 8) + ((k & 7) << 5) + ((((j & 31) >> 3) ^ (int)(k & 3)) << 3) + (j & 7);
}

struct L1Args {
  int64_t K;
  int H;
  int training;
  int gated;  // no-op once DevState::stopped is set (launches queued past the early-stopping epoch)
  const uint32_t* packed;
  int64_t row_words;
  RowSrc src;
  RowSrc src_next;  // rows of the following step (fused forward of the tcgen05 backward kernel)
  int fuse_next;
  int rev;  // tcgen05 backward: walk the CTA's tiles downwards -- odd steps (host-side step parity), so that a walk starts
            // on the tail of the previous step's updates, still in L2: those reads hit and their dirty lines are
            // overwritten in place
  unsigned wait_hid;  // != 0: launched ahead of this step's hidden stack -- wait for DevState::hid_seq >= wait_hid before dZ1 is read
  unsigned wait_bwd;  // with wait_hid: the previous backward of this model may still be running on other SMs when this
                      // CTA starts -- no chunk is loaded before DevState::bwd_cnt >= wait_bwd (all its CTAs are done)
  unsigned long long* tl;  // kernel timeline buffer (diagnostics) or nullptr
  int tl_id;
  float *gamma, *beta, *mmean, *mvar;
  float* W1;
  float *m_gamma, *v_gamma, *m_beta, *v_beta, *mW1, *vW1;
  float* partials;   // [n_partials][kMaxB][H]
  const float* dZ1;  // [kMaxB][H]
  DevState* st;
};

struct HidArgs {
  int H, L, n_before;
  int training;
  int gated;
  int has_targets;  // inference: accumulate the validation loss against locs
  int write_pred;  // inference: also store y2 rows to pred_out
  float p_drop;
  uint64_t seed;
  const uint8_t* masks;  // test hook [nsteps][kMaxB][H] or nullptr
  int64_t n_masks;
  const float* partials;
  int n_partials;
  int64_t partial_stride;  // floats between consecutive partial tiles (kMaxB * H; wide inference: 32 * chunks * H)
  int partial_row0;        // first row of this launch inside a partial tile (wide inference: 32 * chunk)
  float* val_slot;         // inference with targets: {sum of distances, rows} go here instead of DevState
                           // (chunks of one wide pass run concurrently; k_val_accumulate adds them in order)
  // sharded models (tp.cu): the partial tiles are the shards' tiles, complete once every flag >= wait_seq
  const uint32_t* wait_flags;
  int wait_count;
  uint32_t wait_seq;
  int* wait_err;
  float* small;
  const float* w_fs;  // forward slices of the hidden kernels  [L-1][C][H][Hc]
  const float* w_bs;  // backward slices (transposed)          [L-1][C][H][Hc]
  int n_slots;        // shared-memory weight-slice ring size
  float* acts;  // [L][kMaxB][H] post-dropout outputs of Dense(width) layer i
  float* dzs;   // [L][kMaxB][H] d loss / d z_i
  float* outs;  // y1[32][2], dy1[32][2], dy2[32][2], y2[32][2]
  const float* locs;  // [n][2] targets of the bound matrix
  RowSrc src;
  float* pred_out;  // [n][2]
  long long* dbg;   // optional per-CTA clock64() checkpoints [C][256] (profiling builds of the step)
  unsigned wait_bwd;  // != 0: launched ahead of the backward that produces its Z1 tiles -- wait for DevState::bwd_cnt >= wait_bwd
  unsigned hid_seq;   // training launches: value to publish in DevState::hid_seq when everything is written
  unsigned wait_upd;  // != 0: wait for DevState::upd_cnt >= wait_upd before the small weights are read (the update ran
                      // under the previous hidden stack, not directly in front of this launch)
  unsigned long long* tl;  // kernel timeline buffer (diagnostics) or nullptr
  int tl_id;
  // Batches of more than 32 rows (bigbatch.cu): the step's rows go through the stack in 32-row chunks, one launch each.
  int loss_rows;    // rows of the whole step (the loss is their mean): 0 = src.nb
  int row_base;     // first row of this chunk inside the step (dropout stream / mask row)
  int mask_rows;    // rows per step of the injected dropout masks: 0 = kMaxB
  int chunk_flags;  // bit 0: not the step's first chunk (last_loss accumulates); bit 1: not its last (no optimizer bookkeeping)
  DevState* st;
};

constexpr int kMaxGroup = 8;  // replicates per grouped hidden-stack launch
struct HidGroupArgs {
  int n;
  HidArgs a[kMaxGroup];
};

struct UpdArgs {
  int H, L;
  int gated;
  float *small, *m_small, *v_small;
  float *w_fs, *w_bs;  // pre-sliced copies kept in sync with small
  int Hc;
  int slice_mode;  // 0: hidden.cu slices, 1: hidden_tc.cu operand images
  const float* acts;
  const float* dzs;
  const float* outs;
  int nb;
  unsigned wait_hid;  // != 0: wait for DevState::hid_seq >= wait_hid (launched ahead of the hidden stack it consumes)
  unsigned wait_upd;  // with wait_dz: the model's previous update must be complete before this one reads the weights (formally;
                      // a whole first-layer backward lies between them)
  unsigned wait_dz;   // != 0: launched UNDER that hidden stack -- the blocks of layer i only wait for DevState::dz_cnt[i] >= wait_dz
  unsigned long long* tl;  // kernel timeline buffer (diagnostics) or nullptr
  int tl_id;
  DevState* st;
};

// launchers (each returns 0 or sets the error)
int l1_forward_simt(const L1Args& a, int n_partials, cudaStream_t s);
int l1_backward_simt(const L1Args& a, int nblocks, cudaStream_t s);
int hidden_launch(const HidArgs& a, int cluster, cudaStream_t s);
// g.n models (same width, nlayers and cluster size) in one launch, one cluster each: replicate groups
int hidden_group_launch(const HidGroupArgs& g, int cluster, cudaStream_t s);
int hidden_update_launch(const UpdArgs& a, cudaStream_t s, bool overlap_previous = false);
int hidden_update_blocks(int H, int L);  // blocks of one hidden_update_launch (each bumps DevState::upd_cnt once)
int hidden_max_cluster(int H, int L);  // largest usable cluster size (16, 8, ...) for this device
int hidden_slots(int H, int L, int cluster);
int hidden_max_nlayers(int H);  // deepest L in [2, 64] with a slot at some cluster size (host arithmetic), 0 = none
int hidden_reslice(const float* small, float* fs, float* bs, int H, int L, int cluster, cudaStream_t s);
size_t hidden_smem_bytes(int H, int L, int cluster);

// tcgen05 hidden stack (hidden_tc.cu): width 256, one cluster of kHidTcCtas CTAs per model (and SMs: one CTA per SM)
constexpr int kHidTcCtas = 16;
bool hidden_tc_supported(int H, int L);
int hidden_tc_launch(const HidArgs& a, cudaStream_t s, bool overlap_previous = false);
int hidden_tc_group_launch(const HidGroupArgs& g, cudaStream_t s);
int hidden_tc_reslice(const float* small, float* fs, float* bs, int L, cudaStream_t s);

// tcgen05 first layer (l1_tc.cu); available() is false when the shape is unsupported.
bool l1_tc_supported(int64_t K, int H);
int l1_forward_tc(const L1Args& a, int n_partials, cudaStream_t s);
int l1_backward_tc(const L1Args& a, int nblocks, cudaStream_t s, bool overlap_previous = false);
int l1_tc_partials(int64_t K);
// inference forward of up to 256 rows in one pass over W1: out [n_partials][32 * ceil(nrows / 32)][256]
int l1_forward_wide_tc(const L1Args& a, int n_partials, int nrows, float* out, cudaStream_t s);

}  // namespace loc

struct loc_tp;
namespace loc {
// Sum over the split-K partial tiles of element i = blockIdx.x * 128 + (threadIdx.x & 127), for 512-thread
// blocks: four thread groups take a quarter of the tiles each (16 loads in flight per thread), fixed order.
// Valid in threads < 128 after the call.
__device__ __forceinline__ float reduce_partial_tiles(const float* __restrict__ partials, int n_partials, int n,
                                                      float (*sred)[128]) {
  const int e = threadIdx.x & 127, g = threadIdx.x >> 7;
  const int i = blockIdx.x * 128 + e;
  const int pbeg = n_partials * g / 4, pend = n_partials * (g + 1) / 4;
  float s0 = 0.f, s1 = 0.f;
  if (i < n) {
    int p = pbeg;
#pragma unroll 8
    for (; p + 2 <= pend; p += 2) {
      s0 += __ldcg(partials + (int64_t)p * n + i);
      s1 += __ldcg(partials + (int64_t)(p + 1) * n + i);
    }
    if (p < pend) s0 += __ldcg(partials + (int64_t)p * n + i);
  }
  sred[g][e] = s0 + s1;
  __syncthreads();
  return (sred[0][e] + sred[1][e]) + (sred[2][e] + sred[3][e]);
}

// Batches of 33..256 rows (bigbatch.cu): batch statistics of the whole step, first-layer backward + Adam over all of
// its rows (fp32 CUDA cores, either W1 layout), small-layer update over the step's 32-row chunks.
struct BigArgs {
  int64_t K;
  int H, L;
  int gated;
  int tiled;  // W1 / m / v in the tcgen05 layout (w1_tiled_index) instead of row-major
  int nb;     // rows of the step
  const uint32_t* packed;
  int64_t row_words;
  RowSrc src;
  float *gamma, *beta, *mmean, *mvar;
  float *bmean, *bvar;  // [K] batch statistics of the step in flight
  float* W1;
  float *m_gamma, *v_gamma, *m_beta, *v_beta, *mW1, *vW1;
  const float* dzs;     // [chunks][L][kMaxB][H]: dZ1 of row b = dzs[(b / 32) * L * 32 * H + (b % 32) * H + j]
  const float* acts;    // [chunks][L][kMaxB][H]
  const float* outs;    // [chunks][256]
  float *small, *m_small, *v_small, *w_fs, *w_bs;
  int Hc, slice_mode;
  DevState* st;
};
// The same step of up to kMaxGroup models (replicate groups: row count per step and K may differ)
struct BigGroupArgs {
  int n;
  BigArgs a[kMaxGroup];
};
// Step end of the models of a group whose chunks ran side by side: model g's nc[g] per-chunk loss sums are slots[g],
// its step's rows loss_rows[g]
struct BigEndArgs {
  int n;
  DevState* st[kMaxGroup];
  const float* slots[kMaxGroup];
  int nc[kMaxGroup];
  int loss_rows[kMaxGroup];
};
int bb_stats_launch(const BigGroupArgs& g, cudaStream_t s);
int bb_l1_backward_launch(const BigArgs& a, float* pq_part, cudaStream_t s);
int64_t bb_pq_floats(int64_t K, int H);  // scratch of the backward: per column group partial sums for gamma / beta
int bb_hidden_update_launch(const BigArgs& a, cudaStream_t s);
int bb_step_end_launch(const BigEndArgs& e, int gated, cudaStream_t s);
constexpr int kMaxChunks = LOC_MAX_BATCH_SIZE / LOC_MAX_BATCH;

int tp_exchange(loc_tp* tp, const float* partials, int n_partials, cudaStream_t s);
const float* tp_tiles(const loc_tp* tp);
void tp_wait_info(const loc_tp* tp, const uint32_t** flags, int* count, uint32_t* seq, int** err);
int tp_world(const loc_tp* tp);
}  // namespace loc

struct loc_model {
  int dev;
  int64_t K;
  int H, L, B, n_before, max_epochs;
  float p_drop;
  uint64_t seed;
  int cluster;
  int n_partials;   // partial Z1 tiles the forward leaves
  int n_bwd_blocks;
  int cap_partials; // partial tiles the buffers hold (the largest CTA count loc_model_set_l1_ctas accepts)
  int chain_open;   // the stream's last kernels are this model's chained step (train_step): the next hidden stack may overlap them
  cudaStream_t chain_stream;
  int use_tc;       // first layer on tcgen05 (implies the tiled W1 layout)
  int64_t Kpad;     // rows of W1 / m / v in use (K rounded up to 64 when tiled)
  int64_t cap_K;    // K the buffers were allocated for (a pooled handle serves any K <= cap_K, see loc_model_create)
  int cap_epochs;   // rows of the history buffer
  int hid_tc;       // hidden stack on tcgen05 (hidden_tc.cu) instead of CUDA cores (hidden.cu)
  loc::SmallLayout sl;
  // parameters
  float *gamma, *beta, *mmean, *mvar, *W1, *small;
  float *w_fs, *w_bs;  // pre-sliced copies of the hidden kernels for k_hidden
  int n_slots;
  // Adam moments
  float *m_gamma, *v_gamma, *m_beta, *v_beta, *mW1, *vW1, *m_small, *v_small;
  // ModelCheckpoint snapshot (weights only)
  float *best_gamma, *best_beta, *best_mmean, *best_mvar, *best_W1, *best_small;
  // workspaces
  float *partials, *acts, *dzs, *outs, *hist, *pred_tmp;
  float* wide;       // wide inference: split-K partial tiles of up to 256 rows [n_partials][256][H] (tcgen05 path)
  float* val_slots;  // [8][2] per-chunk validation sums of a wide pass
  float *bb_mean, *bb_var;  // [K] batch statistics of a step of more than 32 rows (bigbatch.cu); null for B <= 32
  float* bb_pq;             // [column groups][2][K] partial sums of that step's gamma / beta gradients
  int cap_chunks;           // 32-row chunks the acts / dzs buffers hold
  long long* dbg;
  int tl_id;         // model number in the kernel timeline (diagnostics)
  cudaStream_t side;        // small-layer update runs here, beside the first-layer backward
  cudaEvent_t ev_hid, ev_upd;
  loc::DevState* st;
  // bound data
  const uint32_t *train_packed, *val_packed;
  int64_t n_train, train_row_words, n_val, val_row_words;
  const float *train_locs, *val_locs;
  const uint8_t* masks;
  int64_t n_masks;
  // SNP shard of a larger model (tensor parallelism): columns [k_offset, k_offset + K) of K_global
  int64_t k_offset, K_global;
  int (*exchange)(void* ctx, float* d_tile, int64_t n, void* stream);
  void* exchange_ctx;
  float* z1_tile;  // caller-owned [kMaxB][H]: own partial sum, then the sum over shards
  struct loc_tp* tp;  // peer-memory exchange (tp.cu) instead of the host hook
  // loc_train_steps: the last span left the forward tiles of step span_next of the epoch ordered by span_perm
  const int32_t* span_perm;
  int64_t span_next;
  // host mirrors of DevState::hid_seq / bwd_cnt / optimizer step parity (what the launches made so far will have
  // published once they have run)
  unsigned h_hid_seq, h_bwd_cnt, h_upd_cnt;
  int64_t h_steps;
};
