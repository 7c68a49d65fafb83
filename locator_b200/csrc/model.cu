// loc_model: parameters, Adam state, checkpoint snapshot and the epoch driver.
//
// Reference: load_network locator/locator.py:311-327, load_callbacks :330-362, train_network
// :365-394 (fit + reload of the best checkpoint), predict :414,441.  The callback state machine
// (ModelCheckpoint -> EarlyStopping -> ReduceLROnPlateau, Keras semantics restated in
// oracle/model_ref.py:CallbackState) runs on the device so a whole run of epochs is enqueued
// without a host round trip; launches queued past the stopping epoch are no-ops.
#include <math.h>
#include <stdlib.h>

#include <mutex>
#include <new>
#include <vector>

#include "model.cuh"
#include "philox.cuh"

using namespace loc;

namespace loc {

__global__ void k_fill(float* p, int64_t n, float v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}

// Keras glorot_uniform with the Philox layout shared with oracle/philox_ref.py.
__global__ void k_glorot(float* w, int64_t n, float limit, uint32_t stream, uint64_t seed) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float u = philox_uniform((uint64_t)i, stream, seed);
    w[i] = (2.0f * u - 1.0f) * limit;
  }
}

// W1 in the tiled layout (model.cuh: w1_tiled_index): same Philox element index as the row-major init.
__global__ void k_glorot_tiled(float* w, int64_t K, int H, float limit, uint32_t stream, uint64_t seed,
                               int64_t k_offset) {
  const int64_t n = K * H;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float u = philox_uniform((uint64_t)(i + k_offset * H), stream, seed);  // element index of the whole layer
    w[w1_tiled_index(i / H, (int)(i % H))] = (2.0f * u - 1.0f) * limit;
  }
}

// Keras row-major [K][256] <-> tiled (to_tiled: dst tiled; else dst row-major)
__global__ void k_w1_permute(float* dst, const float* src, int64_t K, int H, int to_tiled) {
  const int64_t n = K * H;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = w1_tiled_index(i / H, (int)(i % H));
    if (to_tiled)
      dst[t] = src[i];
    else
      dst[i] = src[t];
  }
}

__global__ void k_state_reset(DevState* st, float lr, int patience, int max_epochs, int reset_opt) {
  if (reset_opt) {
    st->t = 0;
    st->step_id = 0;
    st->alpha = 0.f;
  }
  st->lr = lr;
  st->loss_total = st->loss_count = st->val_total = st->val_count = 0.f;
  st->epoch = 0;
  st->epoch0 = 0;
  st->stopped = 0;
  st->improved = 0;
  st->best_epoch = -1;
  st->ckpt_best = st->es_best = st->rlr_best = INFINITY;
  st->es_wait = st->rlr_wait = 0;
  st->patience = patience;
  st->rlr_patience = patience / 6;
  st->max_epochs = max_epochs;
  st->nonfinite = 0;
  st->last_loss = st->last_val = 0.f;
  st->chain_timeout = 0;
  st->hid_seq = 0u;  // hand-over flags of the chained step (host mirrors: loc_model::h_hid_seq / h_bwd_cnt / h_upd_cnt)
  st->bwd_cnt = 0u;
  st->upd_cnt = 0u;
  for (int i = 0; i < 64; ++i) st->dz_cnt[i] = 0u;
}

__global__ void k_begin_call(DevState* st) { st->epoch0 = st->epoch; }
// validation sums of the 32-row chunks of one wide inference pass, added in chunk order (same bits as the
// chunk-by-chunk launches of the narrow path)
__global__ void k_val_accumulate(DevState* st, const float* slots, int n, int gated) {
  if (gated && st->stopped) return;
  for (int c = 0; c < n; ++c) {
    st->val_total += slots[2 * c];
    st->val_count += slots[2 * c + 1];
  }
}
__global__ void k_zero_val(DevState* st) { st->val_total = st->val_count = 0.f; }

// on_epoch_end of History + [ModelCheckpoint, EarlyStopping, ReduceLROnPlateau] (locator.py:330-362).
__global__ void k_epoch_end(DevState* st, float* hist) {
  if (st->stopped) {
    st->improved = 0;
    return;
  }
  const int epoch = st->epoch;
  const float loss = st->loss_total / st->loss_count;
  const float val = st->val_total / st->val_count;
  st->last_loss = loss;
  st->last_val = val;
  if (!isfinite(loss) || !isfinite(val)) st->nonfinite = 1;
  // ModelCheckpoint(save_best_only, monitor=val_loss): strict improvement
  const int save = val < st->ckpt_best;
  if (save) {
    st->ckpt_best = val;
    st->best_epoch = epoch;
  }
  st->improved = save;
  // EarlyStopping(min_delta=0, patience)
  st->es_wait += 1;
  int stop = 0;
  if (val < st->es_best) {
    st->es_best = val;
    st->es_wait = 0;
  } else if (st->es_wait >= st->patience && epoch > 0) {
    stop = 1;
  }
  // ReduceLROnPlateau(factor .5, patience/6, min_delta 0, cooldown 0, min_lr 0): logs the lr first
  const float lr_logged = st->lr;
  if (val < st->rlr_best) {
    st->rlr_best = val;
    st->rlr_wait = 0;
  } else {
    st->rlr_wait += 1;
    if (st->rlr_wait >= st->rlr_patience) {
      if (st->lr > 0.f) st->lr = fmaxf(st->lr * 0.5f, 0.f);
      st->rlr_wait = 0;
    }
  }
  hist[3 * epoch + 0] = loss;
  hist[3 * epoch + 1] = val;
  hist[3 * epoch + 2] = lr_logged;
  st->loss_total = st->loss_count = st->val_total = st->val_count = 0.f;
  st->epoch = epoch + 1;
  if (stop || epoch + 1 >= st->max_epochs) st->stopped = 1;
}

struct CopySegs {
  float* dst[6];
  const float* src[6];
  int64_t n[6];
  int count;
};

// ModelCheckpoint / load_weights as a device-to-device copy; `cond` (may be null) gates it.
__global__ void __launch_bounds__(256) k_copy_segs(CopySegs cs, const int* cond) {
  if (cond != nullptr && *cond == 0) return;
  for (int s = 0; s < cs.count; ++s) {
    const int64_t n4 = cs.n[s] / 4;
    const float4* src = reinterpret_cast<const float4*>(cs.src[s]);
    float4* dst = reinterpret_cast<float4*>(cs.dst[s]);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x)
      dst[i] = src[i];
    for (int64_t i = n4 * 4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cs.n[s];
         i += (int64_t)gridDim.x * blockDim.x)
      cs.dst[s][i] = cs.src[s][i];
  }
}

static int fill(float* p, int64_t n, float v, cudaStream_t s) {
  if (n <= 0) return 0;
  int64_t blocks = cdiv(n, 256 * 8);
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  k_fill<<<(unsigned)blocks, 256, 0, s>>>(p, n, v);
  LOC_LAUNCHED();
  return 0;
}

static int copy_weights(loc_model* m, bool to_best, const int* cond, cudaStream_t s) {
  CopySegs cs;
  float* live[6] = {m->W1, m->gamma, m->beta, m->mmean, m->mvar, m->small};
  float* best[6] = {m->best_W1, m->best_gamma, m->best_beta, m->best_mmean, m->best_mvar, m->best_small};
  const int64_t n[6] = {m->Kpad * m->H, m->K, m->K, m->K, m->K, m->sl.total()};
  for (int i = 0; i < 6; ++i) {
    cs.dst[i] = to_best ? best[i] : live[i];
    cs.src[i] = to_best ? live[i] : best[i];
    cs.n[i] = n[i];
  }
  cs.count = 6;
  k_copy_segs<<<sm_count() * 4, 256, 0, s>>>(cs, cond);
  LOC_LAUNCHED();
  return 0;
}

static int reslice(loc_model* m, cudaStream_t s) {
  return m->hid_tc ? hidden_tc_reslice(m->small, m->w_fs, m->w_bs, m->L, s)
                   : hidden_reslice(m->small, m->w_fs, m->w_bs, m->H, m->L, m->cluster, s);
}

// LOC_TIMELINE=1: every step kernel logs (globaltimer, tag, model) at its first / last block's start and end
static unsigned long long* g_tl = nullptr;
static int g_tl_models = 0;
static unsigned long long* timeline_buffer() {
  static bool tried = false;
  if (!tried) {
    tried = true;
    if (getenv("LOC_TIMELINE") != nullptr) {
      const size_t bytes = (1 + 2 * (size_t)kTlCap) * sizeof(unsigned long long);
      if (cudaMalloc(&g_tl, bytes) == cudaSuccess)
        cudaMemset(g_tl, 0, bytes);
      else
        g_tl = nullptr;
    }
  }
  return g_tl;
}

static L1Args l1_args(loc_model* m, const uint32_t* packed, int64_t row_words, const RowSrc& src, int training,
                      int gated) {
  L1Args a;
  a.K = m->K;
  a.H = m->H;
  a.training = training;
  a.gated = gated;
  a.packed = packed;
  a.row_words = row_words;
  a.src = src;
  a.src_next = src;
  a.fuse_next = 0;
  a.rev = (int)(m->h_steps & 1);  // steps launched so far (training hidden stacks): odd steps walk downwards
  a.wait_hid = 0u;
  a.wait_bwd = 0u;
  a.tl = timeline_buffer();
  a.tl_id = m->tl_id;
  a.gamma = m->gamma;
  a.beta = m->beta;
  a.mmean = m->mmean;
  a.mvar = m->mvar;
  a.W1 = m->W1;
  a.m_gamma = m->m_gamma;
  a.v_gamma = m->v_gamma;
  a.m_beta = m->m_beta;
  a.v_beta = m->v_beta;
  a.mW1 = m->mW1;
  a.vW1 = m->vW1;
  a.partials = m->partials;
  a.dZ1 = m->dzs;  // layer 0 slot
  a.st = m->st;
  return a;
}

// Sharded models: own split-K partial tiles -> one tile (fixed order), then the sum over shards.
__global__ void __launch_bounds__(512) k_reduce_partials(const float* __restrict__ partials, int n_partials, float* out,
                                                         int n) {
  __shared__ float sred[4][128];
  const float v = reduce_partial_tiles(partials, n_partials, n, sred);
  const int i = blockIdx.x * 128 + threadIdx.x;
  if (threadIdx.x < 128 && i < n) out[i] = v;
}

static int exchange_partials(loc_model* m, cudaStream_t s) {
  if (m->tp != nullptr) return tp_exchange(m->tp, m->partials, m->n_partials, s);
  if (m->exchange == nullptr) return 0;
  const int n = kMaxB * m->H;
  k_reduce_partials<<<cdiv(n, 128), 512, 0, s>>>(m->partials, m->n_partials, m->z1_tile, n);
  LOC_LAUNCHED();
  LOC_CHECK(m->exchange(m->exchange_ctx, m->z1_tile, n, (void*)s) == 0, "exchange hook failed");
  return 0;
}

static HidArgs hid_args(loc_model* m, const RowSrc& src, int training, int gated, const float* locs, float* pred_out) {
  HidArgs h;
  h.H = m->H;
  h.L = m->L;
  h.n_before = m->n_before;
  h.training = training;
  h.gated = gated;
  h.has_targets = (!training && locs != nullptr) ? 1 : 0;
  h.write_pred = pred_out != nullptr ? 1 : 0;
  h.p_drop = m->p_drop;
  h.seed = m->seed;
  h.masks = m->masks;
  h.n_masks = m->n_masks;
  h.wait_flags = nullptr;
  h.wait_count = 0;
  h.wait_seq = 0;
  h.wait_err = nullptr;
  h.wait_bwd = 0u;
  h.wait_upd = 0u;
  h.hid_seq = 0u;
  h.partials = m->exchange != nullptr ? m->z1_tile : m->partials;
  h.n_partials = m->exchange != nullptr ? 1 : m->n_partials;
  h.partial_stride = (int64_t)kMaxB * m->H;
  h.partial_row0 = 0;
  h.val_slot = nullptr;
  h.loss_rows = 0;
  h.row_base = 0;
  h.mask_rows = 0;
  h.chunk_flags = 0;
  if (m->tp != nullptr) {  // the shards' tiles of the latest exchange, summed in rank order by the kernel
    h.partials = tp_tiles(m->tp);
    h.n_partials = tp_world(m->tp);
    tp_wait_info(m->tp, &h.wait_flags, &h.wait_count, &h.wait_seq, &h.wait_err);
  }
  h.small = m->small;
  h.w_fs = m->w_fs;
  h.w_bs = m->w_bs;
  h.n_slots = m->n_slots;
  h.acts = m->acts;
  h.dzs = m->dzs;
  h.outs = m->outs;
  h.locs = locs;
  h.src = src;
  h.pred_out = pred_out;
  h.dbg = m->dbg;
  h.tl = timeline_buffer();
  h.tl_id = m->tl_id;
  h.st = m->st;
  return h;
}

static int forward_l1(loc_model* m, const L1Args& a, cudaStream_t s) {
  m->chain_open = 0;
  m->span_perm = nullptr;  // a standalone forward overwrites the tiles a loc_train_steps span may have left
  return m->use_tc ? l1_forward_tc(a, m->n_partials, s) : l1_forward_simt(a, m->n_partials, s);
}

static UpdArgs upd_args(loc_model* m, int nb, int gated) {
  UpdArgs u;
  u.H = m->H;
  u.L = m->L;
  u.gated = gated;
  u.small = m->small;
  u.m_small = m->m_small;
  u.v_small = m->v_small;
  u.w_fs = m->w_fs;
  u.w_bs = m->w_bs;
  u.Hc = m->H / m->cluster;
  u.slice_mode = m->hid_tc;
  u.acts = m->acts;
  u.dzs = m->dzs;
  u.outs = m->outs;
  u.nb = nb;
  u.wait_hid = 0u;
  u.wait_dz = 0u;
  u.wait_upd = 0u;
  u.tl = timeline_buffer();
  u.tl_id = m->tl_id;
  u.st = m->st;
  return u;
}

// Rows [off, off + nb) of a batch order.  epoch_stride != 0: the order holds one such row per epoch and the
// device-side epoch counter picks it (row_of).
static RowSrc order_rows(const int32_t* order, int64_t epoch_stride, int64_t off, int64_t nb) {
  return RowSrc{order, epoch_stride, off, 0, (int32_t)nb};
}

// Rows row0 .. row0 + nb - 1 of the bound matrix (validation / predict).
static RowSrc consecutive_rows(int64_t row0, int64_t nb) { return RowSrc{nullptr, 0, 0, (int32_t)row0, (int32_t)nb}; }

// The training step that starts at row `off` of a batch order: batch_size rows, fewer at the end of the epoch.
static RowSrc step_rows(const loc_model* m, const int32_t* order, int64_t epoch_stride, int64_t off) {
  return order_rows(order, epoch_stride, off, m->n_train - off < m->B ? m->n_train - off : m->B);
}

// 32-row chunk c of a step or of a wide inference pass.
static RowSrc chunk_rows(RowSrc src, int c) {
  if (src.rows != nullptr)
    src.offset += (int64_t)kMaxB * c;
  else
    src.row0 += kMaxB * c;
  src.nb = src.nb - kMaxB * c < kMaxB ? src.nb - kMaxB * c : kMaxB;
  return src;
}

// Chunk c of the nc chunks of a wide pass: its Z1 rows start at row 32 c of the pass's split-K tiles in m->wide, and
// its outputs go to the chunk's block of m->outs.
static void wide_chunk(const loc_model* m, HidArgs& h, int nc, int c) {
  h.partials = m->wide;
  h.n_partials = m->n_partials;
  h.partial_stride = (int64_t)nc * kMaxB * m->H;
  h.partial_row0 = kMaxB * c;
  h.outs = m->outs + c * 256;
}

// A training launch of the hidden stack advances the step parity (tile walk direction of the backward) and the
// hand-over flag it publishes when it is done; call right before the launch.
static void begin_training_hidden(loc_model* m, HidArgs& h) {
  ++m->h_steps;
  h.hid_seq = ++m->h_hid_seq;
}

// One model's hidden stack on its family's kernel.  overlap_previous (tcgen05 only): programmatic dependent launch.
static int hidden_stack(const loc_model* m, const HidArgs& h, cudaStream_t s, bool overlap_previous = false) {
  return m->hid_tc ? hidden_tc_launch(h, s, overlap_previous) : hidden_launch(h, m->cluster, s);
}
// The hidden stacks of a replicate group in one launch, one cluster each, on the family of m (every model's).
static int hidden_stacks(const loc_model* m, const HidGroupArgs& g, cudaStream_t s) {
  return m->hid_tc ? hidden_tc_group_launch(g, s) : hidden_group_launch(g, m->cluster, s);
}

// First-layer backward + Adam; on the tcgen05 path also the host mirror of the counter its CTAs bump when they are
// done (l1_backward_tc launches exactly n_bwd_blocks of them).
static int backward_l1(loc_model* m, L1Args& a, cudaStream_t s, bool overlap_previous = false) {
  if (!m->use_tc) return l1_backward_simt(a, m->n_bwd_blocks, s);
  a.rev = (int)(m->h_steps & 1);
  if (l1_backward_tc(a, m->n_bwd_blocks, s, overlap_previous)) return 1;
  m->h_bwd_cnt += (unsigned)m->n_bwd_blocks;
  return 0;
}

// Small-layer update + the host mirror of the counter its blocks bump when they are done.
static int update_launch(loc_model* m, const UpdArgs& u, cudaStream_t s, bool overlap_previous = false) {
  if (hidden_update_launch(u, s, overlap_previous)) return 1;
  m->h_upd_cnt += (unsigned)hidden_update_blocks(m->H, m->L);
  return 0;
}

// The small-layer updates of models ms[0..n) beside their first-layer backwards: each on its model's side stream,
// behind the event ms[0]->ev_hid records now on `s` (after the hidden-stack launch that holds the n models).
// update(i, stream) launches model i's update; join_updates makes `s` wait for all of them.
template <class Update>
static int fork_updates(loc_model* const* ms, int n, cudaStream_t s, Update update) {
  LOC_CUDA(cudaEventRecord(ms[0]->ev_hid, s));
  for (int i = 0; i < n; ++i) {
    LOC_CUDA(cudaStreamWaitEvent(ms[i]->side, ms[0]->ev_hid, 0));
    if (update(i, ms[i]->side)) return 1;
    LOC_CUDA(cudaEventRecord(ms[i]->ev_upd, ms[i]->side));
  }
  return 0;
}
static int join_updates(loc_model* const* ms, int n, cudaStream_t s) {
  for (int i = 0; i < n; ++i) LOC_CUDA(cudaStreamWaitEvent(s, ms[i]->ev_upd, 0));
  return 0;
}

// Can one model's step run as a chain of programmatic dependent launches (see train_step)?  Needs the tcgen05
// kernels and no sharding (the exchange of a sharded model sits between the kernels).
static bool chain_capable(const loc_model* m) {
  const bool off = getenv("LOC_NO_CHAIN") != nullptr;  // read per call: tests compare both schedules in one process
  return !off && m->use_tc && m->hid_tc && m->exchange == nullptr && m->tp == nullptr;
}

static BigArgs big_args(loc_model* m, const RowSrc& src, int gated) {
  BigArgs g;
  g.K = m->K;
  g.H = m->H;
  g.L = m->L;
  g.gated = gated;
  g.tiled = m->use_tc;
  g.nb = src.nb;
  g.packed = m->train_packed;
  g.row_words = m->train_row_words;
  g.src = src;
  g.gamma = m->gamma;
  g.beta = m->beta;
  g.mmean = m->mmean;
  g.mvar = m->mvar;
  g.bmean = m->bb_mean;
  g.bvar = m->bb_var;
  g.W1 = m->W1;
  g.m_gamma = m->m_gamma;
  g.v_gamma = m->v_gamma;
  g.m_beta = m->m_beta;
  g.v_beta = m->v_beta;
  g.mW1 = m->mW1;
  g.vW1 = m->vW1;
  g.dzs = m->dzs;
  g.acts = m->acts;
  g.outs = m->outs;
  g.small = m->small;
  g.m_small = m->m_small;
  g.v_small = m->v_small;
  g.w_fs = m->w_fs;
  g.w_bs = m->w_bs;
  g.Hc = m->H / m->cluster;
  g.slice_mode = m->hid_tc;
  g.st = m->st;
  return g;
}

// One optimizer step of n models created with batch_size > 32 (bigbatch.cu), each over its own number of rows (a
// single model, or the models of a replicate group of loc_group_train_epochs that have a step at this offset):
//   batch statistics over all rows of every model's step (one launch for the group),
//   first-layer forward with those statistics (one wide pass over W1 per model on the tcgen05 path),
//   the step's 32-row chunks through the hidden stack -- tcgen05: side by side, one cluster per chunk, whole models
//     packed into grouped launches by their own chunk counts (up to 8 chunks a launch), then the step end of those
//     models in one launch; a model whose step fits in one chunk gets its own launch, as alone; CUDA cores: chunk by
//     chunk, each after its first-layer forward, in a group chunk c of every model that has one in one launch,
//   one pass over W1 | m | v per model (dW1 over all rows + Adam), back to back,
//   the small-layer update over the chunks: after the backward for a single model; in a group on the model's side
//     stream, forked after the hidden launch that holds its chunks (it runs under the other models' backwards) and
//     joined before the next step.
// Every model's launches are the ones it gets alone, with the same arguments, so the group gives the same bits.
static int train_step_big(loc_model* const* ms, const RowSrc* srcs, int n, int gated, cudaStream_t s) {
  LOC_CHECK(n >= 1 && n <= kMaxGroup, "training step (large batch): bad group size");
  int ncs[kMaxGroup], nc_max = 0;
  BigGroupArgs bg;
  bg.n = n;
  for (int g = 0; g < n; ++g) {
    loc_model* m = ms[g];
    m->chain_open = 0;
    m->span_perm = nullptr;
    ncs[g] = (srcs[g].nb + kMaxB - 1) / kMaxB;
    if (ncs[g] > nc_max) nc_max = ncs[g];
    LOC_CHECK(srcs[g].nb >= 1 && ncs[g] <= m->cap_chunks && m->bb_mean != nullptr,
              "training step: more rows than the model's batch_size");
    LOC_CHECK(m->exchange == nullptr && m->tp == nullptr, "sharded models train with batch_size <= 32");
    bg.a[g] = big_args(m, srcs[g], gated);
  }
  if (bb_stats_launch(bg, s)) return 1;
  const bool no_wide = getenv("LOC_NO_WIDE") != nullptr;
  const bool wide = ms[0]->wide != nullptr && ms[0]->use_tc && ms[0]->hid_tc && !no_wide;
  if (wide) {
    for (int g = 0; g < n; ++g) {
      loc_model* m = ms[g];
      L1Args a = l1_args(m, m->train_packed, m->train_row_words, srcs[g], 0, gated);
      a.mmean = m->bb_mean;  // "inference" forward with the step's batch statistics
      a.mvar = m->bb_var;
      if (l1_forward_wide_tc(a, m->n_partials, srcs[g].nb, m->wide, s)) return 1;
    }
  }
  // Chunk c of model g: its first-layer forward into the model's partial tiles (unless the wide pass left them), then
  // the arguments of its hidden stack.
  auto chunk = [&](int g, int c, HidArgs& h) -> int {
    loc_model* m = ms[g];
    const int nc = ncs[g];
    const RowSrc sc = chunk_rows(srcs[g], c);
    if (!wide) {
      L1Args a = l1_args(m, m->train_packed, m->train_row_words, sc, 0, gated);
      a.mmean = m->bb_mean;
      a.mvar = m->bb_var;
      if (forward_l1(m, a, s)) return 1;
    }
    h = hid_args(m, sc, 1, gated, m->train_locs, nullptr);
    if (wide)
      wide_chunk(m, h, nc, c);
    else
      h.outs = m->outs + c * 256;
    const int64_t chunk_stride = (int64_t)m->L * kMaxB * m->H;
    h.acts = m->acts + c * chunk_stride;
    h.dzs = m->dzs + c * chunk_stride;
    h.loss_rows = srcs[g].nb;
    h.row_base = kMaxB * c;
    h.mask_rows = kMaxB * m->cap_chunks;
    h.chunk_flags = (c > 0 ? 1 : 0) | (c < nc - 1 ? 2 : 0);
    begin_training_hidden(m, h);
    return 0;
  };
  const bool serial = getenv("LOC_BB_SERIAL") != nullptr;  // tests: one hidden launch per chunk and model
  const bool fork = n > 1;
  // tcgen05 hidden stack: the chunks of a model of more than one chunk run side by side, one cluster each
  // (k_hidden_tc_group); their loss sums and the step's optimizer bookkeeping follow in k_bb_step_end.  A model's
  // chunks never straddle two launches: each publishes DevState::hid_seq once all of the model's chunks are done.
  auto side_by_side = [&](int g) { return wide && ncs[g] > 1 && !serial; };
  // CUDA-core hidden stack, a group: chunk by chunk, the forwards of every model, then chunk c of every model in one
  // k_hidden launch (one cluster per model).  Loss and step bookkeeping stay inside the launch, as for one model.
  const bool chunk_lockstep = !wide && fork && !ms[0]->hid_tc && !serial;
  if (chunk_lockstep) {
    for (int c = 0; c < nc_max; ++c) {
      HidGroupArgs hg;
      hg.n = 0;
      for (int g = 0; g < n; ++g)
        if (c < ncs[g] && chunk(g, c, hg.a[hg.n++])) return 1;
      if (hidden_stacks(ms[0], hg, s)) return 1;
    }
    if (fork_updates(ms, n, s, [&](int i, cudaStream_t su) { return bb_hidden_update_launch(bg.a[i], su); })) return 1;
  }
  // Models g0 .. g1 - 1 whose chunks are packed into hg: one grouped launch, then their updates forked.
  HidGroupArgs hg;
  hg.n = 0;
  int g0 = 0;
  auto flush = [&](int g1) -> int {
    if (hg.n > 0 && hidden_tc_group_launch(hg, s)) return 1;
    hg.n = 0;
    if (fork && g1 > g0 &&
        fork_updates(ms + g0, g1 - g0, s, [&](int i, cudaStream_t su) { return bb_hidden_update_launch(bg.a[g0 + i], su); }))
      return 1;
    g0 = g1;
    return 0;
  };
  BigEndArgs e;
  e.n = 0;
  for (int g = 0; !chunk_lockstep && g < n; ++g) {
    loc_model* m = ms[g];
    if (!side_by_side(g) || hg.n + ncs[g] > kMaxGroup)
      if (flush(g)) return 1;
    const int first = hg.n;
    for (int c = 0; c < ncs[g]; ++c) {
      HidArgs h;
      if (chunk(g, c, h)) return 1;
      if (side_by_side(g)) {
        h.chunk_flags = 2;  // nobody bumps the step counters inside the launch
        h.val_slot = m->val_slots + 2 * c;
        hg.a[hg.n++] = h;
        continue;
      }
      if (hidden_stack(m, h, s)) return 1;
    }
    for (int i = first; i < hg.n; ++i) hg.a[i].hid_seq = m->h_hid_seq;  // published concurrently: the same (final) value
    if (side_by_side(g)) {
      e.st[e.n] = m->st;
      e.slots[e.n] = m->val_slots;
      e.nc[e.n] = ncs[g];
      e.loss_rows[e.n] = srcs[g].nb;
      ++e.n;
    } else if (flush(g + 1)) {
      return 1;
    }
  }
  if (!chunk_lockstep && flush(n)) return 1;
  if (e.n > 0 && bb_step_end_launch(e, gated, s)) return 1;
  for (int g = 0; g < n; ++g)
    if (bb_l1_backward_launch(bg.a[g], ms[g]->bb_pq, s)) return 1;
  if (!fork) return bb_hidden_update_launch(bg.a[0], s);
  return join_updates(ms, n, s);
}

// One optimizer step: 3-4 launches.
// `next` (tcgen05 path): rows of the following step -- the backward kernel then also runs that step's
// first-layer forward on the W1 chunks it has just updated (they are still in shared memory), so the
// following step is called with have_fwd = true and skips its own forward launch.
//
// Chained steps (chain_capable): the step's kernels go into ONE stream as  H -> U -> B  (hidden stack on its
// 16-SM cluster, small-layer update, first-layer backward + Adam (+ next forward)), every one of them launched
// with programmatic stream serialization, i.e. scheduled as soon as its predecessor's CTAs are all running instead
// of after it has drained, and handing over through two device flags instead of kernel boundaries:
//   B's CTAs take the 132 SMs H does not use while H still runs: barriers, TMEM and the first ring stages of
//     W1 | m | v are ready when H publishes DevState::hid_seq (after its last write), which B waits for before it
//     touches dZ1.  Its last 16 CTAs get H's SMs when H exits; they hold the smaller tile shares (tile_range in
//     l1_tc.cu), so they still finish with the others.  (With fewer first-layer CTAs than SMs --
//     loc_model_set_l1_ctas, replicate rings -- all of B is resident early.)
//   U's blocks take SMs H leaves idle and wait for the same flag (per layer: DevState::dz_cnt, below);
//   the NEXT step's H is queued behind B and waits for DevState::upd_cnt (every finished block of U) and
//     DevState::bwd_cnt (one count per finished CTA of B) before it reads the small weights and the Z1 tiles B's
//     fused forward left -- not for B's completion as a grid (griddepcontrol.wait), which comes microseconds later.
// Kernel boundaries (drain + launch + ramp: 6-15 us each on this part, `scripts/timeline.py`) disappear from the
// step's critical path; what remains is H + B plus the flags' latency.
static int train_step(loc_model* m, const RowSrc& src, int gated, cudaStream_t s, const RowSrc* next = nullptr,
                      bool have_fwd = false) {
  if (m->B > kMaxB) return train_step_big(&m, &src, 1, gated, s);
  L1Args a = l1_args(m, m->train_packed, m->train_row_words, src, 1, gated);
  if (next != nullptr && m->use_tc) {
    a.src_next = *next;
    a.fuse_next = 1;
  }
  const bool chain = chain_capable(m);
  const bool h_overlaps = chain && have_fwd && m->chain_open && m->chain_stream == s;  // the stream's last kernels: this model's B, U
  m->chain_open = 0;
  if (!have_fwd && (forward_l1(m, a, s) || exchange_partials(m, s))) return 1;
  HidArgs h = hid_args(m, src, 1, gated, m->train_locs, nullptr);
  begin_training_hidden(m, h);
  if (h_overlaps) h.wait_bwd = m->h_bwd_cnt;  // every CTA of the previous step's backward has signed off
  if (chain) h.wait_upd = m->h_upd_cnt;       // ... and every block of the small-layer updates so far
  if (hidden_stack(m, h, s, h_overlaps)) return 1;
  if (chain) {
    // U goes in FRONT of B: its blocks land on the SMs that idle under the hidden stack and update layer i as soon
    // as the stack's backward chain has produced dz_i (DevState::dz_cnt), so the update is finished a couple of
    // microseconds after H instead of occupying the SMs between B's end and the next H.  B's CTAs take the SMs the
    // update's blocks leave.
    UpdArgs u = upd_args(m, src.nb, gated);
    u.wait_hid = h.hid_seq;
    u.wait_dz = (unsigned)kHidTcCtas * h.hid_seq;  // every CTA of every training hidden stack so far
    u.wait_upd = m->h_upd_cnt;                     // every block of the updates launched so far
    if (update_launch(m, u, s, true)) return 1;
    a.wait_hid = h.hid_seq;
    a.wait_bwd = m->h_bwd_cnt;  // every backward launched so far for this model
    if (backward_l1(m, a, s, true)) return 1;
    m->chain_open = 1;
    m->chain_stream = s;
    return 0;
  }
  // Unchained: the small-layer update only needs the hidden kernel's outputs: it runs on a side stream next to
  // the first-layer backward.
  const UpdArgs u = upd_args(m, src.nb, gated);
  if (fork_updates(&m, 1, s, [&](int, cudaStream_t su) { return update_launch(m, u, su); })) return 1;
  if (backward_l1(m, a, s)) return 1;
  if (a.fuse_next && exchange_partials(m, s)) return 1;  // the next step's tile is complete
  return join_updates(&m, 1, s);
}

// Inference-mode forward over n rows (Keras predict / evaluate at batch 32: locator.py:374,414,441).
// tcgen05 path: passes of up to 256 rows -- ONE stream of W1 per pass (k_l1_fwd_wide), then the pass's 32-row
// chunks through the hidden stack side by side (one cluster per chunk, k_hidden_tc_group); per-chunk validation
// sums are added in chunk order, so losses carry the same bits as chunk-by-chunk evaluation would give them.
// Otherwise (CUDA-core kernels, sharded models, <= 32 rows): chunks of 32, one W1 stream each.
static int infer_rows(loc_model* m, const uint32_t* packed, int64_t n, int64_t row_words, const float* locs,
                      float* pred_out, int gated, cudaStream_t s) {
  const bool no_wide = getenv("LOC_NO_WIDE") != nullptr;  // tests / A-B runs: chunk-by-chunk evaluation
  const bool wide = m->wide != nullptr && m->use_tc && m->hid_tc && m->exchange == nullptr && m->tp == nullptr &&
                    n > kMaxB && !no_wide;
  m->span_perm = nullptr;
  m->chain_open = 0;
  if (wide) {
    for (int64_t r0 = 0; r0 < n; r0 += 256) {
      const int nrows = (int)((n - r0) < 256 ? (n - r0) : 256);
      const int nc = (nrows + 31) / 32;
      const RowSrc src = consecutive_rows(r0, nrows);
      L1Args a = l1_args(m, packed, row_words, src, 0, gated);
      if (l1_forward_wide_tc(a, m->n_partials, nrows, m->wide, s)) return 1;
      HidGroupArgs hg;
      hg.n = nc;
      for (int c = 0; c < nc; ++c) {
        HidArgs h = hid_args(m, chunk_rows(src, c), 0, gated, locs, pred_out);
        wide_chunk(m, h, nc, c);
        h.val_slot = locs != nullptr ? m->val_slots + 2 * c : nullptr;
        hg.a[c] = h;
      }
      if (hidden_tc_group_launch(hg, s)) return 1;
      if (locs != nullptr) {
        k_val_accumulate<<<1, 1, 0, s>>>(m->st, m->val_slots, nc, gated);
        LOC_LAUNCHED();
      }
    }
    return 0;
  }
  for (int64_t r0 = 0; r0 < n; r0 += kMaxB) {
    const RowSrc src = consecutive_rows(r0, (n - r0) < kMaxB ? (n - r0) : kMaxB);
    L1Args a = l1_args(m, packed, row_words, src, 0, gated);
    if (forward_l1(m, a, s) || exchange_partials(m, s)) return 1;
    if (hidden_stack(m, hid_args(m, src, 0, gated, locs, pred_out), s)) return 1;
  }
  return 0;
}

// Keras row-major host array <-> tiled device array (through a row-major staging buffer).
static int w1_upload(loc_model* m, float* d_tiled, const float* h_src, cudaStream_t s) {
  const int64_t n = m->K * m->H;
  float* tmp = nullptr;
  LOC_CUDA(cudaMalloc(&tmp, n * sizeof(float)));
  LOC_CUDA(cudaMemcpyAsync(tmp, h_src, n * sizeof(float), cudaMemcpyHostToDevice, s));
  k_w1_permute<<<sm_count() * 8, 256, 0, s>>>(d_tiled, tmp, m->K, m->H, 1);
  loc::g_launches.fetch_add(1);
  LOC_CUDA(cudaStreamSynchronize(s));
  LOC_CUDA(cudaFree(tmp));
  return 0;
}
static int w1_download(loc_model* m, const float* d_tiled, float* h_dst, cudaStream_t s) {
  const int64_t n = m->K * m->H;
  float* tmp = nullptr;
  LOC_CUDA(cudaMalloc(&tmp, n * sizeof(float)));
  k_w1_permute<<<sm_count() * 8, 256, 0, s>>>(tmp, d_tiled, m->K, m->H, 0);
  loc::g_launches.fetch_add(1);
  LOC_CUDA(cudaMemcpyAsync(h_dst, tmp, n * sizeof(float), cudaMemcpyDeviceToHost, s));
  LOC_CUDA(cudaStreamSynchronize(s));
  LOC_CUDA(cudaFree(tmp));
  return 0;
}

}  // namespace loc

extern "C" {

const char* loc_l1_impl(void) { return "tcgen05"; }

}  // extern "C"

// ---- handle pool ----------------------------------------------------------------------------------
// Replicate runs (--bootstrap / --windows, locator.py:519-583,609-681) create and drop one model per replicate.
// A model is ~35 device allocations (4 x K x 256 floats among them): cudaMalloc + cudaFree of those cost
// 30-50 ms per replicate on the host -- as much as 250 optimizer steps at K = 100,000.  Destroyed handles
// therefore go to a small pool (LOC_MODEL_POOL handles, default 8, 0 = off) and loc_model_create takes a
// pooled handle whose buffers are large enough (same width / nlayers, K within [0.6, 1] of its capacity)
// instead of allocating; every buffer create() would have zeroed is zeroed again, so a recycled handle is
// indistinguishable from a fresh one.  loc_model_pool_clear() releases the pool's memory.
namespace {
std::mutex g_pool_mu;
std::vector<loc_model*> g_pool;

int pool_limit() {
  static const int lim = [] {
    const char* e = getenv("LOC_MODEL_POOL");
    const int v = e != nullptr ? atoi(e) : 8;
    return v < 0 ? 0 : (v > 64 ? 64 : v);
  }();
  return lim;
}

void free_model(loc_model* m) {
  float* ptrs[] = {m->W1, m->mW1, m->vW1, m->best_W1, m->gamma, m->beta, m->mmean, m->mvar, m->m_gamma, m->v_gamma,
                   m->m_beta, m->v_beta, m->best_gamma, m->best_beta, m->best_mmean, m->best_mvar, m->small, m->w_fs, m->w_bs,
                   m->m_small, m->v_small, m->best_small, m->partials, m->acts, m->dzs, m->outs, m->hist, m->wide,
                   m->val_slots, m->bb_mean, m->bb_var, m->bb_pq};
  for (float* p : ptrs)
    if (p) cudaFree(p);
  if (m->st) cudaFree(m->st);
  if (m->dbg) cudaFree(m->dbg);
  if (m->side) cudaStreamDestroy(m->side);
  if (m->ev_hid) cudaEventDestroy(m->ev_hid);
  if (m->ev_upd) cudaEventDestroy(m->ev_upd);
  delete m;
}

void pool_clear_locked() {
  for (loc_model* m : g_pool) free_model(m);
  g_pool.clear();
}

// cudaMalloc that gives the pool's memory back before it reports failure
cudaError_t dev_alloc(void** p, size_t bytes) {
  cudaError_t e = cudaMalloc(p, bytes);
  if (e == cudaSuccess) return e;
  cudaGetLastError();
  {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if (g_pool.empty()) return e;
    pool_clear_locked();
  }
  return cudaMalloc(p, bytes);
}
template <class T>
cudaError_t dev_alloc(T** p, size_t bytes) {
  return dev_alloc(reinterpret_cast<void**>(p), bytes);
}

loc_model* pool_take(int dev, int64_t K, int width, int nlayers, int use_tc, int hid_tc, int max_epochs, bool want_dbg,
                     int chunks) {
  std::lock_guard<std::mutex> lk(g_pool_mu);
  for (size_t i = 0; i < g_pool.size(); ++i) {
    loc_model* m = g_pool[i];
    if (m->dev == dev && m->H == width && m->L == nlayers && m->use_tc == use_tc && m->hid_tc == hid_tc &&
        m->cap_K >= K && (double)K >= 0.6 * (double)m->cap_K && m->cap_epochs >= max_epochs && (m->dbg != nullptr) == want_dbg &&
        m->cap_chunks == chunks) {
      g_pool.erase(g_pool.begin() + (long)i);
      return m;
    }
  }
  return nullptr;
}
}  // namespace

// K-dependent launch geometry (also after a pooled handle changes its K)
static void set_geometry(loc_model* m, int64_t K) {
  m->K = K;
  m->K_global = K;
  m->k_offset = 0;
  const int sms = sm_count();
  if (m->use_tc) {
    // One CTA per SM (or per tile for small K).  loc_model_set_l1_ctas lowers the count: replicate groups of
    // large models keep one 16-SM cluster's worth of SMs free for the hidden stacks (ring schedule).  The count
    // fixes the fp32 summation order of the layer.
    m->n_partials = l1_tc_partials(K);
    m->n_bwd_blocks = m->n_partials;
  } else {
    const int64_t nch = cdiv(K, kF1Chunk);
    m->n_partials = (int)(nch < 2 * sms ? nch : 2 * sms);
    const int64_t nch2 = cdiv(K, 32);
    m->n_bwd_blocks = (int)(nch2 < 2 * sms ? nch2 : 2 * sms);
  }
  m->Kpad = m->use_tc ? (K + 63) / 64 * 64 : K;
}

// what loc_model_create guarantees about the contents of a new handle's buffers
static int zero_model(loc_model* m) {
  const int64_t KH = m->Kpad * m->H;
  float* big[] = {m->W1, m->mW1, m->vW1, m->best_W1};
  for (float* p : big) LOC_CUDA(cudaMemsetAsync(p, 0, KH * sizeof(float), 0));  // padding rows stay zero under Adam
  LOC_CUDA(cudaMemsetAsync(m->st, 0, sizeof(DevState), 0));
  LOC_CUDA(cudaMemsetAsync(m->dzs, 0, (size_t)m->cap_chunks * m->L * kMaxB * m->H * sizeof(float), 0));
  LOC_CUDA(cudaMemsetAsync(m->acts, 0, (size_t)m->cap_chunks * m->L * kMaxB * m->H * sizeof(float), 0));
  LOC_CUDA(cudaMemsetAsync(m->hist, 0, (size_t)m->max_epochs * 3 * sizeof(float), 0));
  if (m->dbg) LOC_CUDA(cudaMemsetAsync(m->dbg, 0, 16 * 256 * sizeof(long long), 0));
  LOC_CUDA(cudaStreamSynchronize(0));  // callers may continue on non-blocking streams
  return 0;
}

extern "C" {

int loc_model_create(loc_model** out, int64_t K, int32_t width, int32_t nlayers, int32_t batch_size,
                     float dropout_prop, int32_t max_epochs) {
  LOC_CHECK(out != nullptr, "loc_model_create: null output pointer");
  *out = nullptr;
  LOC_CHECK(K > 0, "loc_model_create: K must be positive");
  LOC_CHECK(width >= 32 && width <= 1024 && width % 32 == 0, "loc_model_create: width must be a multiple of 32 in [32, 1024]");
  LOC_CHECK(nlayers >= 2 && nlayers <= 64, "loc_model_create: nlayers must be in [2, 64]");
  LOC_CHECK(batch_size >= 1 && batch_size <= LOC_MAX_BATCH_SIZE, "loc_model_create: batch_size must be in [1, 256]");
  const int chunks = (batch_size + kMaxB - 1) / kMaxB;  // 32-row chunks of a step (bigbatch.cu for more than one)
  LOC_CHECK(dropout_prop >= 0.f && dropout_prop < 1.f, "loc_model_create: dropout_prop must be in [0, 1)");
  LOC_CHECK(max_epochs >= 1, "loc_model_create: max_epochs must be >= 1");
  int ndev = 0;
  LOC_CUDA(cudaGetDeviceCount(&ndev));
  LOC_CHECK(ndev > 0, "loc_model_create: no CUDA device (this library has no CPU fallback)");
  int dev = 0;
  LOC_CUDA(cudaGetDevice(&dev));
  const int hid_tc = hidden_tc_supported(width, nlayers);
  const int use_tc = l1_tc_supported(K, width);
  const bool want_dbg = getenv("LOC_HID_TRACE") != nullptr;
  if (loc_model* r = pool_limit() > 0 ? pool_take(dev, K, width, nlayers, use_tc, hid_tc, max_epochs, want_dbg, chunks) : nullptr) {
    // a recycled handle: same buffers, new shape and settings, nothing bound
    set_geometry(r, K);
    r->B = batch_size;
    r->max_epochs = max_epochs;
    r->p_drop = dropout_prop;
    r->seed = 0;
    r->train_packed = r->val_packed = nullptr;
    r->train_locs = r->val_locs = nullptr;
    r->n_train = r->n_val = r->train_row_words = r->val_row_words = 0;
    r->masks = nullptr;
    r->n_masks = 0;
    r->exchange = nullptr;
    r->exchange_ctx = nullptr;
    r->z1_tile = nullptr;
    r->tp = nullptr;
    r->span_perm = nullptr;
    r->span_next = 0;
    r->h_steps = 0;
    r->h_hid_seq = r->h_bwd_cnt = r->h_upd_cnt = 0u;
    r->chain_open = 0;
    if (zero_model(r)) {
      free_model(r);
      return 1;
    }
    r->tl_id = g_tl_models++;
    *out = r;
    return 0;
  }
  loc_model* m = new (std::nothrow) loc_model();
  LOC_CHECK(m != nullptr, "loc_model_create: out of host memory");
  memset(m, 0, sizeof(*m));
  m->dev = dev;
  m->H = width;
  m->L = nlayers;
  m->B = batch_size;
  m->n_before = nlayers / 2;
  m->max_epochs = max_epochs;
  m->cap_epochs = max_epochs;
  m->p_drop = dropout_prop;
  m->sl = SmallLayout{width, nlayers};
  m->cluster = hidden_max_cluster(width, nlayers);
  if (m->cluster <= 0) {
    delete m;
    return loc::fail("loc_model_create: no usable thread-block cluster size for this width / nlayers", __FILE__, __LINE__);
  }
  m->n_slots = hidden_slots(width, nlayers, m->cluster);
  m->hid_tc = hid_tc;
  m->use_tc = use_tc;
  set_geometry(m, K);
  m->cap_K = K;
  m->cap_chunks = chunks;
  m->cap_partials = m->use_tc ? l1_tc_partials(K) : m->n_partials;
  const int64_t KH = m->Kpad * width, ns = m->sl.total();
#define LOC_ALLOC(ptr, bytes)                                 \
  do {                                                        \
    if (dev_alloc(&(ptr), (bytes)) != cudaSuccess) {          \
      cudaGetLastError();                                     \
      free_model(m);                                          \
      return loc::fail("loc_model_create: out of device memory", __FILE__, __LINE__); \
    }                                                         \
  } while (0)
  float** big[] = {&m->W1, &m->mW1, &m->vW1, &m->best_W1};
  for (auto p : big) LOC_ALLOC(*p, KH * sizeof(float));
  float** kv[] = {&m->gamma, &m->beta, &m->mmean, &m->mvar, &m->m_gamma, &m->v_gamma, &m->m_beta,
                  &m->v_beta, &m->best_gamma, &m->best_beta, &m->best_mmean, &m->best_mvar};
  for (auto p : kv) LOC_ALLOC(*p, K * sizeof(float));
  float** sm[] = {&m->small, &m->m_small, &m->v_small, &m->best_small};
  for (auto p : sm) LOC_ALLOC(*p, ns * sizeof(float));
  LOC_ALLOC(m->w_fs, (size_t)(nlayers - 1) * width * width * sizeof(float));
  LOC_ALLOC(m->w_bs, (size_t)(nlayers - 1) * width * width * sizeof(float));
  LOC_ALLOC(m->partials, (size_t)m->cap_partials * kMaxB * width * sizeof(float));
  LOC_ALLOC(m->acts, (size_t)chunks * nlayers * kMaxB * width * sizeof(float));
  LOC_ALLOC(m->dzs, (size_t)chunks * nlayers * kMaxB * width * sizeof(float));
  if (chunks > 1) {
    LOC_ALLOC(m->bb_mean, K * sizeof(float));
    LOC_ALLOC(m->bb_var, K * sizeof(float));
    LOC_ALLOC(m->bb_pq, (size_t)bb_pq_floats(K, width) * sizeof(float));
  }
  LOC_ALLOC(m->outs, 8 * 256 * sizeof(float));  // one [256] block per 32-row chunk of a wide pass
  LOC_ALLOC(m->val_slots, 16 * sizeof(float));
  if (m->use_tc && m->hid_tc) LOC_ALLOC(m->wide, (size_t)m->cap_partials * 256 * width * sizeof(float));
  LOC_ALLOC(m->hist, (size_t)max_epochs * 3 * sizeof(float));
  if (want_dbg) LOC_ALLOC(m->dbg, 16 * 256 * sizeof(long long));
  LOC_ALLOC(m->st, sizeof(DevState));
#undef LOC_ALLOC
  if (cudaStreamCreateWithFlags(&m->side, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&m->ev_hid, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&m->ev_upd, cudaEventDisableTiming) != cudaSuccess || zero_model(m)) {
    free_model(m);
    return loc::fail("loc_model_create: stream / event / memset failed", __FILE__, __LINE__);
  }
  m->tl_id = g_tl_models++;
  *out = m;
  return 0;
}

int loc_model_destroy(loc_model* m) {
  if (m == nullptr) return 0;
  int dev = -1;
  cudaGetDevice(&dev);
  if (pool_limit() > 0 && dev == m->dev) {
    // everything queued on the handle's buffers must be done before another model may take them
    cudaDeviceSynchronize();
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if ((int)g_pool.size() >= pool_limit()) {
      free_model(g_pool.front());
      g_pool.erase(g_pool.begin());
    }
    g_pool.push_back(m);
    return 0;
  }
  free_model(m);
  return 0;
}

int loc_model_pool_clear(void) {
  std::lock_guard<std::mutex> lk(g_pool_mu);
  pool_clear_locked();
  return 0;
}

const char* loc_model_impl(const loc_model* m) { return (m != nullptr && m->use_tc) ? "tcgen05" : "simt"; }

const char* loc_model_hidden_impl(const loc_model* m) { return (m != nullptr && m->hid_tc) ? "tcgen05" : "simt"; }

int32_t loc_hidden_max_nlayers(int32_t width) { return hidden_max_nlayers(width); }

int loc_model_init(loc_model* m, uint64_t seed, void* stream) {
  LOC_CHECK(m != nullptr, "loc_model_init: null model");
  cudaStream_t s = (cudaStream_t)stream;
  m->seed = seed;
  const int64_t K = m->K, H = m->H, L = m->L;
  if (fill(m->gamma, K, 1.f, s) || fill(m->beta, K, 0.f, s) || fill(m->mmean, K, 0.f, s) || fill(m->mvar, K, 1.f, s))
    return 1;
  float* zeroK[] = {m->m_gamma, m->v_gamma, m->m_beta, m->v_beta};
  for (float* p : zeroK)
    if (fill(p, K, 0.f, s)) return 1;
  if (fill(m->W1, m->Kpad * H, 0.f, s) || fill(m->mW1, m->Kpad * H, 0.f, s) || fill(m->vW1, m->Kpad * H, 0.f, s)) return 1;
  if (fill(m->small, m->sl.total(), 0.f, s) || fill(m->m_small, m->sl.total(), 0.f, s) ||
      fill(m->v_small, m->sl.total(), 0.f, s))
    return 1;
  // Dense kernel i (0-based over the L+2 Dense layers) draws from Philox stream 16+i.
  auto glorot = [&](float* w, int64_t fan_in, int64_t fan_out, int layer) -> int {
    const float limit = (float)sqrt(6.0 / (double)(fan_in + fan_out));
    const int64_t n = fan_in * fan_out;
    int64_t blocks = cdiv(n, 256 * 4);
    if (blocks > sm_count() * 8) blocks = sm_count() * 8;
    k_glorot<<<(unsigned)blocks, 256, 0, s>>>(w, n, limit, 16u + (uint32_t)layer, seed);
    LOC_LAUNCHED();
    return 0;
  };
  if (m->use_tc) {
    const float limit = (float)sqrt(6.0 / (double)(m->K_global + H));
    k_glorot_tiled<<<sm_count() * 8, 256, 0, s>>>(m->W1, K, (int)H, limit, 16u, seed, m->k_offset);
    LOC_LAUNCHED();
  } else if (glorot(m->W1, K, H, 0)) {
    return 1;
  }
  for (int i = 1; i < L; ++i)
    if (glorot(m->small + m->sl.Wh(i), H, H, i)) return 1;
  if (glorot(m->small + m->sl.Wo1(), H, 2, (int)L)) return 1;
  if (glorot(m->small + m->sl.Wo2(), 2, 2, (int)L + 1)) return 1;
  if (reslice(m, s)) return 1;
  k_state_reset<<<1, 1, 0, s>>>(m->st, 1e-3f, 100, m->max_epochs, 1);
  LOC_LAUNCHED();
  m->h_steps = 0;
  m->h_hid_seq = m->h_bwd_cnt = m->h_upd_cnt = 0u;
  m->chain_open = 0;
  return 0;
}

int loc_model_num_weights(const loc_model* m) { return m ? 4 + 2 * (m->L + 2) : 0; }

namespace {
// Keras order -> (pointer, Adam m, Adam v, length)
struct WRef {
  float *w, *am, *av;
  int64_t n;
};
bool weight_ref(const loc_model* m, int idx, WRef* r) {
  const int64_t K = m->K, H = m->H;
  const int L = m->L;
  if (idx < 0 || idx >= 4 + 2 * (L + 2)) return false;
  switch (idx) {
    case 0: *r = {m->gamma, m->m_gamma, m->v_gamma, K}; return true;
    case 1: *r = {m->beta, m->m_beta, m->v_beta, K}; return true;
    case 2: *r = {m->mmean, nullptr, nullptr, K}; return true;
    case 3: *r = {m->mvar, nullptr, nullptr, K}; return true;
    case 4: *r = {m->W1, m->mW1, m->vW1, K * H}; return true;
    default: break;
  }
  const int d = (idx - 4) / 2, isb = (idx - 4) % 2;  // dense layer d in 0..L+1
  int64_t off, n;
  if (d == 0) {
    off = m->sl.b1();
    n = H;  // only the bias lands here (idx 5)
  } else if (d < L) {
    off = isb ? m->sl.bh(d) : m->sl.Wh(d);
    n = isb ? H : H * H;
  } else if (d == L) {
    off = isb ? m->sl.bo1() : m->sl.Wo1();
    n = isb ? 2 : 2 * H;
  } else {
    off = isb ? m->sl.bo2() : m->sl.Wo2();
    n = isb ? 2 : 4;
  }
  *r = {m->small + off, m->m_small + off, m->v_small + off, n};
  return true;
}
}  // namespace

int64_t loc_model_weight_size(const loc_model* m, int32_t idx) {
  WRef r;
  if (m == nullptr || !weight_ref(m, idx, &r)) return -1;
  return r.n;
}

int loc_model_set_weight(loc_model* m, int32_t idx, const float* h_src, int64_t n, void* stream) {
  WRef r;
  LOC_CHECK(m != nullptr && weight_ref(m, idx, &r), "loc_model_set_weight: bad weight index");
  LOC_CHECK(n == r.n, "loc_model_set_weight: size mismatch");
  if (idx == 4 && m->use_tc) return w1_upload(m, r.w, h_src, (cudaStream_t)stream);
  LOC_CUDA(cudaMemcpyAsync(r.w, h_src, n * sizeof(float), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  if (idx >= 6 && reslice(m, (cudaStream_t)stream)) return 1;
  LOC_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return 0;
}

int loc_model_get_weight(loc_model* m, int32_t idx, float* h_dst, int64_t n, void* stream) {
  WRef r;
  LOC_CHECK(m != nullptr && weight_ref(m, idx, &r), "loc_model_get_weight: bad weight index");
  LOC_CHECK(n == r.n, "loc_model_get_weight: size mismatch");
  if (idx == 4 && m->use_tc) return w1_download(m, r.w, h_dst, (cudaStream_t)stream);
  LOC_CUDA(cudaMemcpyAsync(h_dst, r.w, n * sizeof(float), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  LOC_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return 0;
}

int loc_model_get_adam(loc_model* m, int32_t idx, float* h_m, float* h_v, int64_t n, void* stream) {
  WRef r;
  LOC_CHECK(m != nullptr && weight_ref(m, idx, &r), "loc_model_get_adam: bad weight index");
  LOC_CHECK(r.am != nullptr, "loc_model_get_adam: weight is not trainable");
  LOC_CHECK(n == r.n, "loc_model_get_adam: size mismatch");
  if (idx == 4 && m->use_tc) {
    if (w1_download(m, r.am, h_m, (cudaStream_t)stream)) return 1;
    return w1_download(m, r.av, h_v, (cudaStream_t)stream);
  }
  LOC_CUDA(cudaMemcpyAsync(h_m, r.am, n * sizeof(float), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  LOC_CUDA(cudaMemcpyAsync(h_v, r.av, n * sizeof(float), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  LOC_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return 0;
}

int loc_model_set_shard(loc_model* m, int64_t k_offset, int64_t K_global) {
  LOC_CHECK(m != nullptr && k_offset >= 0 && K_global >= k_offset + m->K, "loc_model_set_shard: bad arguments");
  LOC_CHECK(m->use_tc && m->hid_tc, "loc_model_set_shard: sharded models need the tcgen05 kernels (width 256)");
  LOC_CHECK(m->B <= kMaxB, "loc_model_set_shard: sharded models train with batch_size <= 32");
  m->k_offset = k_offset;
  m->K_global = K_global;
  return 0;
}

int loc_model_set_exchange(loc_model* m, loc_exchange_fn fn, void* ctx, float* d_tile) {
  LOC_CHECK(m != nullptr && (fn == nullptr || d_tile != nullptr), "loc_model_set_exchange: bad arguments");
  LOC_CHECK(fn == nullptr || (m->use_tc && m->hid_tc),
            "loc_model_set_exchange: sharded models need the tcgen05 kernels (width 256)");
  m->exchange = fn;
  m->exchange_ctx = ctx;
  m->z1_tile = d_tile;
  return 0;
}

int loc_model_set_tp(loc_model* m, loc_tp* tp) {
  LOC_CHECK(m != nullptr, "loc_model_set_tp: null model");
  LOC_CHECK(tp == nullptr || (m->use_tc && m->hid_tc), "loc_model_set_tp: sharded models need the tcgen05 kernels (width 256)");
  m->tp = tp;
  return 0;
}

int loc_model_set_l1_ctas(loc_model* m, int32_t n_ctas) {
  LOC_CHECK(m != nullptr && n_ctas >= 1, "loc_model_set_l1_ctas: bad arguments");
  LOC_CHECK(m->use_tc, "loc_model_set_l1_ctas: needs the tcgen05 first layer (width 256)");
  const int full = l1_tc_partials(m->K) < m->cap_partials ? l1_tc_partials(m->K) : m->cap_partials;
  m->n_partials = n_ctas < full ? n_ctas : full;
  m->n_bwd_blocks = m->n_partials;
  return 0;
}

int loc_model_set_schedule(loc_model* m, float lr, int32_t patience) {
  LOC_CHECK(m != nullptr, "loc_model_set_schedule: null model");
  LOC_CHECK(patience >= 0, "loc_model_set_schedule: patience must be >= 0");
  k_state_reset<<<1, 1>>>(m->st, lr, patience, m->max_epochs, 0);
  LOC_LAUNCHED();
  m->h_hid_seq = m->h_bwd_cnt = m->h_upd_cnt = 0u;
  m->chain_open = 0;
  LOC_CUDA(cudaDeviceSynchronize());
  return 0;
}

int loc_model_bind_train(loc_model* m, const uint32_t* d_packed, int64_t n, int64_t row_words, const float* d_locs) {
  LOC_CHECK(m != nullptr && d_packed != nullptr && d_locs != nullptr && n > 0, "loc_model_bind_train: bad arguments");
  LOC_CHECK(row_words >= cdiv(m->K, 16), "loc_model_bind_train: row_words too small for K");
  m->train_packed = d_packed;
  m->n_train = n;
  m->train_row_words = row_words;
  m->train_locs = d_locs;
  return 0;
}

int loc_model_bind_val(loc_model* m, const uint32_t* d_packed, int64_t n, int64_t row_words, const float* d_locs) {
  LOC_CHECK(m != nullptr && d_packed != nullptr && d_locs != nullptr && n > 0, "loc_model_bind_val: bad arguments");
  LOC_CHECK(row_words >= cdiv(m->K, 16), "loc_model_bind_val: row_words too small for K");
  m->val_packed = d_packed;
  m->n_val = n;
  m->val_row_words = row_words;
  m->val_locs = d_locs;
  return 0;
}

int loc_model_set_dropout_masks(loc_model* m, const uint8_t* d_keep, int64_t nsteps) {
  LOC_CHECK(m != nullptr, "loc_model_set_dropout_masks: null model");
  m->masks = d_keep;
  m->n_masks = d_keep ? nsteps : 0;
  return 0;
}

int loc_train_step(loc_model* m, const int32_t* d_rows, int32_t nb, void* stream) {
  LOC_CHECK(m != nullptr && m->train_packed != nullptr, "loc_train_step: no training data bound");
  LOC_CHECK(d_rows != nullptr && nb >= 1 && nb <= m->B, "loc_train_step: bad batch");
  m->span_perm = nullptr;
  return train_step(m, order_rows(d_rows, 0, 0, nb), 0, (cudaStream_t)stream);
}

int loc_debug_stage(loc_model* m, int32_t stage, const int32_t* d_rows, int32_t nb, void* stream) {
  LOC_CHECK(m != nullptr && m->train_packed != nullptr, "loc_debug_stage: no training data bound");
  LOC_CHECK(stage >= 0 && stage < 5 && d_rows != nullptr && nb >= 1 && nb <= m->B, "loc_debug_stage: bad arguments");
  LOC_CHECK(m->B <= kMaxB, "loc_debug_stage: single stages are only available for batch_size <= 32");
  cudaStream_t s = (cudaStream_t)stream;
  m->span_perm = nullptr;
  m->chain_open = 0;
  const RowSrc src = order_rows(d_rows, 0, 0, nb);
  L1Args a = l1_args(m, m->train_packed, m->train_row_words, src, 1, 0);
  switch (stage) {
    case 0:  // first-layer forward (+ the shard exchange)
      return forward_l1(m, a, s) || exchange_partials(m, s);
    case 1: {  // training hidden stack
      HidArgs h = hid_args(m, src, 1, 0, m->train_locs, nullptr);
      begin_training_hidden(m, h);
      return hidden_stack(m, h, s);
    }
    case 2:  // first-layer backward + Adam
      return backward_l1(m, a, s);
    case 3:  // small-layer update
      return update_launch(m, upd_args(m, nb, 0), s);
    default:  // 4: first-layer backward + Adam with the next forward (same rows) fused in on the tcgen05 path
      if (m->use_tc) {
        a.src_next = src;
        a.fuse_next = 1;
      }
      return backward_l1(m, a, s);
  }
}

static int end_epoch(loc_model* m, cudaStream_t s) {
  if (infer_rows(m, m->val_packed, m->n_val, m->val_row_words, m->val_locs, nullptr, 1, s)) return 1;
  k_epoch_end<<<1, 1, 0, s>>>(m->st, m->hist);
  LOC_LAUNCHED();
  return copy_weights(m, true, &m->st->improved, s);
}

// below this many SNPs the first-layer backward is shorter than the hidden stack (42 us ~ 35k SNPs)
static const int64_t kRingMinK = 32768;

int loc_group_train_epochs(loc_model** models, int32_t n_models, const int32_t* const* d_perms, int32_t n_epochs,
                           void* stream) {
  LOC_CHECK(models != nullptr && d_perms != nullptr && n_models >= 1 && n_models <= kMaxGroup && n_epochs >= 1,
            "loc_group_train_epochs: bad arguments");
  loc_model* m0 = models[0];
  int64_t n_max = 0;  // rows of the largest training set: the epoch's last step offset is below it
  for (int g = 0; g < n_models; ++g) {
    loc_model* m = models[g];
    LOC_CHECK(m != nullptr && d_perms[g] != nullptr && m->train_packed != nullptr && m->val_packed != nullptr,
              "loc_group_train_epochs: every model needs bound training / validation data and a batch order");
    LOC_CHECK(m->use_tc == m->hid_tc,
              "loc_group_train_epochs: models whose first layer and hidden stack run on different kernel families (width 256 "
              "with 15..21 layers: tcgen05 first layer, CUDA-core hidden stack) cannot be grouped");
    LOC_CHECK(m->hid_tc == m0->hid_tc,
              "loc_group_train_epochs: the models of a group must all run the tcgen05 kernels (width 256, nlayers <= 14) or all "
              "the CUDA-core kernels");
    LOC_CHECK(m->exchange == nullptr && m->tp == nullptr, "loc_group_train_epochs: sharded models cannot be grouped");
    LOC_CHECK(m->H == m0->H && m->L == m0->L && m->B == m0->B && m->cluster == m0->cluster,
              "loc_group_train_epochs: replicates of a group must share width, nlayers, batch size and hidden-stack cluster "
              "size");
    if (m->n_train > n_max) n_max = m->n_train;
  }
  cudaStream_t s = (cudaStream_t)stream;
  for (int g = 0; g < n_models; ++g) {
    models[g]->chain_open = 0;
    models[g]->span_perm = nullptr;
    k_begin_call<<<1, 1, 0, s>>>(models[g]->st);
    LOC_LAUNCHED();
  }
  // Training sets may differ in size: the step at offset `off` holds the models with off < n_train, each with its own
  // rows, its own next step and its own epoch end -- the arguments it gets alone.
  auto rows = [&](int g, int64_t off) { return step_rows(models[g], d_perms[g], models[g]->n_train, off); };
  auto steps_at = [&](int g, int64_t off) { return off < models[g]->n_train; };
  auto has_next = [&](int g, int64_t off) { return off + m0->B < models[g]->n_train; };
  // Schedule.  "ring" (default whenever every model's first-layer kernels leave one cluster's worth of SMs
  // free, loc_model_set_l1_ctas): one stream, per slot  H(g) -> B(g-1) -> U(g-1)  where H is the 16-CTA hidden
  // stack of model g (plain launch: starts when everything before it is complete), B the first-layer backward
  // + Adam (+ next forward) of the PREVIOUS model in the ring and U that model's small-layer update, both
  // launched with programmatic stream serialization: B starts as soon as H's cluster is placed and streams
  // W1/m/v on the other SMs while H's dependent chain of layer products runs; U takes H's SMs when H exits.
  // B(g-1) only needs H(g-1) (complete since the previous slot) and nothing from H(g).  A slot costs
  // max(B, H) instead of B + H / G -- a gain only when the weight stream outlasts the hidden stack, hence
  // K >= kRingMinK.  "lockstep" (small K, models on all SMs, or LOC_GROUP_SCHEDULE=lockstep): all hidden
  // stacks in one launch, then the backwards back to back, updates on side streams.
  // CUDA-core models (widths other than 256) always run the lockstep, without fused forwards: the CUDA-core
  // first-layer backward has none, and the ring pays only where the tcgen05 weight stream outlasts the stack
  // (LOC_GROUP_SCHEDULE does not apply to them).
  // Models of more than 32 rows a step ("large batch", LOC_GROUP_SCHEDULE does not apply): train_step_big with the
  // whole group, a lockstep of its own -- one statistics launch, hidden stacks packed whole models per launch (tcgen05)
  // or chunk c of every model per launch (CUDA cores), the backwards back to back, updates on side streams.
  const bool big = m0->B > kMaxB;
  const bool fuse = m0->use_tc;  // the backward also runs the next step's forward
  const char* sched = getenv("LOC_GROUP_SCHEDULE");  // "ring" / "lockstep" override the choice by K (tests, A/B)
  bool ring = !big && m0->hid_tc && n_models >= 2 && (m0->K >= kRingMinK || (sched != nullptr && strcmp(sched, "ring") == 0));
  for (int g = 0; g < n_models; ++g) ring = ring && models[g]->n_bwd_blocks <= sm_count() - kHidTcCtas;
  if (sched != nullptr && strcmp(sched, "lockstep") == 0) ring = false;
  struct Pending {
    loc_model* m;
    L1Args a;
    UpdArgs u;
    unsigned hid_seq;  // what the model's hidden stack of this step publishes when it is done
  };
  for (int e = 0; e < n_epochs; ++e) {
    if (ring) {
      // rings of two models (three for the last ring of an odd group): a model comes back after ONE other
      // model's weight stream, so the tail of its previous step's updates is still in L2 (rings of four
      // measured 4 % slower).  Each ring runs its whole epoch; the models are independent.
      for (int g0 = 0; g0 < n_models;) {
        const int g1 = (n_models - g0 == 3) ? n_models : (g0 + 2 < n_models ? g0 + 2 : n_models);
        // Rings of two also hand over through the device flags of the chained step (train_step): in the stream
        // ... B(m) U(m) H(m) ... every hidden stack directly follows its own model's update, so it can be launched
        // with programmatic serialization too -- placed and set up while the OTHER model's backward streams,
        // waiting for its own model's previous backward by DevState::bwd_cnt.  The backward kernels then follow
        // each other without a gap: a slot costs one weight stream, not stream + kernel boundaries.
        const bool chain2 = g1 - g0 == 2 && getenv("LOC_NO_CHAIN") == nullptr;
        bool have_fwd = false;
        Pending pend;
        pend.m = nullptr;
        auto launch_pending = [&](bool overlap) -> int {
          pend.a.wait_hid = pend.hid_seq;
          pend.a.wait_bwd = pend.m->h_bwd_cnt;
          pend.u.wait_hid = pend.hid_seq;
          if (backward_l1(pend.m, pend.a, s, overlap)) return 1;
          return update_launch(pend.m, pend.u, s, overlap);
        };
        for (int64_t off = 0; off < n_max; off += m0->B) {
          for (int g = g0; g < g1; ++g) {
            if (!steps_at(g, off)) continue;  // this model's epoch has ended: its slot is skipped
            loc_model* m = models[g];
            // the other models of the ring have ended their epoch: this model's own previous backward and update go
            // first, and its hidden stack follows them as in a solo chained step
            if (pend.m == m && launch_pending(true)) return 1;
            if (pend.m == m) pend.m = nullptr;
            const RowSrc src = rows(g, off);
            L1Args a = l1_args(m, m->train_packed, m->train_row_words, src, 1, 1);
            if (!have_fwd && forward_l1(m, a, s)) return 1;  // first step of the epoch: later ones are fused
            HidArgs h = hid_args(m, src, 1, 1, m->train_locs, nullptr);
            begin_training_hidden(m, h);
            const bool h_overlaps = chain2 && have_fwd;  // directly behind this model's own backward + update
            if (h_overlaps) h.wait_bwd = m->h_bwd_cnt;
            if (hidden_stack(m, h, s, h_overlaps)) return 1;
            if (pend.m != nullptr && launch_pending(true)) return 1;
            if (has_next(g, off)) {
              a.src_next = rows(g, off + m0->B);
              a.fuse_next = 1;
            }
            pend.m = m;
            pend.a = a;
            pend.u = upd_args(m, src.nb, 1);
            pend.hid_seq = h.hid_seq;
          }
          have_fwd = true;  // every model with a step at the next offset fused its forward into this step's backward
        }
        if (pend.m != nullptr && launch_pending(false)) return 1;  // the ring's last backward and update of the epoch
        g0 = g1;
      }
    }
    for (int64_t off = 0; !ring && off < n_max; off += m0->B) {
      // the models with a step at this offset
      loc_model* ms[kMaxGroup];
      RowSrc srcs[kMaxGroup];
      int act[kMaxGroup], n = 0;
      for (int g = 0; g < n_models; ++g)
        if (steps_at(g, off)) {
          ms[n] = models[g];
          srcs[n] = rows(g, off);
          act[n++] = g;
        }
      if (big) {
        if (train_step_big(ms, srcs, n, 1, s)) return 1;
        continue;
      }
      HidGroupArgs hg;
      hg.n = n;
      // first-layer forwards (first step of the epoch only: later ones are fused into the backward)
      for (int i = 0; i < n; ++i) {
        loc_model* m = ms[i];
        if (!(fuse && off > 0)) {
          L1Args a = l1_args(m, m->train_packed, m->train_row_words, srcs[i], 1, 1);
          if (forward_l1(m, a, s)) return 1;
        }
        hg.a[i] = hid_args(m, srcs[i], 1, 1, m->train_locs, nullptr);
        begin_training_hidden(m, hg.a[i]);
      }
      // all hidden stacks in one launch: one cluster per replicate
      if (hidden_stacks(m0, hg, s)) return 1;
      // small-layer updates on the side streams, first-layer backward (+ next forward) back to back
      if (fork_updates(ms, n, s, [&](int i, cudaStream_t su) {
            return update_launch(ms[i], upd_args(ms[i], srcs[i].nb, 1), su);
          }))
        return 1;
      for (int i = 0; i < n; ++i) {
        loc_model* m = ms[i];
        L1Args a = l1_args(m, m->train_packed, m->train_row_words, srcs[i], 1, 1);
        if (fuse && has_next(act[i], off)) {
          a.src_next = rows(act[i], off + m0->B);
          a.fuse_next = 1;
        }
        if (backward_l1(m, a, s)) return 1;
      }
      if (join_updates(ms, n, s)) return 1;
    }
    for (int g = 0; g < n_models; ++g)
      if (end_epoch(models[g], s)) return 1;
  }
  return 0;
}

int64_t loc_debug_timeline(uint64_t* h_out, int64_t max_records) {
  // records as (ns, tag << 32 | model) pairs; the buffer is cleared.  Tags: 1/2 first-layer backward start / end,
  // 3/4 hidden stack, 5/6 small-layer update, 7/8 first-layer forward (standalone or wide); +16: last block
  unsigned long long* tl = timeline_buffer();
  if (tl == nullptr || h_out == nullptr) return 0;
  cudaDeviceSynchronize();
  unsigned long long n = 0;
  cudaMemcpy(&n, tl, sizeof(n), cudaMemcpyDeviceToHost);
  n &= 0xffffffffull;
  if (n > kTlCap) n = kTlCap;
  const int64_t c = (int64_t)n < max_records ? (int64_t)n : max_records;
  cudaMemcpy(h_out, tl + 1, (size_t)c * 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
  cudaMemset(tl, 0, sizeof(unsigned long long));
  return c;
}

int64_t loc_debug_read(loc_model* m, int32_t which, float* h_dst, int64_t max_n, void* stream) {
  if (m != nullptr && which == 3 && m->dbg != nullptr && h_dst != nullptr) {  // clock trace of k_hidden
    const int64_t n = 16 * 256 * 2;                                             // as float pairs (raw int64 bits)
    const int64_t c = n < max_n ? n : max_n;
    cudaMemcpyAsync(h_dst, m->dbg, c * sizeof(float), cudaMemcpyDeviceToHost, (cudaStream_t)stream);
    cudaStreamSynchronize((cudaStream_t)stream);
    return n;
  }
  if (m == nullptr || h_dst == nullptr || which < 0 || which > 2) {
    loc::fail("loc_debug_read: bad arguments", __FILE__, __LINE__);
    return -1;
  }
  const float* src = which == 0 ? m->partials : (which == 1 ? m->dzs : m->acts);
  const int64_t n = which == 0 ? (int64_t)m->n_partials * kMaxB * m->H : (int64_t)m->L * kMaxB * m->H;
  const int64_t c = n < max_n ? n : max_n;
  if (cudaMemcpyAsync(h_dst, src, c * sizeof(float), cudaMemcpyDeviceToHost, (cudaStream_t)stream) != cudaSuccess ||
      cudaStreamSynchronize((cudaStream_t)stream) != cudaSuccess) {
    loc::fail("loc_debug_read: copy failed", __FILE__, __LINE__);
    return -1;
  }
  return n;
}

// Steps [step0, step0 + nsteps) of one epoch (batch order `perm`, or perm + (epoch - epoch0) * epoch_stride when the
// device-side epoch counter selects the row of a multi-epoch order).  Inside an epoch every backward also runs
// the NEXT step's first-layer forward (tcgen05 path), so only a span that starts without such a forward
// launches one of its own.  *have_fwd: in = the tiles of step0 are already there; out = those of the step
// after the span are.
static int run_span(loc_model* m, const int32_t* perm, int64_t epoch_stride, int64_t step0, int64_t nsteps, int gated,
                    bool* have_fwd, cudaStream_t s) {
  const bool fuse = m->use_tc && m->B <= kMaxB;
  for (int64_t st = step0; st < step0 + nsteps; ++st) {
    const int64_t off = st * m->B;
    const RowSrc src = step_rows(m, perm, epoch_stride, off);
    const bool has_next = fuse && off + m->B < m->n_train;  // within the epoch (the validation pass reuses the tiles)
    const RowSrc next = has_next ? step_rows(m, perm, epoch_stride, off + m->B) : src;
    if (train_step(m, src, gated, s, has_next ? &next : nullptr, *have_fwd)) return 1;
    *have_fwd = has_next;
  }
  return 0;
}

int loc_train_epochs(loc_model* m, const int32_t* d_perms, int32_t n_epochs, void* stream) {
  LOC_CHECK(m != nullptr && m->train_packed != nullptr && m->val_packed != nullptr,
            "loc_train_epochs: training and validation data must be bound");
  LOC_CHECK(d_perms != nullptr && n_epochs >= 1, "loc_train_epochs: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  m->span_perm = nullptr;
  k_begin_call<<<1, 1, 0, s>>>(m->st);
  LOC_LAUNCHED();
  const int64_t spe = cdiv(m->n_train, m->B);
  for (int e = 0; e < n_epochs; ++e) {
    bool have_fwd = false;  // the previous step's backward already left this step's Z1 partial tiles
    if (run_span(m, d_perms, m->n_train, 0, spe, 1, &have_fwd, s)) return 1;
    if (end_epoch(m, s)) return 1;
  }
  return 0;
}

int loc_train_steps(loc_model* m, const int32_t* d_perm, int32_t step0, int32_t n_steps, void* stream) {
  LOC_CHECK(m != nullptr && m->train_packed != nullptr, "loc_train_steps: no training data bound");
  const int64_t spe = m != nullptr ? cdiv(m->n_train, m->B) : 0;
  LOC_CHECK(d_perm != nullptr && step0 >= 0 && n_steps >= 1 && (int64_t)step0 + n_steps <= spe,
            "loc_train_steps: the span must lie inside one epoch");
  const bool ends_epoch = (int64_t)step0 + n_steps == spe;
  LOC_CHECK(!ends_epoch || m->val_packed != nullptr, "loc_train_steps: a span that ends the epoch needs validation data");
  cudaStream_t s = (cudaStream_t)stream;
  // continuing the span of the previous call: its last backward already ran this span's first forward
  bool have_fwd = step0 > 0 && m->span_perm == d_perm && m->span_next == step0;
  m->span_perm = nullptr;
  if (run_span(m, d_perm, 0, step0, n_steps, 0, &have_fwd, s)) return 1;
  if (ends_epoch) return end_epoch(m, s);
  if (have_fwd) {
    m->span_perm = d_perm;
    m->span_next = (int64_t)step0 + n_steps;
  }
  return 0;
}

int loc_eval(loc_model* m, const uint32_t* d_packed, int64_t n, int64_t row_words, const float* d_locs, float* h_loss,
             void* stream) {
  LOC_CHECK(m != nullptr && d_packed != nullptr && d_locs != nullptr && h_loss != nullptr && n > 0,
            "loc_eval: bad arguments");
  LOC_CHECK(row_words >= cdiv(m->K, 16), "loc_eval: row_words too small for K");
  cudaStream_t s = (cudaStream_t)stream;
  k_zero_val<<<1, 1, 0, s>>>(m->st);
  LOC_LAUNCHED();
  if (infer_rows(m, d_packed, n, row_words, d_locs, nullptr, 0, s)) return 1;
  DevState h;
  LOC_CUDA(cudaMemcpyAsync(&h, m->st, sizeof(h), cudaMemcpyDeviceToHost, s));
  k_zero_val<<<1, 1, 0, s>>>(m->st);
  LOC_LAUNCHED();
  LOC_CUDA(cudaStreamSynchronize(s));
  *h_loss = h.val_total / h.val_count;
  return 0;
}

int loc_predict(loc_model* m, const uint32_t* d_packed, int64_t n, int64_t row_words, float* d_out, void* stream) {
  LOC_CHECK(m != nullptr && d_out != nullptr, "loc_predict: bad arguments");
  if (n <= 0) return 0;
  LOC_CHECK(d_packed != nullptr && row_words >= cdiv(m->K, 16), "loc_predict: bad matrix");
  return infer_rows(m, d_packed, n, row_words, nullptr, d_out, 0, (cudaStream_t)stream);
}

int loc_restore_best(loc_model* m, void* stream) {
  LOC_CHECK(m != nullptr, "loc_restore_best: null model");
  DevState h;
  LOC_CUDA(cudaMemcpyAsync(&h, m->st, sizeof(h), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  LOC_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  LOC_CHECK(h.best_epoch >= 0, "loc_restore_best: no checkpoint has been taken");
  if (copy_weights(m, false, nullptr, (cudaStream_t)stream)) return 1;
  return reslice(m, (cudaStream_t)stream);
}

int loc_snapshot(loc_model* m, void* stream) {
  LOC_CHECK(m != nullptr, "loc_snapshot: null model");
  return copy_weights(m, true, nullptr, (cudaStream_t)stream);
}

int loc_model_state(loc_model* m, loc_state* h_out, void* stream) {
  LOC_CHECK(m != nullptr && h_out != nullptr, "loc_model_state: bad arguments");
  DevState h;
  LOC_CUDA(cudaMemcpyAsync(&h, m->st, sizeof(h), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  LOC_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  h_out->t = h.t;
  h_out->epoch = h.epoch;
  h_out->stopped = h.stopped;
  h_out->improved = h.improved;
  h_out->best_epoch = h.best_epoch;
  h_out->es_wait = h.es_wait;
  h_out->rlr_wait = h.rlr_wait;
  h_out->nonfinite = h.nonfinite;
  LOC_CHECK(h.chain_timeout == 0,
            "loc_model_state: a kernel of a chained training step timed out waiting for its producer (device flags "
            "hid_seq / bwd_cnt / upd_cnt / dz_cnt); results of this model are invalid -- LOC_NO_CHAIN=1 disables chaining");
  h_out->lr = h.lr;
  h_out->ckpt_best = h.ckpt_best;
  h_out->last_loss = h.last_loss;
  h_out->last_val_loss = h.last_val;
  return 0;
}

int loc_model_history(loc_model* m, float* h_out, int32_t max_rows, void* stream) {
  LOC_CHECK(m != nullptr && h_out != nullptr && max_rows >= 0, "loc_model_history: bad arguments");
  const int rows = max_rows < m->max_epochs ? max_rows : m->max_epochs;
  if (rows == 0) return 0;
  LOC_CUDA(cudaMemcpyAsync(h_out, m->hist, (size_t)rows * 3 * sizeof(float), cudaMemcpyDeviceToHost,
                           (cudaStream_t)stream));
  LOC_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return 0;
}

}  // extern "C"
