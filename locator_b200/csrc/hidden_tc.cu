// The 256-wide stack on the 5th-generation tensor cores: one 16-CTA cluster per step, split
// 4 batch groups x 4 column groups.
//
// Reference: load_network locator/locator.py:311-327, model.fit :367-376 (same math as hidden.cu,
// which remains the exact-fp32 CUDA-core variant and the path for other widths).
//
// CTA (rb, cj) owns batch rows [8 rb, 8 rb + 8) and columns [64 cj, 64 cj + 64) of every layer:
//   forward   D[j, b] = sum_k W_i[k, 64cj + j] * a[b, k]      M = 64, N = 8, K = 256 (32 MMAs)
//   backward  D[i, b] = sum_j W_i[64cj + i, j] * dz[b, j]     M = 64, N = 8, K = 256
// Batch rows never mix, so the all-gather after a layer only runs inside a batch group: a CTA
// sends its [8 x 64] slice (2 KB, already in the K-major swizzled B-operand image) to the 4 CTAs
// of its group with shared::cta -> shared::cluster bulk copies completing on their mbarriers --
// 6x less DSMEM traffic than a column-only split.  Weight slices are kept in HBM as ready-made
// operand images (forward: MN-major 128B/32B-atom swizzle; backward: K-major 128B swizzle) and
// stream into a 2-slot ring with cp.async.bulk one layer ahead.  Operands are TF32 (activations
// rounded to nearest, weights as stored), accumulation fp32 in TMEM -- the numerics TensorFlow
// uses for these matmuls on Ampere+ GPUs; elu / dropout / loss / elu' run in fp32 on exact values.
#include "model.cuh"
#include "philox.cuh"
#include "hidden_slices.cuh"

namespace loc {
namespace htc {

constexpr int kH = 256, kC = kHidTcCtas, kRB = 8, kCW = 64;
constexpr int kThreads = 512;
constexpr int kSlot = kH * kCW * 4;    // 64 KB weight-slice image
constexpr int kGath = kRB * kH * 4;    // 8 KB gathered B operand: [8 k-atoms][8 rows][128 B]
constexpr int kStage = kRB * kCW * 4;  // 2 KB own slice: 2 k-atoms

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ unsigned cluster_rank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_barrier() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | ((uint64_t)1 << 46) | ((uint64_t)layout << 61);
}
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn, int b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d),
      "l"(a), "l"(b), "r"(idesc), "r"(acc)
      : "memory");
}
// One lane of a converged warp (elect.sync): the compiler then emits the uniform-datapath
// tcgen05 instructions directly instead of a per-active-lane loop around each of them.
__device__ __forceinline__ bool elect_one() {
  uint32_t p;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(p));
  return p != 0;
}
__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
// byte offset of element (row b, k) inside a K-major 128B-swizzled operand of 8 rows
__device__ __forceinline__ uint32_t b_off(int b, int k) {
  return (uint32_t)((k >> 5) * 1024 + b * 128 + ((((k & 31) >> 2) ^ b) << 4) + ((k & 3) << 2));
}

__device__ __forceinline__ void hidden_tc_body(const HidArgs& a) {
  // programmatic dependent launch: once the whole cluster is running, a kernel queued behind this one with the
  // programmatic-serialization attribute may start (ring schedule of loc_group_train_epochs: ANOTHER model's
  // first-layer backward fills the other SMs while this latency-bound stack runs)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (a.gated && a.st->stopped) {  // past the stopping epoch: a no-op that still keeps the hand-over flag in step
    if (a.training && threadIdx.x == 0 && cluster_rank() == 0) a.st->hid_seq = a.hid_seq;
    if (a.training && threadIdx.x >= 1 && (int)threadIdx.x < a.L) atomicAdd(&a.st->dz_cnt[threadIdx.x], 1u);
    return;
  }
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ int64_t s_rows[kRB];
  __shared__ __align__(8) uint64_t wbar[2], ready[2], mma_bar;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int L = a.L;
  const int r = (int)cluster_rank(), rb = r >> 2, cj = r & 3;
  const int j0 = cj * kCW, b0 = rb * kRB;
  const int nb = a.src.nb;
  const int loss_rows = a.loss_rows > 0 ? a.loss_rows : nb;  // steps of more than 32 rows come in 32-row chunks (bigbatch.cu)
  const int mask_rows = a.mask_rows > 0 ? a.mask_rows : kMaxB;
  const SmallLayout sl{kH, L};
  if (tid == 0 && (r == 0 || r == kC - 1)) tl_mark(a.tl, r ? 19u : 3u, (unsigned)a.tl_id);
  int dbg_n = 0;
  auto mark = [&]() {
    if (a.dbg != nullptr && tid == 0 && dbg_n < 256) a.dbg[r * 256 + dbg_n++] = clock64();
  };
  mark();

  uint8_t* wslot = sm;                                   // [2][64 KB]
  uint8_t* gath = wslot + 2 * kSlot;                     // [2][8 KB]
  uint8_t* stage = gath + 2 * kGath;                     // [2][2 KB]
  float* zbuf = (float*)(stage + 2 * kStage);            // [8][64] accumulator dump
  float* red = zbuf + kRB * kCW;                         // [4][8][64] split-K partial groups
  float* own_a = red + 4 * kRB * kCW;                    // [L][8][64] elu outputs (pre-dropout, fp32)
  float* own_dz = own_a + L * kRB * kCW;                 // [L][8][64]
  float* keep = own_dz + L * kRB * kCW;                  // [8][64]
  float* sbias = keep + kRB * kCW;                       // [L][64]
  float* sout = sbias + L * kCW;                         // Wo1[256][2], bo1[2], Wo2[4], bo2[2]
  float* ysm = sout + 520;                               // y1[8][2], y2[8][2], dy1[8][2], dy2[8][2], dist[8]
  float* y1s = ysm, *y2s = ysm + 16, *dy1s = ysm + 32, *dy2s = ysm + 48, *dist = ysm + 64;

  const int n_uses = a.training ? 2 * (L - 1) : (L - 1);
  auto issue_load = [&](int u) {  // thread 0: weight-slice image of use u -> slot u & 1
    const int layer = u < L - 1 ? u + 1 : 2 * (L - 1) - u;
    const float* src = (u < L - 1 ? a.w_fs : a.w_bs) + (int64_t)(layer - 1) * kH * kH + (int64_t)cj * kH * kCW;
    mbar_expect_tx(&wbar[u & 1], kSlot);
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(wslot + (u & 1) * kSlot)),
                 "l"(src), "r"((uint32_t)kSlot), "r"(smem_u32(&wbar[u & 1]))
                 : "memory");
  };
  // Launched with programmatic stream serialization (train_step's chain, the replicate rings): the results of the
  // kernels in front of it in the stream are complete after this wait.  A no-op for plain launches.
  // It is left out when both producers are named by flags -- wait_upd for the small-layer update (the weight-slice
  // images and biases read below), wait_bwd for the backward's Z1 tiles, each published behind a fence -- as in a
  // chained single-model step: the grid-level wait also covers the backward's completion as a GRID, several
  // microseconds after its last CTA has signed off.
  if (!(a.wait_bwd != 0 && a.wait_upd != 0)) asm volatile("griddepcontrol.wait;" ::: "memory");
  __shared__ int s_dz_done;  // lowest layer whose dz this CTA has written completely (backward chain)
  if (a.wait_upd != 0) {  // the small-layer update of the previous step ran under that step's hidden stack
    if (tid == 0) wait_counter(&a.st->upd_cnt, a.wait_upd, &a.st->chain_timeout, 20u);
    __syncthreads();
  }
  if (tid == 0) {
    s_dz_done = a.L;
    mbar_init(&wbar[0], 1);
    mbar_init(&wbar[1], 1);
    mbar_init(&ready[0], 1);
    mbar_init(&ready[1], 1);
    mbar_init(&mma_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int u = 0; u < 2 && u < n_uses; ++u) issue_load(u);
  }
  // Cluster start-up barrier, split: arrive now (this CTA is running and -- thread 0, in program order -- its
  // mbarriers are initialised), wait just before the first write into a peer's shared memory, so the skew
  // between the CTAs' start times hides under the split-K partial loads below
  __syncwarp();
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(32u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // set-up loads go out first (registers), the split-K partial sums next, the shared-memory writes
  // last: all of the prologue's global-memory latency overlaps
  float r_bias[2], r_out[2];
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int i = tid + q * kThreads;
    r_bias[q] = i < L * kCW ? a.small[((i / kCW) == 0 ? sl.b1() : sl.bh(i / kCW)) + j0 + (i % kCW)] : 0.f;
    r_out[q] = i < 2 * kH + 8 ? a.small[sl.Wo1() + i] : 0.f;
  }
  const int64_t r_row = (tid < kRB && (b0 + tid) < nb) ? row_of(a.src, a.st, b0 + tid) : 0;
  const int step_id = a.st->step_id;
  // Optimizer bookkeeping of this step (Keras Adam: alpha from t >= 1), computed now by the thread that will
  // publish it, off the critical path: the two powf cost about a microsecond at the very end otherwise.
  __shared__ float s_alpha_next;
  __shared__ int s_t_next;
  if (a.training && tid == kThreads - 1 && r == 0) {  // a thread nobody waits for before the kernel's last barrier
    const int t_next = a.st->t + 1;
    const float b1p = powf(kAdamB1, (float)t_next), b2p = powf(kAdamB2, (float)t_next);
    s_t_next = t_next;
    s_alpha_next = a.st->lr * sqrtf(1.f - b2p) / (1.f - b1p);
  }
  const float keep_scale = 1.0f / (1.0f - a.p_drop);
  const bool drop_on = a.training && a.p_drop > 0.f;
  // ---- layer 0, first half: split-K partial tiles of Z1 for the own [8 x 64] block (fixed order).
  //      Issued before the rest of the prologue so that barrier / TMEM / bias set-up and the
  //      cluster start-up barrier run in the shadow of these L2 reads. ----
  if (a.wait_flags != nullptr) {
    // sharded model: the tiles are pushed by the peers over NVLink; one thread per (sender, block) flag
    // polls the local flags (acquire.sys), the barrier orders everybody's loads behind them.  A peer that
    // never arrives is reported after ~2 s instead of hanging the GPU.
    if (tid < a.wait_count) {
      const long long t0 = clock64();
      const uint32_t* f = a.wait_flags + tid;
      while (true) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
        if ((int32_t)(v - a.wait_seq) >= 0) break;
        if (clock64() - t0 > 4000000000ll) {
          *a.wait_err = 1;
          break;
        }
      }
    }
    __syncthreads();
  }
  if (a.wait_bwd != 0) {
    // launched ahead of the first-layer backward whose fused forward leaves this step's Z1 partial tiles: every
    // CTA of that kernel bumps DevState::bwd_cnt once all it wrote is visible
    if (tid == 0) wait_counter(&a.st->bwd_cnt, a.wait_bwd, &a.st->chain_timeout, 20u);  // 16 pollers in all: poll tightly
    __syncthreads();
    if (tid == 0 && r == 0) tl_mark(a.tl, 23u, (unsigned)a.tl_id);  // the backward's tiles are there
  }
  if (a.training && r == 0 && tid == kThreads - 1) {
    // Nothing reads the previous step's alpha any more (its backward and update are complete: waited for above or
    // ordered by the stream): this step's value goes out now, for the update blocks that start under this kernel.
    a.st->alpha = s_alpha_next;
  }
  const int p0_item = tid & 127, p0_g = tid >> 7;  // 128 float4 outputs x 4 partial groups
  const int p0_b = p0_item >> 4, p0_jl = (p0_item & 15) * 4;
  float4 p0_s = make_float4(0.f, 0.f, 0.f, 0.f);
  {
    const int pbeg = a.n_partials * p0_g / 4, pend = a.n_partials * (p0_g + 1) / 4;
    const float4* src =
        reinterpret_cast<const float4*>(a.partials + (int64_t)(a.partial_row0 + b0 + p0_b) * kH + j0 + p0_jl);
    const int64_t pstride = a.partial_stride >> 2;  // float4 units between partial tiles
#pragma unroll 16
    for (int p = pbeg; p < pend; ++p) {
      const float4 v = __ldcg(src + (int64_t)p * pstride);
      p0_s.x += v.x;
      p0_s.y += v.y;
      p0_s.z += v.z;
      p0_s.w += v.w;
    }
  }
  mark();

#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int i = tid + q * kThreads;
    if (i < L * kCW) sbias[i] = r_bias[q];
    if (i < 2 * kH + 8) sout[i] = r_out[q];
  }
  if (tid < kRB) s_rows[tid] = r_row;
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_slot;
  mark();

  int pub = 0;   // publishes so far: publish n uses stage / gathered buffer n & 1
  int nmma = 0;  // MMA batches so far (parity of mma_bar)
  // All-gather inside the batch group: the staged [8 x 64] slice goes to the 4 CTAs (rb, 0..3).
  auto publish_staged = [&]() {
    mark();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    mark();
    if (lane == 0 && warp < 4) {
      const uint32_t src = smem_u32(stage + (pub & 1) * kStage);
      const uint32_t dst_local = smem_u32(gath + (pub & 1) * kGath + cj * kStage);
      const uint32_t bar_local = smem_u32(&ready[pub & 1]);
      const unsigned dest = (unsigned)(rb * 4 + warp);
      uint32_t dst, bar;
      asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(dst) : "r"(dst_local), "r"(dest));
      asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(bar) : "r"(bar_local), "r"(dest));
      asm volatile(
          "cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
          "r"(src), "r"((uint32_t)kStage), "r"(bar)
          : "memory");
    }
    ++pub;
  };
  auto wait_gather = [&](int n) -> const uint8_t* {
    if (tid == 0) mbar_expect_tx(&ready[n & 1], 4 * kStage);
    mbar_wait(&ready[n & 1], (uint32_t)(n >> 1) & 1u);
    return gath + (n & 1) * kGath;
  };
  // One layer product on the tensor core: D[64 x 8] (TMEM) = A (weight-slice image) x B (gathered).
  // Only the four worker warps (tid < 128) run the layer chain: warp 0 waits for the operands and issues, all four
  // read the accumulator (row m lives in TMEM lane 32*(m/16) + m%16: lanes 0-15 of each warp's quarter hold
  // 16 columns x 8 batch rows) and hand rows 4-7 to lanes 16-31, so that every worker thread finishes
  // z[b][jl] for jl = w_jl, b = w_b0 .. w_b0 + 3 straight from registers -- no shared-memory round trip and no
  // block-wide barrier inside the chain.  The other warps sleep at the __syncthreads() behind the chain.
  const int w_jl = 16 * warp + (lane & 15), w_b0 = 4 * (lane >> 4);
  auto layer_mma = [&](int u, bool backward, float (&z)[4]) {
    if (warp == 0) {
      const uint8_t* B = wait_gather(pub - 1);
      mark();
      mbar_wait(&wbar[u & 1], (uint32_t)(u >> 1) & 1u);
      mark();
      if (elect_one()) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t wb = smem_u32(wslot + (u & 1) * kSlot), bb = smem_u32(B);
        // base descriptors once per layer; the 32 K-steps only add compile-time constants to the
        // 14-bit start-address field (a single thread issues: keep its instruction stream short).
        // Four accumulators (TMEM columns 0-7, 8-15, 16-23, 24-31) take every 4th K-step so that
        // consecutive MMAs do not wait on each other's accumulate; the epilogue adds them.
        const uint64_t b0d = smem_desc(bb, 16, 1024, 2);
        if (!backward) {  // A: MN-major [2 j-chunks][256 k rows][128 B], 32B-atom swizzle; 8 k rows = 1024 B per step
          const uint64_t a0d = smem_desc(wb, kH * 128, 512, 1);
          constexpr uint32_t idesc = make_idesc(64, 8, 1, 0);
#pragma unroll
          for (int ks = 0; ks < kH / 8; ++ks)
            umma_tf32(tmem + (uint32_t)((ks & 3) * 8), a0d + (uint64_t)(ks * 64),
                      b0d + (uint64_t)((ks >> 2) * 64 + (ks & 3) * 2), idesc, ks >= 4 ? 1u : 0u);
        } else {          // A: K-major [8 k-chunks][8 row groups][8 rows][128 B], 128B swizzle
          const uint64_t a0d = smem_desc(wb, 16, 1024, 2);
          constexpr uint32_t idesc = make_idesc(64, 8, 0, 0);
#pragma unroll
          for (int ks = 0; ks < kH / 8; ++ks)
            umma_tf32(tmem + (uint32_t)((ks & 3) * 8), a0d + (uint64_t)((ks >> 2) * 512 + (ks & 3) * 2),
                      b0d + (uint64_t)((ks >> 2) * 64 + (ks & 3) * 2), idesc, ks >= 4 ? 1u : 0u);
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&mma_bar))
                     : "memory");
      }
      __syncwarp();
    }
    mbar_wait(&mma_bar, (uint32_t)nmma & 1u);
    mark();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (tid == 0 && u + 2 < n_uses) issue_load(u + 2);  // the slot is free: prefetch two uses ahead
    uint32_t v[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(tmem + ((uint32_t)(32 * warp) << 16))
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");  // the next layer's MMAs overwrite these columns
    float s8[8];
#pragma unroll
    for (int b = 0; b < kRB; ++b)
      s8[b] = (__uint_as_float(v[b]) + __uint_as_float(v[8 + b])) + (__uint_as_float(v[16 + b]) + __uint_as_float(v[24 + b]));
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float hi = __shfl_sync(0xffffffffu, s8[4 + i], lane & 15);  // rows 4..7 go to lanes 16..31
      z[i] = lane < 16 ? s8[i] : hi;
    }
    mark();
  };
  // worker warps: the own [8 x 64] slice is staged -> to the 4 CTAs of the batch group
  auto publish_workers = [&](int dz_layer_done = -1) {
    mark();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("bar.sync 1, 128;" ::: "memory");
    mark();
    // backward chain: every worker's dz of this layer is in global memory -- tell the signalling warp
    if (dz_layer_done >= 0 && tid == 0)
      asm volatile("st.release.cta.shared.s32 [%0], %1;" ::"r"(smem_u32(&s_dz_done)), "r"(dz_layer_done) : "memory");
    if (lane == 0) {
      const uint32_t src = smem_u32(stage + (pub & 1) * kStage);
      const uint32_t dst_local = smem_u32(gath + (pub & 1) * kGath + cj * kStage);
      const uint32_t bar_local = smem_u32(&ready[pub & 1]);
      const unsigned dest = (unsigned)(rb * 4 + warp);
      uint32_t dst, bar;
      asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(dst) : "r"(dst_local), "r"(dest));
      asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(bar) : "r"(bar_local), "r"(dest));
      asm volatile(
          "cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
          "r"(src), "r"((uint32_t)kStage), "r"(bar)
          : "memory");
    }
  };
  auto stage_store = [&](int b, int jl, float v) {
    *reinterpret_cast<float*>(stage + (pub & 1) * kStage + b_off(b, jl)) = to_tf32(v);
  };
  // dropout multiplier of element (row b, column jl) of the layer in front of the Dropout (1 when dropout is off)
  auto drop_mult = [&](int b, int jl) -> float {
    if (!drop_on) return 1.f;
    bool kp;
    if (a.masks != nullptr) {
      const int64_t s = step_id < a.n_masks ? step_id : a.n_masks - 1;
      kp = a.masks[(s * mask_rows + a.row_base + b0 + b) * kH + j0 + jl] != 0;
    } else {
      kp = philox_uniform((uint64_t)(a.row_base + b0 + b) * kH + j0 + jl, kDropoutStreamBase + (uint32_t)step_id, a.seed) >=
           a.p_drop;
    }
    return kp ? keep_scale : 0.f;
  };
  auto finish_fwd_elem = [&](int i, int b, int jl, float z) {
    float act = elu_fast(z + sbias[i * kCW + jl]);
    own_a[(i * kRB + b) * kCW + jl] = act;
    if (i == a.n_before - 1) {
      const float mult = drop_mult(b, jl);
      act *= mult;
      keep[b * kCW + jl] = mult;
    }
    const float out = (b0 + b) < nb ? act : 0.f;
    stage_store(b, jl, out);
    // the update kernels read the (dropout-scaled) activations from global memory: store them now,
    // off the critical path, instead of in a loop at the end of the kernel
    if (a.training) a.acts[((int64_t)i * kMaxB + b0 + b) * kH + j0 + jl] = out;
  };
  // the same for rows bq .. bq + 3 of one column (worker threads of the layer chain): the four elu chains are
  // independent, every load comes before every store
  auto finish_fwd4 = [&](int i, int bq, int jl, const float (&z)[4]) {
    const float bias = sbias[i * kCW + jl];
    float act[4], out[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) act[e] = elu_fast(z[e] + bias);
#pragma unroll
    for (int e = 0; e < 4; ++e) own_a[(i * kRB + bq + e) * kCW + jl] = act[e];
    if (i == a.n_before - 1) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float mult = drop_mult(bq + e, jl);
        act[e] *= mult;
        keep[(bq + e) * kCW + jl] = mult;
      }
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      out[e] = (b0 + bq + e) < nb ? act[e] : 0.f;
      stage_store(bq + e, jl, out[e]);
    }
    if (a.training) {
#pragma unroll
      for (int e = 0; e < 4; ++e) a.acts[((int64_t)i * kMaxB + b0 + bq + e) * kH + j0 + jl] = out[e];
    }
  };
  auto finish_bwd_elem = [&](int i, int b, int jl, float da) {
    if (i == a.n_before - 1) da *= keep[b * kCW + jl];
    const float dz = (b0 + b) < nb ? da * elu_grad_from_out(own_a[(i * kRB + b) * kCW + jl]) : 0.f;
    stage_store(b, jl, dz);
    a.dzs[((int64_t)i * kMaxB + b0 + b) * kH + j0 + jl] = dz;
  };
  auto finish_bwd4 = [&](int i, int bq, int jl, const float (&da)[4]) {
    float g[4], dz[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      g[e] = elu_grad_from_out(own_a[(i * kRB + bq + e) * kCW + jl]);
      if (i == a.n_before - 1) g[e] *= keep[(bq + e) * kCW + jl];
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      dz[e] = (b0 + bq + e) < nb ? da[e] * g[e] : 0.f;
      stage_store(bq + e, jl, dz[e]);
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) a.dzs[((int64_t)i * kMaxB + b0 + bq + e) * kH + j0 + jl] = dz[e];
  };

  // ---- layer 0: finish the split-K reduction started in the prologue ----
  {
    *reinterpret_cast<float4*>(red + (p0_g * kRB + p0_b) * kCW + p0_jl) = p0_s;
    __syncthreads();
    mark();
    for (int idx = tid; idx < kRB * kCW; idx += kThreads) {
      const int bb = idx / kCW, jj = idx % kCW;
      const float z = (red[bb * kCW + jj] + red[(kRB + bb) * kCW + jj]) +
                      (red[(2 * kRB + bb) * kCW + jj] + red[(3 * kRB + bb) * kCW + jj]);
      finish_fwd_elem(0, bb, jj, z);
    }
    mark();
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");  // every CTA of the cluster is running
    publish_staged();
    mark();
  }

  // ---- layers 1..L-1 forward ----
  int use = 0;
  for (int i = 1; i < L; ++i, ++use) {
    if (warp < 4) {
      float z[4];
      layer_mma(use, false, z);
      finish_fwd4(i, w_b0, w_jl, z);
      publish_workers();
    }
    ++pub;
    ++nmma;
  }
  __syncthreads();  // the other warps rejoin: everything the chain left in shared memory is visible to them

  // ---- Dense(2), Dense(2), loss for the own 8 rows (the 4 CTAs of a batch group agree) ----
  const uint8_t* gat = wait_gather(pub - 1);  // a_{L-1} of the own rows (tf32-rounded)
  if (warp < kRB) {
    const int b = warp;  // one warp per row
    float s0 = 0.f, s1 = 0.f;
    for (int k = lane; k < kH; k += 32) {
      const float av = *reinterpret_cast<const float*>(gat + b_off(b, k));
      s0 = fmaf(av, sout[2 * k], s0);
      s1 = fmaf(av, sout[2 * k + 1], s1);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s0 += __shfl_xor_sync(0xffffffffu, s0, o);
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    }
    if (lane == 0) {
      y1s[2 * b] = s0;
      y1s[2 * b + 1] = s1;
    }
  }
  __syncthreads();
  if (tid < kRB) {
    const int b = tid, gb = b0 + b;
    const float* bo1 = sout + 2 * kH;
    const float* Wo2 = bo1 + 2;
    const float* bo2 = Wo2 + 4;
    const float u0 = y1s[2 * b] + bo1[0], u1 = y1s[2 * b + 1] + bo1[1];
    const float v0 = u0 * Wo2[0] + u1 * Wo2[2] + bo2[0];
    const float v1 = u0 * Wo2[1] + u1 * Wo2[3] + bo2[1];
    float d = 0.f, g0 = 0.f, g1 = 0.f;
    if (gb < nb && (a.training || a.has_targets)) {
      const float t0 = a.locs[2 * s_rows[b]], t1 = a.locs[2 * s_rows[b] + 1];
      const float e0 = v0 - t0, e1 = v1 - t1;
      d = sqrtf(e0 * e0 + e1 * e1);
      const float den = d * (float)loss_rows;  // no epsilon: NaN when the prediction hits the target, as in the reference
      g0 = e0 / den;
      g1 = e1 / den;
    }
    const float h0 = g0 * Wo2[0] + g1 * Wo2[1], h1 = g0 * Wo2[2] + g1 * Wo2[3];
    dy1s[2 * b] = h0;
    dy1s[2 * b + 1] = h1;
    if (cj == 0) {  // one CTA per batch group publishes the rows' results
      if (a.write_pred && gb < nb) {
        a.pred_out[2 * s_rows[b]] = v0;
        a.pred_out[2 * s_rows[b] + 1] = v1;
      }
      a.outs[2 * gb] = u0;
      a.outs[2 * gb + 1] = u1;
      a.outs[64 + 2 * gb] = h0;
      a.outs[64 + 2 * gb + 1] = h1;
      a.outs[128 + 2 * gb] = g0;
      a.outs[128 + 2 * gb + 1] = g1;
      a.outs[192 + gb] = d;  // per-row distance, summed by rank 0 after the closing cluster barrier
    }
  }
  __syncthreads();

  if (a.training) {
    // ---- backward: d loss / d a_{L-1} through Dense(2), then the chain of W^T products ----
    for (int idx = tid; idx < kRB * kCW; idx += kThreads) {
      const int b = idx / kCW, jl = idx % kCW, i = j0 + jl;
      finish_bwd_elem(L - 1, b, jl, dy1s[2 * b] * sout[2 * i] + dy1s[2 * b + 1] * sout[2 * i + 1]);
    }
    publish_staged();
    // Warp 4 hands finished layers to the small-layer update, which may already be resident on other SMs
    // (UpdArgs::wait_dz): dz of layer L-1 is complete here (block-wide barrier in publish_staged above); the chain
    // below reports further layers through s_dz_done.  The fence + atomic stay off the worker warps' chain.
    if (warp == 4) {
      int next = L - 1;  // highest layer not signalled yet
      int done = L - 1;
      while (next >= 1) {
        if (done <= next) {
          if (lane == 0) {
            __threadfence();
            for (int k = next; k >= done; --k) atomicAdd(&a.st->dz_cnt[k], 1u);
          }
          next = done - 1;
          if (next < 1) break;
        }
        int d;
        asm volatile("ld.acquire.cta.shared.s32 %0, [%1];" : "=r"(d) : "r"(smem_u32(&s_dz_done)) : "memory");
        done = d < done ? d : done;
        if (done > next) __nanosleep(100);
      }
    }
    for (int i = L - 1; i >= 1; --i, ++use) {
      if (warp < 4) {
        float z[4];
        layer_mma(use, true, z);
        finish_bwd4(i - 1, w_b0, w_jl, z);
        if (i > 1) publish_workers(i - 1);
      }
      if (i > 1) ++pub;
      ++nmma;
    }
    __syncthreads();
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  cluster_barrier();  // nobody exits while peers may still address its shared memory; global writes visible
  if (a.training && r == 0 && tid == 0) {
    // Hand-over first: the kernels launched ahead of this one's end (first-layer backward, small-layer update) wait
    // for hid_seq.  dz / activations of every CTA were written before the cluster barrier above; the optimizer
    // state they read is written here; the loss bookkeeping below is nobody's input and comes after.
    DevState* st = a.st;
    if (!(a.chunk_flags & 2)) {  // (a chunk of a larger step that is not its last leaves the step counters alone)
      st->t = s_t_next;
      st->step_id = step_id + 1;
    }
    st->alpha = s_alpha_next;
    __threadfence();
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(&st->hid_seq), "r"(a.hid_seq) : "memory");
    tl_mark(a.tl, 24u, (unsigned)a.tl_id);  // published
  }
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(32u) : "memory");
  if (tid == 0 && (r == 0 || r == kC - 1)) tl_mark(a.tl, r ? 20u : 4u, (unsigned)a.tl_id);
  if (r == 0 && warp == 0 && (a.training || a.has_targets)) {
    DevState* st = a.st;
    // per-row distances of all batch groups (written before the barrier): one L2 round trip, fixed-order sum
    float s = lane < nb ? __ldcg(a.outs + 192 + lane) : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
      const float mean = s / (float)nb;
      if (a.training && a.val_slot != nullptr) {  // chunks of a large step side by side: k_bb_step_end adds them in order
        a.val_slot[0] = s;
        a.val_slot[1] = (float)nb;
      } else if (a.training) {
        st->loss_total += mean * (float)nb;
        st->loss_count += (float)nb;
        if (a.loss_rows > 0) {  // chunk of a larger step: the step's loss is the mean over all of its rows
          const float acc = ((a.chunk_flags & 1) ? st->step_sum : 0.f) + s;
          st->step_sum = acc;
          st->last_loss = acc / (float)loss_rows;
        } else {
          st->last_loss = mean;
        }
        if (!isfinite(mean)) st->nonfinite = 1;
      } else if (a.val_slot != nullptr) {  // chunks of a wide pass run concurrently: summed in order afterwards
        a.val_slot[0] = mean * (float)nb;
        a.val_slot[1] = (float)nb;
      } else {
        st->val_total += mean * (float)nb;
        st->val_count += (float)nb;
      }
    }
  }
}

__global__ void __launch_bounds__(kThreads, 1) k_hidden_tc(HidArgs a) { hidden_tc_body(a); }

// Several independent models (replicates) in one launch: cluster c runs model c.  The models' steps
// are issued in lockstep by loc_group_train_epochs, so their latency-bound hidden stacks overlap on
// different SMs instead of each idling 132 of them.
__global__ void __launch_bounds__(kThreads, 1) k_hidden_tc_group(HidGroupArgs g) { hidden_tc_body(g.a[blockIdx.x / kC]); }

__global__ void k_reslice_tc(const float* __restrict__ small, float* fs, float* bs, int L) {
  const SmallLayout sl{kH, L};
  const int64_t n = (int64_t)(L - 1) * kH * kH;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int layer = 1 + (int)(i / (kH * kH));
    const int k = (int)((i / kH) % kH), j = (int)(i % kH);
    store_images(fs, bs, layer, k, j, small[sl.Wh(layer) + (int64_t)k * kH + j]);
  }
}

static size_t smem_bytes(int L) {
  return (size_t)2 * kSlot + 2 * kGath + 2 * kStage +
         sizeof(float) * ((size_t)kRB * kCW * (1 + 4 + 2 * L + 1) + (size_t)L * kCW + 520 + 80) + 1024;
}

}  // namespace htc

static int launch_tc(const HidArgs& a, cudaStream_t s, bool dry, bool overlap_previous = false) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(htc::kC);
  cfg.blockDim = dim3(htc::kThreads);
  cfg.dynamicSmemBytes = htc::smem_bytes(a.L);
  cfg.stream = s;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = htc::kC;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  // overlap_previous: programmatic dependent launch behind this model's small-layer update (train_step's chain):
  // the cluster is placed and set up while the first-layer backward still streams; the kernel itself waits for
  // the update (griddepcontrol.wait) and for the backward's tiles (DevState::bwd_cnt)
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = overlap_previous ? 2 : 1;
  if (dry) {
    int n = 0;
    cfg.numAttrs = 1;
    if (cudaOccupancyMaxActiveClusters(&n, htc::k_hidden_tc, &cfg) != cudaSuccess) {
      cudaGetLastError();
      return 0;
    }
    return n;
  }
  LOC_CUDA(cudaLaunchKernelEx(&cfg, htc::k_hidden_tc, a));
  loc::g_launches.fetch_add(1);
  return 0;
}

int hidden_tc_group_launch(const HidGroupArgs& g, cudaStream_t s) {
  LOC_CHECK(g.n >= 1 && g.n <= kMaxGroup, "hidden stack group: bad group size");
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(htc::kC * g.n);
  cfg.blockDim = dim3(htc::kThreads);
  cfg.dynamicSmemBytes = htc::smem_bytes(g.a[0].L);
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = htc::kC;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(htc::k_hidden_tc_group, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    attr_set = true;
  }
  LOC_CUDA(cudaFuncSetAttribute(htc::k_hidden_tc_group, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cfg.dynamicSmemBytes));
  LOC_CUDA(cudaLaunchKernelEx(&cfg, htc::k_hidden_tc_group, g));
  loc::g_launches.fetch_add(1);
  return 0;
}

bool hidden_tc_supported(int H, int L) {
  if (H != htc::kH || L < 2) return false;
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return false;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (major != 10) return false;
  const size_t smem = htc::smem_bytes(L);
  if (smem > 227 * 1024) return false;
  cudaFuncSetAttribute(htc::k_hidden_tc, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  if (cudaFuncSetAttribute(htc::k_hidden_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  HidArgs dummy = {};
  dummy.L = L;
  return launch_tc(dummy, 0, true) > 0;
}

int hidden_tc_launch(const HidArgs& a, cudaStream_t s, bool overlap_previous) {
  LOC_CHECK(a.H == htc::kH, "hidden stack (tcgen05): width must be 256");
  LOC_CUDA(cudaFuncSetAttribute(htc::k_hidden_tc, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)htc::smem_bytes(a.L)));
  return launch_tc(a, s, false, overlap_previous);
}

int hidden_tc_reslice(const float* small, float* fs, float* bs, int L, cudaStream_t s) {
  if (L < 2) return 0;
  htc::k_reslice_tc<<<148 * 4, 256, 0, s>>>(small, fs, bs, L);
  LOC_LAUNCHED();
  return 0;
}

}  // namespace loc
