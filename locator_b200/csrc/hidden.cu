// The width-H stack behind the first layer: Dense(H,elu) x (L-1) (+Dropout), Dense(2), Dense(2),
// Euclidean-distance loss, and the backward chain down to dZ1 -- one thread-block cluster per step.
//
// Reference: load_network locator/locator.py:311-327 (layers, loss :314-315), model.fit :367-376;
// Keras semantics restated in oracle/model_ref.py (RefLocator.forward / gradients).
//
// Work split: CTA r of the C-CTA cluster owns columns [r*Hc, (r+1)*Hc) of every layer's output.
// The step is a chain of 2L tiny dependent products, so everything is arranged around latency:
//   * weights never wait on L2: each CTA's slice of every layer is kept in HBM in two pre-sliced
//     copies (forward slices W[:, cols] and backward slices W[rows, :]^T, both [H][Hc] contiguous)
//     and streamed into a ring of shared-memory slots with cp.async.bulk + mbarrier several layers
//     ahead of use;
//   * activations never go through L2 on the critical path: a CTA publishes its [32 x Hc] slice
//     straight into the shared memory of all C CTAs with one shared::cta -> shared::cluster bulk
//     copy per destination, whose bytes complete on the receiver's mbarrier (no fence, no
//     cluster-wide barrier per layer), double-buffered;
//   * each slice product splits the reduction dimension over the 16 warps with a fixed-order
//     cross-warp sum (deterministic).
// dW + Adam of these layers is NOT done here: activations and dz of every layer are also left in
// global memory for k_hidden_update, which runs off the critical path.
#include "model.cuh"
#include "philox.cuh"
#include "hidden_slices.cuh"

namespace loc {

__device__ __forceinline__ unsigned cluster_rank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ unsigned cluster_size() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ unsigned cluster_id() {
  unsigned r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return r;
}
// Release/acquire at cluster scope: (distributed) shared-memory and global writes made before it by
// any CTA of the cluster are visible to every CTA after it.
__device__ __forceinline__ void cluster_barrier() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t hid_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// 16-byte store into CTA `rank`'s shared memory whose completion is counted (complete_tx) on that
// CTA's mbarrier: the receiver just waits for the expected byte count of the layer.
__device__ __forceinline__ void st_async_f4(uint32_t local_addr, uint32_t local_bar, unsigned rank, float4 v) {
  uint32_t raddr, rbar;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(raddr) : "r"(local_addr), "r"(rank));
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rbar) : "r"(local_bar), "r"(rank));
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(
                   raddr),
               "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"(rbar)
               : "memory");
}

constexpr int kHidThreads = 512;
constexpr int kHidWarps = kHidThreads / 32;
constexpr int kMaxSlots = 16;

// Gathered activations live slice-major: [source CTA r][batch row b][Hc + pad] so that a source
// CTA's slice is one contiguous block (one bulk copy per destination) and rows of one slice are
// an odd number of 16-byte chunks apart (conflict-free float4 reads across batch rows).
__host__ __device__ inline int hid_row_pitch(int Hc) { return Hc + (((Hc / 4) % 2 == 0) ? 4 : 0); }

__host__ __device__ inline int hid_nparts(int H) {
  const int gpw = (H / 4 + kHidWarps - 1) / kHidWarps;
  return (H / 4 + gpw - 1) / gpw;
}

// Packed fp32 FMA (FFMA2): d.lo += a.lo * b.lo, d.hi += a.hi * b.hi in one issue slot.
__device__ __forceinline__ void ffma2(unsigned long long& d, unsigned long long a, unsigned long long b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(a), "l"(b));
}
__device__ __forceinline__ float sum2(unsigned long long v) {
  return __uint_as_float((uint32_t)v) + __uint_as_float((uint32_t)(v >> 32));
}

// red[w][b][jl] = sum over warp w's share of k of A[b][k] * W[k][jl].
// Ws is the weight slice in shared memory with k pairs interleaved: Ws[k/2][jl][k&1], so that both
// FFMA2 operands -- (A[b][k], A[b][k+1]) and (W[k][jl], W[k+1][jl]) -- are natural 64-bit pairs of
// the 128-bit loads; even and odd k accumulate separately and are added at the end.
template <int TH, int THc>
__device__ __noinline__ void slice_matmul(const float* gathered, const float* Ws, float* red, int rH, int rHc) {
  const int H = TH ? TH : rH, Hc = THc ? THc : rHc;
  const int HcP = hid_row_pitch(Hc), SL = kMaxB * HcP;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // the H/4 four-wide k groups are dealt to the warps in contiguous runs (hid_nparts warps get work)
  const int gpw = (H / 4 + kHidWarps - 1) / kHidWarps;
  const int kbeg = warp * gpw * 4;
  const int kend = (kbeg + gpw * 4) < H ? (kbeg + gpw * 4) : H;
  if (kbeg >= H) return;
  const int jq_n = Hc / 4;
  const int ntile = (kMaxB / 4) * jq_n;
  for (int tile = lane; tile < ntile; tile += 32) {
    const int bq = tile / jq_n, jq = tile % jq_n;  // batch rows bq, bq+8, bq+16, bq+24
    unsigned long long acc[4][4];
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
      for (int y = 0; y < 4; ++y) acc[x][y] = 0ull;
#pragma unroll 4
    for (int k = kbeg; k < kend; k += 4) {
      const float* arow = gathered + (k / Hc) * SL + bq * HcP + (k % Hc);
      const float* wrow = Ws + (k / 2) * (2 * Hc) + 8 * jq;
      ulonglong2 a2[4], w2[4];  // a2[bb] = {(a[k],a[k+1]), (a[k+2],a[k+3])}
#pragma unroll
      for (int bb = 0; bb < 4; ++bb) a2[bb] = *reinterpret_cast<const ulonglong2*>(arow + 8 * bb * HcP);
      // w2[0], w2[1]: k pair 0, columns (0,1), (2,3);  w2[2], w2[3]: k pair 1
      w2[0] = *reinterpret_cast<const ulonglong2*>(wrow);
      w2[1] = *reinterpret_cast<const ulonglong2*>(wrow + 4);
      w2[2] = *reinterpret_cast<const ulonglong2*>(wrow + 2 * Hc);
      w2[3] = *reinterpret_cast<const ulonglong2*>(wrow + 2 * Hc + 4);
#pragma unroll
      for (int bb = 0; bb < 4; ++bb) {
        ffma2(acc[bb][0], a2[bb].x, w2[0].x);
        ffma2(acc[bb][1], a2[bb].x, w2[0].y);
        ffma2(acc[bb][2], a2[bb].x, w2[1].x);
        ffma2(acc[bb][3], a2[bb].x, w2[1].y);
        ffma2(acc[bb][0], a2[bb].y, w2[2].x);
        ffma2(acc[bb][1], a2[bb].y, w2[2].y);
        ffma2(acc[bb][2], a2[bb].y, w2[3].x);
        ffma2(acc[bb][3], a2[bb].y, w2[3].y);
      }
    }
#pragma unroll
    for (int bb = 0; bb < 4; ++bb)
      *reinterpret_cast<float4*>(red + ((int64_t)warp * kMaxB + bq + 8 * bb) * Hc + 4 * jq) =
          make_float4(sum2(acc[bb][0]), sum2(acc[bb][1]), sum2(acc[bb][2]), sum2(acc[bb][3]));
  }
}

// TH / THc: compile-time width and slice width (0 = take them from the arguments): the common
// 256-wide, 16-CTA configuration gets shift-and-mask index arithmetic and fully unrolled loops.
// One launch runs g.n independent models (a single model is a group of one): cluster c runs model c with
// g.a[c], exactly as a launch of that model alone would.  Every model-specific location -- DevState, dropout
// stream, masks, partial tiles, acts / dzs / outs, dbg -- comes from g.a[c], and the CTA's place
// inside its model is its cluster rank, so clusters never touch each other's data or wait on each other.
template <int TH, int THc>
__global__ void __launch_bounds__(kHidThreads, 1) k_hidden(HidGroupArgs g) {
  const HidArgs& a = g.a[cluster_id()];
  if (a.gated && a.st->stopped) return;
  extern __shared__ __align__(16) float smem[];
  __shared__ int64_t s_rows[kMaxB];
  __shared__ __align__(8) uint64_t wbar[kMaxSlots];
  __shared__ __align__(8) uint64_t ready[2];  // gathered-buffer full barriers (bytes from all C CTAs)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int H = TH ? TH : a.H, L = a.L;
  const int C = (TH && THc) ? TH / THc : (int)cluster_size();
  const int r = (int)cluster_rank();
  const int Hc = THc ? THc : H / C, j0 = r * Hc;
  const int HcP = hid_row_pitch(Hc), SL = kMaxB * HcP;
  const int nb = a.src.nb;
  const int loss_rows = a.loss_rows > 0 ? a.loss_rows : nb;  // steps of more than 32 rows come in 32-row chunks (bigbatch.cu)
  const int mask_rows = a.mask_rows > 0 ? a.mask_rows : kMaxB;
  const int NS = a.n_slots;
  const SmallLayout sl{H, L};
  int dbg_n = 0;
  auto mark = [&]() {
    if (a.dbg != nullptr && tid == 0 && dbg_n < 256) a.dbg[r * 256 + dbg_n++] = clock64();
  };
  mark();

  float* full0 = smem;                              // [2][C][32][HcP] gathered activations / dz (double buffer)
  float* stage = full0 + 2 * C * SL;                // [2][32][HcP]    own slice staged for the bulk copies
  float* red = stage + 2 * SL;                      // [16][32][Hc]    per-warp partial sums
  float* own_a = red + kHidWarps * kMaxB * Hc;      // [L][32][Hc] elu outputs (pre-dropout) of the own slice
  float* own_dz = own_a + (int64_t)L * kMaxB * Hc;  // [L][32][Hc] dz of the own slice
  float* keep = own_dz + (int64_t)L * kMaxB * Hc;   // [32][Hc]    dropout multiplier of the own slice
  float* ysm = keep + kMaxB * Hc;                   // y1, y2, dy1, dy2 [32][2] each, dist[32]
  float* sbias = ysm + 320;                         // [L][Hc] own bias slices
  float* sout = sbias + ((L * Hc + 3) & ~3);        // Wo1[H][2], bo1[2], Wo2[4], bo2[2]
  float* wslot = sout + ((2 * H + 8 + 3) & ~3);     // [NS][H][Hc] weight-slice ring
  float* y1s = ysm;
  float* y2s = ysm + 64;
  float* dy1s = ysm + 128;
  float* dy2s = ysm + 192;
  float* dist = ysm + 256;

  // ---- weight-slice ring: uses 0..L-2 are the forward slices of layers 1..L-1, then the backward
  //      slices of layers L-1..1; use u lives in slot u % NS and is fetched NS uses ahead ----
  const int n_uses = a.training ? 2 * (L - 1) : (L - 1);
  const uint32_t slice_bytes = (uint32_t)(H * Hc * sizeof(float));
  auto issue_load = [&](int u) {  // thread 0 only
    const int slot = u % NS;
    const int layer = u < L - 1 ? u + 1 : 2 * (L - 1) - u;
    const float* src = (u < L - 1 ? a.w_fs : a.w_bs) + (int64_t)(layer - 1) * H * H + (int64_t)r * H * Hc;
    const uint32_t bar = hid_smem_u32(&wbar[slot]);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(slice_bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     hid_smem_u32(wslot + (int64_t)slot * H * Hc)),
                 "l"(src), "r"(slice_bytes), "r"(bar)
                 : "memory");
  };
  auto mbar_wait = [&](uint32_t bar, uint32_t parity) {
    uint32_t ok = 0;
    while (!ok) {
      asm volatile(
          "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(ok)
          : "r"(bar), "r"(parity)
          : "memory");
    }
  };
  auto wait_slice = [&](int u) -> const float* {
    mbar_wait(hid_smem_u32(&wbar[u % NS]), (uint32_t)(u / NS) & 1u);
    return wslot + (int64_t)(u % NS) * H * Hc;
  };
  if (tid == 0) {
    for (int s = 0; s < NS; ++s)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(hid_smem_u32(&wbar[s])) : "memory");
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(hid_smem_u32(&ready[0])) : "memory");
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(hid_smem_u32(&ready[1])) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int u = 0; u < NS && u < n_uses; ++u) issue_load(u);
  }
  for (int i = tid; i < L * Hc; i += kHidThreads) {
    const int layer = i / Hc, jl = i % Hc;
    sbias[i] = a.small[(layer == 0 ? sl.b1() : sl.bh(layer)) + j0 + jl];
  }
  for (int i = tid; i < 2 * H + 8; i += kHidThreads) sout[i] = a.small[sl.Wo1() + i];
  if (tid < kMaxB) s_rows[tid] = tid < nb ? row_of(a.src, a.st, tid) : 0;
  const int step_id = a.st->step_id;
  const float keep_scale = 1.0f / (1.0f - a.p_drop);
  const bool drop_on = a.training && a.p_drop > 0.f;
  __syncthreads();
  cluster_barrier();  // every CTA of the cluster is running before anyone writes into its shared memory

  // Finishing passes work on items = (batch row, 4 consecutive columns of the own slice).
  const int items = kMaxB * Hc / 4;
  int pub = 0;  // number of publishes so far: publish n uses stage / gathered buffer n & 1
  // All-gather of the staged own slice: one bulk copy per destination CTA, completing on the
  // destination's mbarrier (the receiver just waits for C slices worth of bytes).
  const uint32_t slice_tx = (uint32_t)(SL * sizeof(float));
  auto publish_staged = [&]() {
    mark();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    mark();
    // one issuing lane per warp: bulk copies are uniform-datapath instructions, lanes of one warp serialise
    for (int d = warp; d < C; d += kHidWarps) {
      if (lane != 0) continue;
      const uint32_t src = hid_smem_u32(stage + (pub & 1) * SL);
      const uint32_t dst_local = hid_smem_u32(full0 + ((pub & 1) * C + r) * SL);
      const uint32_t bar_local = hid_smem_u32(&ready[pub & 1]);
      uint32_t dst, bar;
      asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(dst) : "r"(dst_local), "r"(d));
      asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(bar) : "r"(bar_local), "r"(d));
      asm volatile(
          "cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
          "r"(src), "r"(slice_tx), "r"(bar)
          : "memory");
    }
    ++pub;
  };
  // Wait until publish n (C slices) has landed in this CTA's gathered buffer n & 1.
  auto wait_gather = [&](int n) -> const float* {
    const uint32_t bar = hid_smem_u32(&ready[n & 1]);
    if (tid == 0)
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(slice_tx * (uint32_t)C)
                   : "memory");
    mbar_wait(bar, (uint32_t)(n >> 1) & 1u);
    return full0 + (n & 1) * C * SL;
  };
  // Finishing passes: 4 consecutive lanes share one item (b, 4 columns): each sums a quarter of the
  // per-warp partials, a 2-step shuffle combines them (fixed order), then lane e finishes column e.
  auto red_quad = [&](int nparts, int item, int sub) -> float {
    const int b = (item * 4) / Hc, jl = (item * 4) % Hc;
    float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int w = sub; w < nparts; w += 4) {
      const float4 v = *reinterpret_cast<const float4*>(red + ((int64_t)w * kMaxB + b) * Hc + jl);
      s4.x += v.x;
      s4.y += v.y;
      s4.z += v.z;
      s4.w += v.w;
    }
#pragma unroll
    for (int o = 1; o <= 2; o <<= 1) {
      s4.x += __shfl_xor_sync(0xffffffffu, s4.x, o);
      s4.y += __shfl_xor_sync(0xffffffffu, s4.y, o);
      s4.z += __shfl_xor_sync(0xffffffffu, s4.z, o);
      s4.w += __shfl_xor_sync(0xffffffffu, s4.w, o);
    }
    return sub == 0 ? s4.x : (sub == 1 ? s4.y : (sub == 2 ? s4.z : s4.w));
  };
  const int fin_n = (items * 4 + kHidThreads - 1) / kHidThreads * kHidThreads;  // whole warps stay converged
  // bias, elu, (dropout) of the own slice of layer i from the partial sums in red -> stage
  auto finish_fwd = [&](int i, int nparts, const float* bias) {
    for (int idx = tid; idx < fin_n; idx += kHidThreads) {
      const int item = idx >> 2, e = idx & 3;
      const bool on = item < items;
      const float z = red_quad(nparts, on ? item : 0, e);
      if (!on) continue;
      const int b = (item * 4) / Hc, jl = (item * 4) % Hc + e;
      float act = elu_f(z + bias[jl]);
      own_a[((int64_t)i * kMaxB + b) * Hc + jl] = act;
      if (i == a.n_before - 1) {
        float mult = 1.f;
        if (drop_on) {
          bool kp;
          if (a.masks != nullptr) {
            const int64_t s = step_id < a.n_masks ? step_id : a.n_masks - 1;
            kp = a.masks[(s * mask_rows + a.row_base + b) * H + j0 + jl] != 0;
          } else {
            kp = philox_uniform((uint64_t)(a.row_base + b) * H + j0 + jl, kDropoutStreamBase + (uint32_t)step_id, a.seed) >=
                 a.p_drop;
          }
          mult = kp ? keep_scale : 0.f;
          act *= mult;
        }
        keep[b * Hc + jl] = mult;
      }
      stage[(pub & 1) * SL + b * HcP + jl] = b < nb ? act : 0.f;
    }
    publish_staged();
  };
  // dz of layer i for one element of the own slice from d loss / d (post-dropout activation)
  auto finish_bwd = [&](int i, int b, int jl, float da) {
    if (i == a.n_before - 1) da *= keep[b * Hc + jl];
    const float act = own_a[((int64_t)i * kMaxB + b) * Hc + jl];
    const float dz = b < nb ? da * elu_grad_from_out(act) : 0.f;
    stage[(pub & 1) * SL + b * HcP + jl] = dz;
    own_dz[((int64_t)i * kMaxB + b) * Hc + jl] = dz;
  };

  // ---- layer 0: reduce the split-K partial tiles of Z1 (fixed order), bias, elu ----
  {
    int G = kHidThreads / items;  // thread groups splitting the partial range
    if (G < 1) G = 1;
    if (G > kHidWarps) G = kHidWarps;
    const int hv = H / 4;
    for (int idx = tid; idx < items * G; idx += kHidThreads) {
      const int o = idx % items, g = idx / items;
      const int b = (o * 4) / Hc, jl = (o * 4) % Hc;
      const int pbeg = a.n_partials * g / G, pend = a.n_partials * (g + 1) / G;
      const float4* src = reinterpret_cast<const float4*>(a.partials) + ((int64_t)b * H + j0 + jl) / 4;
      float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
      for (int p = pbeg; p < pend; ++p) {
        const float4 v = __ldcg(src + (int64_t)p * kMaxB * hv);
        s.x += v.x;
        s.y += v.y;
        s.z += v.z;
        s.w += v.w;
      }
      *reinterpret_cast<float4*>(red + ((int64_t)g * kMaxB + b) * Hc + jl) = s;
    }
    __syncthreads();
    mark();
    finish_fwd(0, G, sbias);
    mark();
  }

  // ---- layers 1..L-1 forward ----
  int use = 0;
  for (int i = 1; i < L; ++i, ++use) {
    const float* Ws = wait_slice(use);
    mark();
    const float* in = wait_gather(pub - 1);
    mark();
    slice_matmul<TH, THc>(in, Ws, red, H, Hc);
    __syncthreads();
    mark();
    if (tid == 0 && use + NS < n_uses) issue_load(use + NS);
    finish_fwd(i, hid_nparts(H), sbias + i * Hc);
    mark();
  }

  // ---- Dense(2), Dense(2), loss (every CTA, redundantly) ----
  const float* gat = wait_gather(pub - 1);  // a_{L-1}
  mark();
  {
    const float* Wo1 = sout;
    for (int b = warp; b < kMaxB; b += kHidWarps) {
      float s0 = 0.f, s1 = 0.f;
      for (int k = lane; k < H; k += 32) {
        const float av = gat[(k / Hc) * SL + b * HcP + (k % Hc)];
        s0 = fmaf(av, Wo1[2 * k], s0);
        s1 = fmaf(av, Wo1[2 * k + 1], s1);
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
  }
  __syncthreads();
  if (tid < kMaxB) {
    const int b = tid;
    const float* bo1 = sout + 2 * H;
    const float* Wo2 = bo1 + 2;
    const float* bo2 = Wo2 + 4;
    const float u0 = y1s[2 * b] + bo1[0], u1 = y1s[2 * b + 1] + bo1[1];
    y1s[2 * b] = u0;
    y1s[2 * b + 1] = u1;
    const float v0 = u0 * Wo2[0] + u1 * Wo2[2] + bo2[0];
    const float v1 = u0 * Wo2[1] + u1 * Wo2[3] + bo2[1];
    y2s[2 * b] = v0;
    y2s[2 * b + 1] = v1;
    float d = 0.f, g0 = 0.f, g1 = 0.f;
    if (b < nb && (a.training || a.has_targets)) {
      const float t0 = a.locs[2 * s_rows[b]], t1 = a.locs[2 * s_rows[b] + 1];
      const float e0 = v0 - t0, e1 = v1 - t1;
      d = sqrtf(e0 * e0 + e1 * e1);
      const float den = d * (float)loss_rows;  // no epsilon: NaN when the prediction hits the target, as in the reference
      g0 = e0 / den;
      g1 = e1 / den;
    }
    dist[b] = d;
    dy2s[2 * b] = g0;
    dy2s[2 * b + 1] = g1;
    dy1s[2 * b] = g0 * Wo2[0] + g1 * Wo2[1];
    dy1s[2 * b + 1] = g0 * Wo2[2] + g1 * Wo2[3];
    if (r == 0 && a.write_pred && b < nb) {
      a.pred_out[2 * s_rows[b]] = v0;
      a.pred_out[2 * s_rows[b] + 1] = v1;
    }
  }
  __syncthreads();
  if (r == 0) {
    if (tid < 64) {
      a.outs[tid] = y1s[tid];
      a.outs[64 + tid] = dy1s[tid];
      a.outs[128 + tid] = dy2s[tid];
      a.outs[192 + tid] = y2s[tid];
    }
    if (tid == 0 && (a.training || a.has_targets)) {
      float s = 0.f;
      for (int b = 0; b < nb; ++b) s += dist[b];
      const float mean = s / (float)nb;
      DevState* st = a.st;
      if (a.training) {
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
      } else {
        st->val_total += mean * (float)nb;
        st->val_count += (float)nb;
      }
    }
  }
  if (!a.training) {
    cluster_barrier();  // nobody exits while peers may still address its shared memory
    return;
  }

  // ---- backward: d loss / d a_{L-1} through Dense(2) ----
  {
    const float* Wo1 = sout;
    for (int idx = tid; idx < kMaxB * Hc; idx += kHidThreads) {
      const int b = idx / Hc, jl = idx % Hc;
      const int i = j0 + jl;
      finish_bwd(L - 1, b, jl, dy1s[2 * b] * Wo1[2 * i] + dy1s[2 * b + 1] * Wo1[2 * i + 1]);
    }
    publish_staged();
    mark();
  }
  for (int i = L - 1; i >= 1; --i, ++use) {
    const float* Ws = wait_slice(use);  // [j][il] = W_i[j0 + il][j]
    mark();
    const float* in = wait_gather(pub - 1);
    mark();
    slice_matmul<TH, THc>(in, Ws, red, H, Hc);
    __syncthreads();
    mark();
    if (tid == 0 && use + NS < n_uses) issue_load(use + NS);
    for (int idx = tid; idx < fin_n; idx += kHidThreads) {
      const int item = idx >> 2, e = idx & 3;
      const bool on = item < items;
      const float da = red_quad(hid_nparts(H), on ? item : 0, e);
      if (on) finish_bwd(i - 1, (item * 4) / Hc, (item * 4) % Hc + e, da);
    }
    if (i > 1)
      publish_staged();
    else
      __syncthreads();
    mark();
  }
  // ---- leave activations and dz of every layer in global memory for the update kernels ----
  for (int idx = tid; idx < L * items; idx += kHidThreads) {
    const int i = idx / items, item = idx % items;
    const int b = (item * 4) / Hc, jl = (item * 4) % Hc;
    float4 act = *reinterpret_cast<const float4*>(own_a + ((int64_t)i * kMaxB + b) * Hc + jl);
    if (i == a.n_before - 1) {
      const float4 km = *reinterpret_cast<const float4*>(keep + b * Hc + jl);
      act.x *= km.x;
      act.y *= km.y;
      act.z *= km.z;
      act.w *= km.w;
    }
    if (b >= nb) act = make_float4(0.f, 0.f, 0.f, 0.f);
    *reinterpret_cast<float4*>(a.acts + ((int64_t)i * kMaxB + b) * H + j0 + jl) = act;
    *reinterpret_cast<float4*>(a.dzs + ((int64_t)i * kMaxB + b) * H + j0 + jl) =
        *reinterpret_cast<const float4*>(own_dz + ((int64_t)i * kMaxB + b) * Hc + jl);
  }
  mark();
  cluster_barrier();  // nobody exits while peers may still address its shared memory
  mark();
  // Optimizer bookkeeping for the update kernels of this step (Keras Adam: alpha from t >= 1).
  if (r == 0 && tid == 0 && !(a.chunk_flags & 2)) {
    DevState* st = a.st;
    const int t = st->t + 1;
    st->t = t;
    st->step_id = step_id + 1;
    const float b1p = powf(kAdamB1, (float)t), b2p = powf(kAdamB2, (float)t);
    st->alpha = st->lr * sqrtf(1.f - b2p) / (1.f - b1p);
  }
}

__global__ void k_reslice(const float* __restrict__ small, float* fs, float* bs, int H, int L, int Hc) {
  const SmallLayout sl{H, L};
  const int64_t n = (int64_t)(L - 1) * H * H;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int layer = 1 + (int)(i / ((int64_t)H * H));
    const int k = (int)((i / H) % H), j = (int)(i % H);
    store_sliced(fs, bs, H, Hc, layer, k, j, small[sl.Wh(layer) + (int64_t)k * H + j]);
  }
}

// ---------------------------------------------------------------------------------------------
// dW + Adam of the small layers.  Blocks [0, (L-1)*H/16): 16 input rows x H outputs of hidden
// layer i; last block: b1, Dense(2), Dense(2).  blockDim = H, thread <-> output column j.
// ---------------------------------------------------------------------------------------------
constexpr int kUpdRows = 16;

// (register cap: two 256-thread blocks per SM)
__global__ void __maxnreg__(120) k_hidden_update(UpdArgs a) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the next hidden stack may be scheduled behind us
  if (a.gated && a.st->stopped) {  // past the stopping epoch: a no-op that still keeps the hand-over counter in step
    if (threadIdx.x == 0) atomicAdd(&a.st->upd_cnt, 1u);
    return;
  }
  __shared__ float as[kUpdRows][kMaxB + 1];
  const int H = a.H, L = a.L, j = threadIdx.x;
  const SmallLayout sl{H, L};
  const int rb_n = H / kUpdRows;
  const int nblk_hidden = (L - 1) * rb_n;
  const bool hidden_block = (int)blockIdx.x < nblk_hidden;
  // Weights and Adam moments of the block's 16 rows do not depend on the hidden stack this launch may be waiting
  // for (the previous update wrote them): their loads go out BEFORE the wait, while HBM idles under that stack.
  float w16[kUpdRows], m16[kUpdRows], v16[kUpdRows];
  int64_t row0 = 0;
  if (a.wait_dz != 0 && a.wait_upd != 0) {
    if (threadIdx.x == 0) wait_counter(&a.st->upd_cnt, a.wait_upd, &a.st->chain_timeout);
    __syncthreads();
  }
  if (hidden_block) {
    const int i = 1 + blockIdx.x / rb_n, rb = blockIdx.x % rb_n;
    row0 = sl.Wh(i) + (int64_t)(rb * kUpdRows) * H + j;
#pragma unroll
    for (int r = 0; r < kUpdRows; ++r) {
      const int64_t idx = row0 + (int64_t)r * H;
      w16[r] = a.small[idx];
      m16[r] = a.m_small[idx];
      v16[r] = a.v_small[idx];
    }
  }
  {
    // Launched ahead of the end of the hidden stack whose activations / dz it consumes.  wait_dz: launched UNDER it --
    // the blocks of hidden layer i start as soon as all 16 CTAs of the stack have written dz_i (the stack's backward
    // chain reaches layer i long before it ends); only the last block (b1, Dense(2), Dense(2)) needs its end.
    const int layer = 1 + (int)blockIdx.x / rb_n;
    if (a.wait_dz != 0 && hidden_block) {
      if (threadIdx.x == 0) wait_counter(&a.st->dz_cnt[layer], a.wait_dz, &a.st->chain_timeout);
      __syncthreads();
    } else if (a.wait_hid != 0) {
      if (threadIdx.x == 0) wait_counter(&a.st->hid_seq, a.wait_hid, &a.st->chain_timeout);
      __syncthreads();
    }
  }
  if (threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1)) tl_mark(a.tl, blockIdx.x ? 21u : 5u, (unsigned)a.tl_id);
  const float alpha = a.st->alpha;
  auto adam_at = [&](int64_t idx, float g) -> float {
    float w = a.small[idx], m = a.m_small[idx], v = a.v_small[idx];
    adam_update(w, m, v, g, alpha);
    a.small[idx] = w;
    a.m_small[idx] = m;
    a.v_small[idx] = v;
    return w;
  };
  if ((int)blockIdx.x < nblk_hidden) {
    const int i = 1 + blockIdx.x / rb_n, rb = blockIdx.x % rb_n;
    // This kernel runs next to (or right behind) the first-layer backward, which saturates HBM: a memory round
    // trip costs several microseconds then.  Everything the block needs -- dz of the layer, its 16 activation
    // rows, 16 rows of weights and Adam moments -- is therefore requested up front, ONE round trip, before the
    // first dependent instruction (stores to the same arrays would otherwise fence later loads in).
    float dz[kMaxB];
#pragma unroll
    for (int b = 0; b < kMaxB; ++b) dz[b] = a.dzs[((int64_t)i * kMaxB + b) * H + j];
    constexpr int kAsPer = 2;  // kUpdRows * kMaxB / 256 staged activations per thread (H >= 256) or more (strided below)
    float as_reg[kAsPer];
#pragma unroll
    for (int q = 0; q < kAsPer; ++q) {
      const int idx = threadIdx.x + q * blockDim.x;
      const int kk = idx % kUpdRows, b = idx / kUpdRows;
      as_reg[q] = idx < kUpdRows * kMaxB ? a.acts[((int64_t)(i - 1) * kMaxB + b) * H + rb * kUpdRows + kk] : 0.f;
    }
    float bsum = 0.f;
#pragma unroll
    for (int b = 0; b < kMaxB; ++b) bsum += dz[b];
#pragma unroll
    for (int q = 0; q < kAsPer; ++q) {
      const int idx = threadIdx.x + q * blockDim.x;
      if (idx < kUpdRows * kMaxB) as[idx % kUpdRows][idx / kUpdRows] = as_reg[q];
    }
    for (int idx = threadIdx.x + kAsPer * blockDim.x; idx < kUpdRows * kMaxB; idx += blockDim.x) {  // widths < 256
      const int kk = idx % kUpdRows, b = idx / kUpdRows;
      as[kk][b] = a.acts[((int64_t)(i - 1) * kMaxB + b) * H + rb * kUpdRows + kk];
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kUpdRows; ++r) {
      float g = 0.f;
#pragma unroll
      for (int b = 0; b < kMaxB; ++b) g = fmaf(as[r][b], dz[b], g);
      adam_update(w16[r], m16[r], v16[r], g, alpha);
    }
#pragma unroll
    for (int r = 0; r < kUpdRows; ++r) {
      const int k = rb * kUpdRows + r;
      const int64_t idx = row0 + (int64_t)r * H;
      a.small[idx] = w16[r];
      a.m_small[idx] = m16[r];
      a.v_small[idx] = v16[r];
      if (a.slice_mode == 1)
        store_images(a.w_fs, a.w_bs, i, k, j, w16[r]);
      else
        store_sliced(a.w_fs, a.w_bs, H, a.Hc, i, k, j, w16[r]);
    }
    if (rb == 0) adam_at(sl.bh(i) + j, bsum);
  } else {
    // b1: gradient is the column sum of dZ1
    float g = 0.f;
    for (int b = 0; b < kMaxB; ++b) g += a.dzs[(int64_t)b * H + j];
    adam_at(sl.b1() + j, g);
    // Dense(2): Wo1[k][c] = sum_b a_{L-1}[b][k] dy1[b][c]
    const float* y1 = a.outs;
    const float* dy1 = a.outs + 64;
    const float* dy2 = a.outs + 128;
    float g0 = 0.f, g1 = 0.f;
    for (int b = 0; b < kMaxB; ++b) {
      const float av = a.acts[((int64_t)(L - 1) * kMaxB + b) * H + j];
      g0 = fmaf(av, dy1[2 * b], g0);
      g1 = fmaf(av, dy1[2 * b + 1], g1);
    }
    adam_at(sl.Wo1() + 2 * j, g0);
    adam_at(sl.Wo1() + 2 * j + 1, g1);
    if (j < 2) {  // bo1
      float s = 0.f;
      for (int b = 0; b < kMaxB; ++b) s += dy1[2 * b + j];
      adam_at(sl.bo1() + j, s);
    } else if (j < 6) {  // Wo2[i][c] = sum_b y1[b][i] dy2[b][c]
      const int q = j - 2, i2 = q / 2, c = q % 2;
      float s = 0.f;
      for (int b = 0; b < kMaxB; ++b) s = fmaf(y1[2 * b + i2], dy2[2 * b + c], s);
      adam_at(sl.Wo2() + q, s);
    } else if (j < 8) {  // bo2
      const int c = j - 6;
      float s = 0.f;
      for (int b = 0; b < kMaxB; ++b) s += dy2[2 * b + c];
      adam_at(sl.bo2() + c, s);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {  // the next hidden stack of this model reads what this block wrote
    __threadfence();
    atomicAdd(&a.st->upd_cnt, 1u);
    if (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1) tl_mark(a.tl, blockIdx.x ? 22u : 6u, (unsigned)a.tl_id);
  }
}

static size_t hidden_fixed_floats(int H, int L, int cluster) {
  const int Hc = H / cluster;
  const size_t SL = (size_t)kMaxB * hid_row_pitch(Hc);
  return 2 * cluster * SL + 2 * SL + (size_t)kHidWarps * kMaxB * Hc + (size_t)2 * L * kMaxB * Hc + (size_t)kMaxB * Hc +
         320 + (size_t)((L * Hc + 3) & ~3) + (size_t)((2 * H + 8 + 3) & ~3);
}

int hidden_slots(int H, int L, int cluster) {
  const size_t budget = 226 * 1024;
  const size_t fixed = hidden_fixed_floats(H, L, cluster) * sizeof(float);
  const size_t slot = (size_t)H * (H / cluster) * sizeof(float);
  if (fixed + slot > budget) return 0;
  size_t ns = (budget - fixed) / slot;
  const size_t want = (size_t)2 * (L - 1);
  if (ns > want) ns = want;
  if (ns > kMaxSlots) ns = kMaxSlots;
  return (int)ns;
}

size_t hidden_smem_bytes(int H, int L, int cluster) {
  const int ns = hidden_slots(H, L, cluster);
  return hidden_fixed_floats(H, L, cluster) * sizeof(float) + (size_t)ns * H * (H / cluster) * sizeof(float);
}

typedef void (*hidden_fn)(HidGroupArgs);
static hidden_fn hidden_kernel(int H, int cluster) {
  return (H == 256 && cluster == 16) ? k_hidden<256, 16> : k_hidden<0, 0>;
}

// One cluster of `cluster` CTAs per model of the group.  The clusters need not be co-resident: none waits on another.
static int launch_hidden_cluster(const HidGroupArgs& g, int cluster, cudaStream_t s, bool dry) {
  const HidArgs& a = g.a[0];
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(cluster * g.n));
  cfg.blockDim = dim3(kHidThreads);
  cfg.dynamicSmemBytes = hidden_smem_bytes(a.H, a.L, cluster);
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)cluster;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  if (dry) {
    int n = 0;
    cudaError_t e = cudaOccupancyMaxActiveClusters(&n, hidden_kernel(a.H, cluster), &cfg);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return 0;
    }
    return n;
  }
  LOC_CUDA(cudaLaunchKernelEx(&cfg, hidden_kernel(a.H, cluster), g));
  loc::g_launches.fetch_add(1);
  return 0;
}

static const int kClusterCands[5] = {16, 8, 4, 2, 1};

int hidden_max_nlayers(int H) {
  if (H < 32 || H > 1024 || H % 32 != 0) return 0;
  // fixed shared memory grows with L, so the shapes with a slot are L = 2 .. deepest
  for (int L = 64; L >= 2; --L)
    for (int c : kClusterCands)
      if (H % (4 * c) == 0 && hidden_slots(H, L, c) >= 1) return L;
  return 0;
}

int hidden_max_cluster(int H, int L) {
  cudaFuncSetAttribute(k_hidden<256, 16>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  cudaFuncSetAttribute(k_hidden<0, 0>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  cudaGetLastError();
  for (int c : kClusterCands) {
    if (H % (4 * c) != 0) continue;
    if (hidden_slots(H, L, c) < 1) continue;
    const size_t smem = hidden_smem_bytes(H, L, c);
    if (cudaFuncSetAttribute(hidden_kernel(H, c), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
      cudaGetLastError();
      continue;
    }
    HidGroupArgs dummy = {};
    dummy.n = 1;
    dummy.a[0].H = H;
    dummy.a[0].L = L;
    if (launch_hidden_cluster(dummy, c, 0, true) > 0) return c;
  }
  return 0;
}

int hidden_group_launch(const HidGroupArgs& g, int cluster, cudaStream_t s) {
  LOC_CHECK(g.n >= 1 && g.n <= kMaxGroup, "hidden stack group: bad group size");
  const HidArgs& a = g.a[0];
  LOC_CHECK(cluster > 0 && a.H % (4 * cluster) == 0, "hidden stack: width must be a multiple of 4 x cluster size");
  LOC_CHECK(a.H % 32 == 0, "hidden stack: width must be a multiple of 32");
  LOC_CHECK(a.n_slots >= 1, "hidden stack: shared memory budget exceeded for this width / nlayers");
  for (int i = 1; i < g.n; ++i)  // one launch has one shared-memory size and one slice geometry
    LOC_CHECK(g.a[i].H == a.H && g.a[i].L == a.L && g.a[i].n_slots == a.n_slots,
              "hidden stack group: the models of one launch must share width, nlayers and cluster size");
  const size_t smem = hidden_smem_bytes(a.H, a.L, cluster);
  LOC_CUDA(cudaFuncSetAttribute(hidden_kernel(a.H, cluster), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  return launch_hidden_cluster(g, cluster, s, false);
}

int hidden_launch(const HidArgs& a, int cluster, cudaStream_t s) {
  HidGroupArgs g;
  g.n = 1;
  g.a[0] = a;
  return hidden_group_launch(g, cluster, s);
}

int hidden_reslice(const float* small, float* fs, float* bs, int H, int L, int cluster, cudaStream_t s) {
  if (L < 2) return 0;
  k_reslice<<<148 * 4, 256, 0, s>>>(small, fs, bs, H, L, H / cluster);
  LOC_LAUNCHED();
  return 0;
}

int hidden_update_blocks(int H, int L) { return (L - 1) * (H / kUpdRows) + 1; }

int hidden_update_launch(const UpdArgs& a, cudaStream_t s, bool overlap_previous) {
  LOC_CHECK(a.H % kUpdRows == 0 && a.H >= 32 && a.H <= 1024, "hidden update: bad width");
  const int nblk = hidden_update_blocks(a.H, a.L);
  // overlap_previous: programmatic dependent launch (see l1_backward_tc) -- the update of a model whose hidden
  // stack finished a slot earlier runs next to another model's first-layer backward
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)nblk);
  cfg.blockDim = dim3((unsigned)a.H);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = overlap_previous ? 1 : 0;
  LOC_CUDA(cudaLaunchKernelEx(&cfg, k_hidden_update, a));
  loc::g_launches.fetch_add(1);
  return 0;
}

}  // namespace loc
