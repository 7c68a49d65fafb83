// Optimizer steps of 33..256 rows (--batch_size > 32: locator/locator.py:69,371 pass any batch size to model.fit).
//
// The fused tensor-core kernels of the default path hold ONE 32-row batch tile (l1_tc.cu, hidden_tc.cu).  Only the
// BatchNormalization in front of the first Dense couples the rows of a batch; everything behind it is row-wise, and
// every gradient is a sum over rows.  A larger step is therefore run as
//
//   k_bb_stats         batch mean / variance of every SNP over ALL rows of the step (+ moving statistics)
//   first-layer forward with those statistics (the inference kernels read them in place of the moving ones:
//                      one wide pass over W1 for up to 256 rows on the tcgen05 path), then the 32-row chunks
//                      through the unchanged hidden stack (tcgen05 path: side by side, one cluster per chunk of a
//                      grouped launch, k_bb_step_end closing the step; else one launch each): loss scaled by the
//                      step's row count, dropout stream indexed by the row's position in the step, activations /
//                      dz kept per chunk
//   k_bb_l1_bwd        S = (x - mean)^T dZ1 over all rows (mma.sync), dW1 = inv S + beta c0, Adam on W1 | m | v in
//                      one pass over the weights, either W1 layout; k_bb_gamma_beta: BatchNorm gamma / beta Adam
//   k_bb_hidden_update dW + Adam of the small layers summed over the chunks
//
// so W1 | m | v are still streamed once per optimizer step.  Keras semantics as restated in oracle/model_ref.py
// (RefLocator.gradients / train_step); algebra of the first layer as in l1_simt.cu.
#include <cuda_fp16.h>

#include "model.cuh"
#include "hidden_slices.cuh"

namespace loc {

constexpr int kBbT = 16;  // SNPs per chunk of the backward = one packed word per row

__device__ __forceinline__ void bb_moments(int n1, int n2, int nb, float& mean, float& var) {
  // tf.nn.moments: mean, then mean of squared differences (as l1_simt.cu: batch_moments)
  const float fn = (float)nb;
  const int n0 = nb - n1 - n2;
  mean = (float)(n1 + 2 * n2) / fn;
  const float d0 = 0.f - mean, d1 = 1.f - mean, d2 = 2.f - mean;
  var = ((float)n0 * d0 * d0 + (float)n1 * d1 * d1 + (float)n2 * d2 * d2) / fn;
}

// Genotype counts over the step's rows -> batch statistics.  256 threads = 32 packed words (16 SNPs each) x 8 row
// slices; the slices' counts meet in shared memory (integer atomics: order-free), then one thread per SNP finishes.
// blockIdx.y: model of a replicate group (the grid covers the largest K of the group).
__global__ void __launch_bounds__(256) k_bb_stats(BigGroupArgs ga) {
  const BigArgs& a = ga.a[blockIdx.y];
  if ((int64_t)blockIdx.x * 32 * 16 >= a.K) return;
  if (a.gated && a.st->stopped) return;
  __shared__ int64_t s_rows[LOC_MAX_BATCH_SIZE];
  __shared__ unsigned cnt[32][2][16];
  const int nb = a.nb, tid = threadIdx.x;
  for (int b = tid; b < nb; b += blockDim.x) s_rows[b] = row_of(a.src, a.st, b);
  for (int i = tid; i < 32 * 2 * 16; i += blockDim.x) (&cnt[0][0][0])[i] = 0u;
  __syncthreads();
  const int wl = tid & 31, slice = tid >> 5;
  const int64_t w = (int64_t)blockIdx.x * 32 + wl;
  if (w * 16 < a.K) {
    unsigned n1[16], n2[16];  // rows with one / two alternate alleles, per SNP of the word
#pragma unroll
    for (int t = 0; t < 16; ++t) n1[t] = n2[t] = 0u;
#pragma unroll 4
    for (int b = slice; b < nb; b += 8) {
      const uint32_t x = __ldg(a.packed + s_rows[b] * a.row_words + w);
      const uint32_t lo = x & 0x55555555u, hi = (x >> 1) & 0x55555555u;
      const uint32_t is1 = lo & ~hi, is2 = hi & ~lo;
#pragma unroll
      for (int t = 0; t < 16; ++t) {
        n1[t] += (is1 >> (2 * t)) & 1u;
        n2[t] += (is2 >> (2 * t)) & 1u;
      }
    }
#pragma unroll
    for (int t = 0; t < 16; ++t) {
      atomicAdd(&cnt[wl][0][t], n1[t]);
      atomicAdd(&cnt[wl][1][t], n2[t]);
    }
  }
  __syncthreads();
  for (int i = tid; i < 32 * 16; i += blockDim.x) {
    const int64_t k = ((int64_t)blockIdx.x * 32 + (i >> 4)) * 16 + (i & 15);
    if (k < a.K) {
      float mean, var;
      bb_moments((int)cnt[i >> 4][0][i & 15], (int)cnt[i >> 4][1][i & 15], nb, mean, var);
      a.bmean[k] = mean;
      a.bvar[k] = var;
      a.mmean[k] = a.mmean[k] * kBnMom + mean * kBnOneMinusMom;
      a.mvar[k] = a.mvar[k] * kBnMom + var * kBnOneMinusMom;
    }
  }
}

__device__ __forceinline__ const float* bb_dz1(const BigArgs& a, int b) {  // dZ1 row b of the step
  return a.dzs + ((int64_t)(b >> 5) * a.L * kMaxB + (b & 31)) * a.H;
}

// ---------------------------------------------------------------------------------------------------------------
// First-layer backward + Adam of a large step:  S[k][j] = sum_b (x[b][k] - mean_k) dZ1[b][j]  on the warp-level tensor
// core path (mma.sync m16n8k16, fp16 operands, fp32 accumulate) with the precision of the 32-row kernel (l1_tc.cu):
// centred genotypes carry 11 significant bits (fp16 here, tf32 there: exact whenever the row count is a power of
// two), dZ1 goes in as hi + lo parts (22 bits) -- of dZ1 scaled by a power of two per block so that its largest
// entry sits just below fp16's maximum (the scale is taken out of S again, exactly).  Half the tensor instructions of
// the tf32 shape (m16n8k8, hi + lo: 264 us at 256 rows, tensor-bound on this legacy path) for the same bits.  The
// product is small next to the W1 | m | v stream (24 K H bytes, once per step); the tensor cores are here to keep the
// instruction count of the product below that of Adam, not for their peak.
//
// Grid = (column groups of CW = 64 (or 32) columns) x (SNP ranges); 512 threads = 16 warps.  The block's slice of
// dZ1 is split into hi / lo once and kept in shared memory in B-fragment order for the whole SNP range; per
// iteration the block takes 32 packed words (16 SNPs each) of every row of the step into shared memory, and each
// warp owns two of them, one after the other (a 16-SNP m-tile x all CW columns): A fragments are expanded from the
// 2-bit genotypes in registers, one 16-byte shared load per (16 rows, 8 columns) brings both parts of a B fragment.
// The warp then runs Adam on its 16 x CW block of W1 | m | v straight from the accumulator fragments (16-byte
// accesses; three units = 9 loads per thread stay in flight, the first three requested before the products), and
// leaves P_k = sum_j W1 S, Q_k = sum_j W1 c0 of its column group in global memory: BatchNorm gamma / beta need them
// over ALL columns (k_bb_gamma_beta).
constexpr int kBbThreads = 512;
constexpr int kBbWarps = kBbThreads / 32;
constexpr int kBbWordsPerIter = 2 * kBbWarps;  // 32

// two floats -> packed fp16 pair (round to nearest even); `lo` lands in the lower half
__device__ __forceinline__ uint32_t bb_h2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float bb_h_round(float x) {  // x rounded to fp16, as a float
  return __half2float(__float2half_rn(x));
}
__device__ __forceinline__ void bb_mma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// Which column of the block's column group sits at accumulator column c (0..7) of n-tile n.  Not n * 8 + c: inside
// every 32-column chunk the four n-tiles are interleaved so that the thread that owns accumulator columns 2 tig,
// 2 tig + 1 of all four owns columns 4 tig .. 4 tig + 3 and 16 + 4 tig .. 16 + 4 tig + 3 of the chunk: its share of a
// row of W1 | m | v is two 16-byte accesses, and a warp instruction covers whole 32-byte sectors (8 rows x 64 bytes)
// instead of 8 rows x four quarter-used sectors.
__host__ __device__ __forceinline__ int bb_phys_col(int n, int c) {
  return 32 * (n >> 2) + 16 * ((n & 3) >> 1) + 4 * (c >> 1) + 2 * (n & 1) + (c & 1);
}

// Keras Adam with the hardware's approximate root and quotient (~1 ulp each), as the 32-row kernel (l1_tc.cu)
__device__ __forceinline__ void bb_adam(float& w, float& m, float& v, float g, float alpha) {
  m = m + (g - m) * kAdam1mB1;
  v = v + (g * g - v) * kAdam1mB2;
  float rt;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(rt) : "f"(v));
  w = w - __fdividef(m * alpha, rt + kAdamEps);
}

template <int CW, bool TILED>
__global__ void __launch_bounds__(kBbThreads, 1) k_bb_l1_bwd(BigArgs a, float* __restrict__ pq_part) {
  if (a.gated && a.st->stopped) return;
  constexpr int NT = CW / 8;  // 8-column n-tiles of the column group
  extern __shared__ __align__(16) uint8_t bb_raw[];
  const int H = a.H, nb = a.nb, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, tig = lane & 3;
  const int nk = (nb + 15) >> 4;      // k-steps of 16 rows
  const int xw_pitch = nk * 16 + 1;   // words of one packed column in shared memory (odd: conflict-free transposing writes)
  uint4* dzf = reinterpret_cast<uint4*>(bb_raw);                                // [nk][NT][32]: (hi b0, hi b1, lo b0, lo b1), fp16 pairs
  uint32_t* xw0 = reinterpret_cast<uint32_t*>(dzf + (size_t)nk * NT * 32);      // [2 buffers][32 words][xw_pitch]
  float* raw0 = reinterpret_cast<float*>(xw0 + (size_t)2 * kBbWordsPerIter * xw_pitch);  // [2 buffers][mean, var, gamma, beta][512 SNPs]
  float* c0s = raw0 + 2 * 4 * kBbThreads;                                        // [CW] column sums of dZ1
  __shared__ int64_t s_rows[LOC_MAX_BATCH_SIZE];
  __shared__ float s_red[kBbWarps];
  const int J0 = blockIdx.x * CW;
  for (int b = tid; b < nb; b += kBbThreads) s_rows[b] = row_of(a.src, a.st, b);
  // power-of-two scale of the block's slice of dZ1: largest entry into [2^14, 2^15)
  float amax = 0.f;
  for (int i = tid; i < nb * CW; i += kBbThreads) amax = fmaxf(amax, fabsf(__ldg(bb_dz1(a, i / CW) + J0 + i % CW)));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
  if (lane == 0) s_red[warp] = amax;
  __syncthreads();
  amax = 0.f;
  for (int w = 0; w < kBbWarps; ++w) amax = fmaxf(amax, s_red[w]);
  const bool scalable = amax > 0.f && amax < 3.0e38f;  // (zeros, inf / nan: no scaling; non-finite values propagate as they are)
  const int sexp = scalable ? 14 - ilogbf(amax) : 0;
  const float dscale = scalbnf(1.f, sexp), dunscale = scalbnf(1.f, -sexp);
  for (int i = tid; i < nk * NT * 32; i += kBbThreads) {
    const int ln = i & 31, n = (i >> 5) % NT, ks = (i >> 5) / NT;
    const int r0 = ks * 16 + 2 * (ln & 3), col = J0 + bb_phys_col(n, ln >> 2);
    float v[4], h[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int r = r0 + (e & 1) + 8 * (e >> 1);  // rows 2 tig, 2 tig + 1 (b0), 2 tig + 8, 2 tig + 9 (b1)
      v[e] = r < nb ? __ldg(bb_dz1(a, r) + col) * dscale : 0.f;
      h[e] = bb_h_round(v[e]);
    }
    dzf[i] = make_uint4(bb_h2(h[0], h[1]), bb_h2(h[2], h[3]), bb_h2(v[0] - h[0], v[1] - h[1]), bb_h2(v[2] - h[2], v[3] - h[3]));
  }
  if (tid < CW) {
    float s = 0.f;
    for (int b = 0; b < nb; ++b) s += __ldg(bb_dz1(a, b) + J0 + tid);
    c0s[tid] = s;
  }
  const float alpha = a.st->alpha;

  const int64_t nwords = (a.K + kBbT - 1) / kBbT;
  const int64_t c_begin = nwords * blockIdx.y / gridDim.y, c_end = nwords * (blockIdx.y + 1) / gridDim.y;
  // The iteration's inputs -- 32 packed words of every row, batch statistics / gamma / beta of its 512 SNPs -- are
  // requested one iteration ahead with cp.async into the other half of a double buffer (no registers, no stall: the
  // first version loaded them at the top of the iteration and the whole block sat through a DRAM round trip there,
  // 30 % of the kernel's stall samples at 64 rows).  Consecutive threads take consecutive words of one row (coalesced).
  auto stage = [&](int64_t cgn, int bi) {
    uint32_t* xw = xw0 + (size_t)bi * kBbWordsPerIter * xw_pitch;
    for (int i = tid; i < kBbWordsPerIter * nk * 16; i += kBbThreads) {
      const int wi = i & (kBbWordsPerIter - 1), b = i / kBbWordsPerIter;
      const bool ok = b < nb && cgn + wi < c_end;
      const uint32_t* src = ok ? a.packed + s_rows[b] * a.row_words + cgn + wi : a.packed;
      asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(xw + wi * xw_pitch + b)),
                   "l"(src), "r"(ok ? 4 : 0)
                   : "memory");  // (size 0: zero fill)
    }
    const int64_t k = cgn * kBbT + tid;  // 512 threads = 32 words x 16 SNPs
    const bool ok = k < c_end * kBbT && k < a.K;
    const float* srcs[4] = {a.bmean, a.bvar, a.gamma, a.beta};
#pragma unroll
    for (int q = 0; q < 4; ++q)
      asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(
                       (uint32_t)__cvta_generic_to_shared(raw0 + (bi * 4 + q) * kBbThreads + tid)),
                   "l"(ok ? srcs[q] + k : srcs[q]), "r"(ok ? 4 : 0)
                   : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  // per-thread parts of the W1 | m | v offsets (see `unit` below)
  const int tb = TILED ? (g * 32 + 4 * (tig & 1) + (J0 >> 5) * 256) : (g * H + J0 + 4 * tig);
  const int xo0 = TILED ? (((tig >> 1) ^ (g & 3)) << 3) : 0, xo1 = TILED ? (((2 + (tig >> 1)) ^ (g & 3)) << 3) : 16;
  __syncthreads();  // s_rows
  stage(c_begin, 0);
  int it = 0;
  for (int64_t cg = c_begin; cg < c_end; cg += kBbWordsPerIter, ++it) {
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();  // this iteration's inputs are there; everybody is done with the previous iteration's (and the set-up)
    if (cg + kBbWordsPerIter < c_end) stage(cg + kBbWordsPerIter, (it + 1) & 1);
    const uint32_t* xw = xw0 + (size_t)(it & 1) * kBbWordsPerIter * xw_pitch;
    const float* raw = raw0 + (it & 1) * 4 * kBbThreads;
    {
      // L2 prefetch of the iteration's rows of W1 | m | v (393 KB at CW = 64): they are needed after the products
      // below, a few microseconds from now -- the DRAM reads run under the tensor-core phase instead of after it
      constexpr int LPW = 16 * CW / 32;  // 128-byte lines per (word, array)
      for (int i = tid; i < kBbWordsPerIter * 3 * LPW; i += kBbThreads) {
        const int l = i % LPW, arr = (i / LPW) % 3, wi = i / (3 * LPW);
        const int64_t cw = cg + wi;
        if (cw >= c_end) continue;
        const float* base = arr == 0 ? a.W1 : (arr == 1 ? a.mW1 : a.vW1);
        int64_t off;
        bool on;
        if (TILED) {  // per (8 SNPs, 32 columns): 1 KB contiguous (rows are padded to a multiple of 64 SNPs)
          const int per_chunk = 8, cc = (l / per_chunk) % (CW / 32), sb = l / (per_chunk * (CW / 32));
          off = w1_tiled_index(cw * kBbT + 8 * sb, J0 + 32 * cc) + 32 * (l % per_chunk);
          on = true;
        } else {
          const int t = l / (CW / 32), part = l % (CW / 32);
          off = (cw * kBbT + t) * H + J0 + 32 * part;
          on = cw * kBbT + t < a.K;
        }
        if (on) asm volatile("prefetch.global.L2 [%0];" ::"l"(base + off));
      }
    }
    // ---- each warp: its two words of the iteration, one after the other: products (one 16-SNP m-tile x all CW columns
    //      of the group), then Adam on that 16 x CW block of W1 | m | v straight from the accumulator fragments
    //      acc[n] = {S(g, c), S(g, c + 1), S(g + 8, c), S(g + 8, c + 1)}, accumulator column c = 2 tig of n-tile n = column
    //      J0 + bb_phys_col(n, c) of the layer.  The word's first three units are requested BEFORE the products.
#pragma unroll 1
    for (int mt = 0; mt < 2; ++mt) {
      const int wi = 2 * warp + mt;
      const int64_t cw = cg + wi;
      if (cw >= c_end) break;  // (whole warps; the barriers at the top of the iteration are reached by everybody)
      const int64_t k0 = cw * kBbT;
      const bool on_lo = k0 + g < a.K, on_hi = k0 + g + 8 < a.K;
      // One unit = (32-column chunk q, SNP g or g + 8, half h): the thread's columns 16 h + 4 tig .. + 3 of the chunk, 16 bytes
      // of each of W1 | m | v.  Three units are in flight while a fourth is updated in place (9 loads per thread).
      constexpr int NU = 4 * (NT / 4);
      // element offset of unit u (w1_tiled_index of model.cuh, or row-major, with everything that does not depend on u
      // folded into the word's base pointers)
      auto unit = [&](int u) -> int {
        const int h = u & 1, hi = (u >> 1) & 1, q = u >> 2;
        return TILED ? (hi * 2048 + q * 256 + (h ? xo1 : xo0)) : (hi * 8 * H + 32 * q + (h ? xo1 : xo0));
      };
      const int64_t wb = (TILED ? ((k0 >> 3) << 11) : k0 * H) + tb;
      float* const pW = a.W1 + wb;
      float* const pM = a.mW1 + wb;
      float* const pV = a.vW1 + wb;
      float4 buf[4][3];  // [slot][W, m, v]
      auto fetch = [&](int u, float4 (&d)[3]) {
        const bool on = ((u >> 1) & 1) ? on_hi : on_lo;
        const int off = unit(u);
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        d[0] = on ? *reinterpret_cast<const float4*>(pW + off) : z;
        d[1] = on ? *reinterpret_cast<const float4*>(pM + off) : z;
        d[2] = on ? *reinterpret_cast<const float4*>(pV + off) : z;
      };
      fetch(0, buf[0]);
      fetch(1, buf[1]);
      fetch(2, buf[2]);
      float acc[NT][4];
#pragma unroll
      for (int n = 0; n < NT; ++n)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[n][e] = 0.f;
      {
        const float mean_lo = raw[wi * kBbT + g], mean_hi = raw[wi * kBbT + g + 8];  // SNPs g, g + 8
        const uint32_t* xa = xw + (size_t)wi * xw_pitch + 2 * tig;
        const uint4* bf = dzf + lane;
        // 2-bit genotype -> float without a conversion instruction: 2^23 + x as bits, minus 2^23 (exact), then centred
        auto cen = [](uint32_t x2, float mean) { return (__uint_as_float(0x4B000000u | (x2 & 3u)) - 8388608.f) - mean; };
#pragma unroll 2
        for (int ks = 0; ks < nk; ++ks) {
          const uint32_t* xr = xa + ks * 16;
          const uint32_t x0 = xr[0] >> (2 * g), x1 = xr[1] >> (2 * g);  // rows 16 ks + 2 tig, + 1
          const uint32_t x8 = xr[8] >> (2 * g), x9 = xr[9] >> (2 * g);  // rows 16 ks + 2 tig + 8, + 9
          uint32_t af[4];
          af[0] = bb_h2(cen(x0, mean_lo), cen(x1, mean_lo));              // (SNP g,     rows 2 tig, 2 tig + 1)
          af[1] = bb_h2(cen(x0 >> 16, mean_hi), cen(x1 >> 16, mean_hi));  // (SNP g + 8, rows 2 tig, 2 tig + 1)
          af[2] = bb_h2(cen(x8, mean_lo), cen(x9, mean_lo));              // (SNP g,     rows 2 tig + 8, + 9)
          af[3] = bb_h2(cen(x8 >> 16, mean_hi), cen(x9 >> 16, mean_hi));  // (SNP g + 8, rows 2 tig + 8, + 9)
#pragma unroll
          for (int n = 0; n < NT; ++n) {
            const uint4 b4 = bf[(ks * NT + n) * 32];
            bb_mma(acc[n], af, b4.x, b4.y);  // hi part of dZ1
            bb_mma(acc[n], af, b4.z, b4.w);  // lo part
          }
        }
      }
      // inv = gamma * rsqrt(var + eps), times the scale of dZ1 taken back out of S
      const float inv_lo = rsqrtf(raw[kBbThreads + wi * kBbT + g] + kBnEps) * raw[2 * kBbThreads + wi * kBbT + g] * dunscale;
      const float inv_hi = rsqrtf(raw[kBbThreads + wi * kBbT + g + 8] + kBnEps) * raw[2 * kBbThreads + wi * kBbT + g + 8] * dunscale;
      const float be_lo = raw[3 * kBbThreads + wi * kBbT + g], be_hi = raw[3 * kBbThreads + wi * kBbT + g + 8];
      float P[2] = {0.f, 0.f}, Q[2] = {0.f, 0.f};
#pragma unroll
      for (int u = 0; u < NU; ++u) {
        const int h = u & 1, hi = (u >> 1) & 1, q = u >> 2;
        if (u + 3 < NU) fetch(u + 3, buf[(u + 3) & 3]);
        const float inv = hi ? inv_hi : inv_lo, be = hi ? be_hi : be_lo;
        float4& w = buf[u & 3][0];
        float4& m = buf[u & 3][1];
        float4& v = buf[u & 3][2];
        // columns 16 h + 4 tig + {0, 1, 2, 3} of the chunk = accumulator columns 2 tig, 2 tig + 1 of n-tiles 4 q + 2 h, + 1
        const float4 c0 = *reinterpret_cast<const float4*>(c0s + 32 * q + 16 * h + 4 * tig);
        const float S0 = acc[4 * q + 2 * h][2 * hi], S1 = acc[4 * q + 2 * h][2 * hi + 1];
        const float S2 = acc[4 * q + 2 * h + 1][2 * hi], S3 = acc[4 * q + 2 * h + 1][2 * hi + 1];
        P[hi] = fmaf(w.x, S0, fmaf(w.y, S1, fmaf(w.z, S2, fmaf(w.w, S3, P[hi]))));
        Q[hi] = fmaf(w.x, c0.x, fmaf(w.y, c0.y, fmaf(w.z, c0.z, fmaf(w.w, c0.w, Q[hi]))));
        bb_adam(w.x, m.x, v.x, inv * S0 + be * c0.x, alpha);
        bb_adam(w.y, m.y, v.y, inv * S1 + be * c0.y, alpha);
        bb_adam(w.z, m.z, v.z, inv * S2 + be * c0.z, alpha);
        bb_adam(w.w, m.w, v.w, inv * S3 + be * c0.w, alpha);
        if (hi ? on_hi : on_lo) {
          const int off = unit(u);
          *reinterpret_cast<float4*>(pW + off) = w;
          *reinterpret_cast<float4*>(pM + off) = m;
          *reinterpret_cast<float4*>(pV + off) = v;
        }
      }
      // sums over the warp's columns: the four lanes of a group hold different column pairs of the same SNPs
#pragma unroll
      for (int hi = 0; hi < 2; ++hi) {
        P[hi] *= dunscale;  // P = sum_j W1 S with the true S
#pragma unroll
        for (int o = 1; o <= 2; o <<= 1) {
          P[hi] += __shfl_xor_sync(0xffffffffu, P[hi], o);
          Q[hi] += __shfl_xor_sync(0xffffffffu, Q[hi], o);
        }
        const int64_t k = k0 + g + 8 * hi;
        if (tig == 0 && k < a.K) {
          pq_part[((int64_t)blockIdx.x * 2) * a.K + k] = P[hi];
          pq_part[((int64_t)blockIdx.x * 2 + 1) * a.K + k] = Q[hi];
        }
      }
    }
  }
}

// BatchNorm gamma / beta of a large step: P_k, Q_k summed over the column groups in order, then Adam.
__global__ void __launch_bounds__(256) k_bb_gamma_beta(BigArgs a, const float* __restrict__ pq_part, int ncg) {
  if (a.gated && a.st->stopped) return;
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= a.K) return;
  const float alpha = a.st->alpha;
  float P = 0.f, Q = 0.f;
  for (int g = 0; g < ncg; ++g) {
    P += pq_part[((int64_t)g * 2) * a.K + k];
    Q += pq_part[((int64_t)g * 2 + 1) * a.K + k];
  }
  const float rs = rsqrtf(a.bvar[k] + kBnEps);
  const float dgamma = rs * P;  // exactly 0 for a SNP that is constant in the batch (centred genotypes: S = 0)
  const float dbeta = Q;
  float gm = a.gamma[k], mo = a.m_gamma[k], vo = a.v_gamma[k];
  adam_update(gm, mo, vo, dgamma, alpha);
  a.gamma[k] = gm;
  a.m_gamma[k] = mo;
  a.v_gamma[k] = vo;
  float bt = a.beta[k];
  mo = a.m_beta[k];
  vo = a.v_beta[k];
  adam_update(bt, mo, vo, dbeta, alpha);
  a.beta[k] = bt;
  a.m_beta[k] = mo;
  a.v_beta[k] = vo;
}

// dW + Adam of the small layers over the chunks of the step.  Blocks [0, (L-1)*H/16): 16 input rows x H outputs of
// hidden layer i; last block: b1, Dense(2), Dense(2).  blockDim = (H, S): thread (j, s) <-> output column j, chunks
// s, s + S, ... (every chunk costs a memory round trip; S of them run side by side), partial sums meet in shared memory
// in split order, and split s finishes rows r = s, s + S, ... of the block.
constexpr int kBbRows = 16;
constexpr int kBbSplits = 4;

__global__ void __launch_bounds__(1024) k_bb_hidden_update(BigArgs a) {
  if (a.gated && a.st->stopped) return;
  extern __shared__ float bb_red[];  // [S][16 rows + 1][H]: partial dW rows, then the partial bias gradient
  __shared__ float as[kBbSplits][kBbRows][kMaxB + 1];
  const int H = a.H, L = a.L, j = threadIdx.x, sp = threadIdx.y, S = blockDim.y;
  const SmallLayout sl{H, L};
  const int rb_n = H / kBbRows;
  const int nblk_hidden = (L - 1) * rb_n;
  const int nchunks = (a.nb + kMaxB - 1) / kMaxB;
  const int64_t chunk_stride = (int64_t)L * kMaxB * H;
  const float alpha = a.st->alpha;
  auto adam_at = [&](int64_t idx, float g) {
    float w = a.small[idx], m = a.m_small[idx], v = a.v_small[idx];
    adam_update(w, m, v, g, alpha);
    a.small[idx] = w;
    a.m_small[idx] = m;
    a.v_small[idx] = v;
  };
  if ((int)blockIdx.x < nblk_hidden) {
    const int i = 1 + blockIdx.x / rb_n, rb = blockIdx.x % rb_n;
    float g16[kBbRows];
#pragma unroll
    for (int r = 0; r < kBbRows; ++r) g16[r] = 0.f;
    float bsum = 0.f;
    for (int c0 = 0; c0 < nchunks; c0 += S) {  // (uniform trip count: the barriers below are block-wide)
      const int ci = c0 + sp;
      const bool on = ci < nchunks;
      const float* dzs = a.dzs + (on ? ci : 0) * chunk_stride;
      const float* acts = a.acts + (on ? ci : 0) * chunk_stride;
      float dz[kMaxB];
#pragma unroll
      for (int b = 0; b < kMaxB; ++b) dz[b] = on ? dzs[((int64_t)i * kMaxB + b) * H + j] : 0.f;
      __syncthreads();  // the previous round's activations have been consumed
      for (int idx = j; idx < kBbRows * kMaxB; idx += H) {
        const int kk = idx % kBbRows, b = idx / kBbRows;
        as[sp][kk][b] = on ? acts[((int64_t)(i - 1) * kMaxB + b) * H + rb * kBbRows + kk] : 0.f;
      }
      __syncthreads();
#pragma unroll
      for (int b = 0; b < kMaxB; ++b) bsum += dz[b];
#pragma unroll
      for (int r = 0; r < kBbRows; ++r) {
        float g = 0.f;
#pragma unroll
        for (int b = 0; b < kMaxB; ++b) g = fmaf(as[sp][r][b], dz[b], g);
        g16[r] += g;
      }
    }
#pragma unroll
    for (int r = 0; r < kBbRows; ++r) bb_red[((size_t)sp * (kBbRows + 1) + r) * H + j] = g16[r];
    bb_red[((size_t)sp * (kBbRows + 1) + kBbRows) * H + j] = bsum;
    __syncthreads();
    for (int r = sp; r < kBbRows + 1; r += S) {
      float g = 0.f;
      for (int q = 0; q < S; ++q) g += bb_red[((size_t)q * (kBbRows + 1) + r) * H + j];  // split order
      if (r == kBbRows) {
        if (rb == 0) adam_at(sl.bh(i) + j, g);
        continue;
      }
      const int k = rb * kBbRows + r;
      const int64_t idx = sl.Wh(i) + (int64_t)k * H + j;
      float w = a.small[idx], m = a.m_small[idx], v = a.v_small[idx];
      adam_update(w, m, v, g, alpha);
      a.small[idx] = w;
      a.m_small[idx] = m;
      a.v_small[idx] = v;
      if (a.slice_mode == 1)
        store_images(a.w_fs, a.w_bs, i, k, j, w);
      else
        store_sliced(a.w_fs, a.w_bs, H, a.Hc, i, k, j, w);
    }
  } else if (sp == 0) {
    float gb1 = 0.f, g0 = 0.f, g1 = 0.f, sb = 0.f;
    for (int ci = 0; ci < nchunks; ++ci) {
      const float* dzs = a.dzs + ci * chunk_stride;
      const float* acts = a.acts + ci * chunk_stride;
      const float* y1 = a.outs + ci * 256;
      const float* dy1 = y1 + 64;
      const float* dy2 = y1 + 128;
#pragma unroll 8
      for (int b = 0; b < kMaxB; ++b) {
        gb1 += dzs[(int64_t)b * H + j];  // b1: column sum of dZ1
        const float av = acts[((int64_t)(L - 1) * kMaxB + b) * H + j];  // Dense(2): Wo1[k][c] = sum_b a_{L-1}[b][k] dy1[b][c]
        g0 = fmaf(av, dy1[2 * b], g0);
        g1 = fmaf(av, dy1[2 * b + 1], g1);
      }
      if (j < 2) {  // bo1
        for (int b = 0; b < kMaxB; ++b) sb += dy1[2 * b + j];
      } else if (j < 6) {  // Wo2[i][c] = sum_b y1[b][i] dy2[b][c]
        const int q = j - 2, i2 = q / 2, c = q % 2;
        for (int b = 0; b < kMaxB; ++b) sb = fmaf(y1[2 * b + i2], dy2[2 * b + c], sb);
      } else if (j < 8) {  // bo2
        for (int b = 0; b < kMaxB; ++b) sb += dy2[2 * b + (j - 6)];
      }
    }
    adam_at(sl.b1() + j, gb1);
    adam_at(sl.Wo1() + 2 * j, g0);
    adam_at(sl.Wo1() + 2 * j + 1, g1);
    if (j < 2)
      adam_at(sl.bo1() + j, sb);
    else if (j < 6)
      adam_at(sl.Wo2() + (j - 2), sb);
    else if (j < 8)
      adam_at(sl.bo2() + (j - 6), sb);
  }
}

// End of a large step whose chunks ran through the hidden stack side by side (grouped launches): per-chunk loss sums
// added in chunk order (same bits as chunk-by-chunk launches), then the optimizer bookkeeping of the step.  One block
// per model of a replicate group.
__global__ void k_bb_step_end(BigEndArgs e, int gated) {
  DevState* st = e.st[blockIdx.x];
  const float* slots = e.slots[blockIdx.x];
  if (gated && st->stopped) return;
  float acc = 0.f;
  for (int c = 0; c < e.nc[blockIdx.x]; ++c) {
    const float s = slots[2 * c], n = slots[2 * c + 1];
    const float mean = s / n;
    st->loss_total += mean * n;
    st->loss_count += n;
    acc += s;
    if (!isfinite(mean)) st->nonfinite = 1;
  }
  st->step_sum = acc;
  st->last_loss = acc / (float)e.loss_rows[blockIdx.x];
  const int t = st->t + 1;
  st->t = t;
  st->step_id = st->step_id + 1;
  const float b1p = powf(kAdamB1, (float)t), b2p = powf(kAdamB2, (float)t);
  st->alpha = st->lr * sqrtf(1.f - b2p) / (1.f - b1p);
}

int bb_step_end_launch(const BigEndArgs& e, int gated, cudaStream_t s) {
  LOC_CHECK(e.n >= 1 && e.n <= kMaxGroup, "step end (large batch): bad group size");
  k_bb_step_end<<<(unsigned)e.n, 1, 0, s>>>(e, gated);
  LOC_LAUNCHED();
  return 0;
}

int bb_stats_launch(const BigGroupArgs& g, cudaStream_t s) {
  LOC_CHECK(g.n >= 1 && g.n <= kMaxGroup, "batch statistics: bad group size");
  int64_t kmax = 0;
  for (int i = 0; i < g.n; ++i) {
    LOC_CHECK(g.a[i].nb >= 1 && g.a[i].nb <= LOC_MAX_BATCH_SIZE, "batch statistics: a step holds 1..256 rows");
    if (g.a[i].K > kmax) kmax = g.a[i].K;
  }
  k_bb_stats<<<dim3((unsigned)cdiv(cdiv(kmax, 16), 32), (unsigned)g.n), 256, 0, s>>>(g);
  LOC_LAUNCHED();
  return 0;
}

int64_t bb_pq_floats(int64_t K, int H) { return 2 * (int64_t)(H / (H % 64 == 0 ? 64 : 32)) * K; }

template <int CW, bool TILED>
static int bb_l1_backward_cw(const BigArgs& a, float* pq_part, cudaStream_t s) {
  constexpr int NT = CW / 8;
  const int ncg = a.H / CW;
  const int nk = (a.nb + 15) / 16;
  const size_t smem = (size_t)nk * NT * 32 * sizeof(uint4) + (size_t)2 * kBbWordsPerIter * (nk * 16 + 1) * sizeof(uint32_t) +
                      (size_t)(2 * 4 * kBbThreads + CW) * sizeof(float);
  LOC_CUDA(cudaFuncSetAttribute(k_bb_l1_bwd<CW, TILED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t niter = cdiv(cdiv(a.K, kBbT), kBbWordsPerIter);
  int64_t by = cdiv((int64_t)sm_count(), ncg);  // one 512-thread block per SM
  if (by > niter) by = niter;
  if (by < 1) by = 1;
  k_bb_l1_bwd<CW, TILED><<<dim3((unsigned)ncg, (unsigned)by), kBbThreads, smem, s>>>(a, pq_part);
  LOC_LAUNCHED();
  k_bb_gamma_beta<<<(unsigned)cdiv(a.K, 256), 256, 0, s>>>(a, pq_part, ncg);
  LOC_LAUNCHED();
  return 0;
}

int bb_l1_backward_launch(const BigArgs& a, float* pq_part, cudaStream_t s) {
  LOC_CHECK(a.H % 32 == 0 && a.H >= 32 && a.H <= 1024, "first layer (large batch): width must be a multiple of 32 in [32, 1024]");
  LOC_CHECK(pq_part != nullptr, "first layer (large batch): no scratch for the gamma / beta partial sums");
  if (a.H % 64 == 0) return a.tiled ? bb_l1_backward_cw<64, true>(a, pq_part, s) : bb_l1_backward_cw<64, false>(a, pq_part, s);
  return a.tiled ? bb_l1_backward_cw<32, true>(a, pq_part, s) : bb_l1_backward_cw<32, false>(a, pq_part, s);
}

int bb_hidden_update_launch(const BigArgs& a, cudaStream_t s) {
  LOC_CHECK(a.H % kBbRows == 0 && a.H >= 32 && a.H <= 1024, "hidden update (large batch): bad width");
  const int nblk = (a.L - 1) * (a.H / kBbRows) + 1;
  const int nchunks = (a.nb + kMaxB - 1) / kMaxB;
  int S = 1024 / a.H;  // chunks side by side in a block
  if (S > kBbSplits) S = kBbSplits;
  if (S > nchunks) S = nchunks;
  if (S < 1) S = 1;
  const size_t smem = (size_t)S * (kBbRows + 1) * a.H * sizeof(float);
  static size_t smem_set = 0;
  if (smem > smem_set) {
    LOC_CUDA(cudaFuncSetAttribute(k_bb_hidden_update, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  k_bb_hidden_update<<<nblk, dim3((unsigned)a.H, (unsigned)S), smem, s>>>(a);
  LOC_LAUNCHED();
  return 0;
}

}  // namespace loc
