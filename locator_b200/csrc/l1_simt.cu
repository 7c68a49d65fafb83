// First layer (BatchNorm folded into Dense(K -> H)), CUDA-core fp32 version.
//
// This is the exact-fp32 variant of the first-layer kernels: used for widths the tcgen05 kernels do
// not cover and as the on-device cross-check of l1_tc.cu.  Same decomposition, same scratch buffers.
//
// Reference: BatchNormalization + Dense + their gradients + Adam inside model.fit,
// locator/locator.py:318-320,367-376 (Keras semantics restated in oracle/model_ref.py).
//
// Algebra used by both variants (x in {0,1,2} is the raw genotype, per SNP k):
//   forward   xhat[b,k] = x*inv_k + shift_k,  inv_k = gamma_k*rsqrt(var_k+eps), shift_k = beta_k - mean_k*inv_k
//             Z1[b,j]   = sum_k xhat[b,k] W1[k,j]
//   backward  S[k,j]    = sum_b (x[b,k] - mean_k) dZ1[b,j],   c0[j] = sum_b dZ1[b,j]
//             dW1[k,j]  = inv_k*S[k,j] + beta_k*c0[j]
//             P_k = sum_j W1[k,j] S[k,j],  Q_k = sum_j W1[k,j] c0[j]
//             dgamma_k  = rs_k*P_k,  dbeta_k = Q_k
//   (centred genotypes keep dgamma exactly 0 for a SNP that is constant within the batch, as in
//   the reference; Adam would turn rounding noise there into full-size steps)
#include "model.cuh"

namespace loc {

// Genotypes of SNP k for the nb rows of the step, 2 bits each, in one 64-bit word (+ counts).
struct SnpBatch {
  unsigned long long bits;
  int n1, n2;
};

__device__ __forceinline__ SnpBatch load_snp(const uint32_t* __restrict__ packed, int64_t row_words,
                                             const int64_t* __restrict__ s_rows, int nb, int64_t k) {
  SnpBatch r;
  r.bits = 0ull;
  r.n1 = 0;
  r.n2 = 0;
  const int64_t w = k >> 4;
  const int sh = 2 * (int)(k & 15);
#pragma unroll 8
  for (int b = 0; b < nb; ++b) {
    const unsigned x = (__ldg(packed + s_rows[b] * row_words + w) >> sh) & 3u;
    r.bits |= (unsigned long long)x << (2 * b);
    r.n1 += (x == 1u);
    r.n2 += (x == 2u);
  }
  return r;
}

// Batch statistics the way tf.nn.moments computes them (mean, then mean of squared differences).
__device__ __forceinline__ void batch_moments(const SnpBatch& s, int nb, float& mean, float& var) {
  const float fn = (float)nb;
  const int n0 = nb - s.n1 - s.n2;
  mean = (float)(s.n1 + 2 * s.n2) / fn;  // true division: a constant column gives mean == x exactly
  const float d0 = 0.f - mean, d1 = 1.f - mean, d2 = 2.f - mean;
  var = ((float)n0 * d0 * d0 + (float)s.n1 * d1 * d1 + (float)s.n2 * d2 * d2) / fn;
}

__global__ void __launch_bounds__(1024) k_l1_fwd_simt(L1Args a, int n_partials) {
  if (a.gated && a.st->stopped) return;
  extern __shared__ float xh[];  // [kF1Chunk][kMaxB + 1]
  __shared__ int64_t s_rows[kMaxB];
  const int tid = threadIdx.x;
  const int H = a.H;
  const int nb = a.src.nb;
  if (tid < nb) s_rows[tid] = row_of(a.src, a.st, tid);
  __syncthreads();

  const int64_t nchunks = (a.K + kF1Chunk - 1) / kF1Chunk;
  const int64_t c_begin = nchunks * blockIdx.x / n_partials;
  const int64_t c_end = nchunks * (blockIdx.x + 1) / n_partials;

  float acc[kMaxB];
#pragma unroll
  for (int b = 0; b < kMaxB; ++b) acc[b] = 0.f;

  for (int64_t c = c_begin; c < c_end; ++c) {
    const int64_t k0 = c * kF1Chunk;
    for (int t = tid; t < kF1Chunk; t += blockDim.x) {
      const int64_t k = k0 + t;
      float* row = xh + t * (kMaxB + 1);
      if (k < a.K) {
        SnpBatch sb = load_snp(a.packed, a.row_words, s_rows, nb, k);
        float mean, var;
        if (a.training) {
          batch_moments(sb, nb, mean, var);
          a.mmean[k] = a.mmean[k] * kBnMom + mean * kBnOneMinusMom;
          a.mvar[k] = a.mvar[k] * kBnMom + var * kBnOneMinusMom;
        } else {
          mean = a.mmean[k];
          var = a.mvar[k];
        }
        const float inv = rsqrtf(var + kBnEps) * a.gamma[k];
        const float shift = a.beta[k] - mean * inv;
        const unsigned long long miss = sb.bits & (sb.bits >> 1) & 0x5555555555555555ull;  // x = 3 at bit 2b
        for (int b = 0; b < kMaxB; ++b) {
          const float x = (float)((sb.bits >> (2 * b)) & 3ull);
          row[b] = (b < nb) ? x * inv + shift : 0.f;
        }
        // x = 3 (missing call or absent site of a query, never in training): xhat = beta, BatchNorm's output at the
        // moving mean
        if (miss != 0ull)
          for (int b = 0; b < nb; ++b)
            if ((miss >> (2 * b)) & 1ull) row[b] = a.beta[k];
      } else {
        for (int b = 0; b < kMaxB; ++b) row[b] = 0.f;
      }
    }
    __syncthreads();
    if (tid < H) {
      const int tmax = (int)((a.K - k0) < kF1Chunk ? (a.K - k0) : kF1Chunk);
      const float* wp = a.W1 + k0 * H + tid;
#pragma unroll 4
      for (int t = 0; t < tmax; ++t) {
        const float w = __ldg(wp + (int64_t)t * H);
        const float* row = xh + t * (kMaxB + 1);
#pragma unroll
        for (int b = 0; b < kMaxB; ++b) acc[b] = fmaf(row[b], w, acc[b]);
      }
    }
    __syncthreads();
  }
  if (tid < H) {
    float* out = a.partials + (int64_t)blockIdx.x * kMaxB * H + tid;
#pragma unroll
    for (int b = 0; b < kMaxB; ++b) out[(int64_t)b * H] = acc[b];
  }
}

constexpr int kB1Chunk = 32;

__global__ void __launch_bounds__(1024) k_l1_bwd_simt(L1Args a) {
  if (a.gated && a.st->stopped) return;
  __shared__ float xs[kB1Chunk][kMaxB + 1];
  __shared__ float sc[kB1Chunk][4];            // inv, beta, rs
  __shared__ float pq[32][kB1Chunk][2];        // per-warp partial P, Q
  __shared__ int64_t s_rows[kMaxB];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nwarps = blockDim.x >> 5;
  const int H = a.H;
  const int nb = a.src.nb;
  if (tid < nb) s_rows[tid] = row_of(a.src, a.st, tid);
  __syncthreads();
  const float alpha = a.st->alpha;

  float dz[kMaxB];
  float c0 = 0.f;
#pragma unroll
  for (int b = 0; b < kMaxB; ++b) {
    dz[b] = (tid < H && b < nb) ? a.dZ1[b * H + tid] : 0.f;
    c0 += dz[b];
  }

  const int64_t nchunks = (a.K + kB1Chunk - 1) / kB1Chunk;
  const int64_t c_begin = nchunks * blockIdx.x / gridDim.x;
  const int64_t c_end = nchunks * (blockIdx.x + 1) / gridDim.x;
  for (int64_t c = c_begin; c < c_end; ++c) {
    const int64_t k0 = c * kB1Chunk;
    const int tmax = (int)((a.K - k0) < kB1Chunk ? (a.K - k0) : kB1Chunk);
    if (tid < tmax) {
      const int64_t k = k0 + tid;
      SnpBatch sb = load_snp(a.packed, a.row_words, s_rows, nb, k);
      float mean, var;
      batch_moments(sb, nb, mean, var);
      const float rs = rsqrtf(var + kBnEps);
      const float inv = rs * a.gamma[k];
      sc[tid][0] = inv;
      sc[tid][1] = a.beta[k];
      sc[tid][2] = rs;
      for (int b = 0; b < kMaxB; ++b) xs[tid][b] = b < nb ? (float)((sb.bits >> (2 * b)) & 3ull) - mean : 0.f;
    }
    __syncthreads();
    for (int t = 0; t < tmax; ++t) {
      float p = 0.f, q = 0.f;
      if (tid < H) {
        const int64_t idx = (k0 + t) * H + tid;
        float S = 0.f;
#pragma unroll
        for (int b = 0; b < kMaxB; ++b) S = fmaf(xs[t][b], dz[b], S);
        float w = a.W1[idx], m = a.mW1[idx], v = a.vW1[idx];
        const float g = sc[t][0] * S + sc[t][1] * c0;
        p = w * S;
        q = w * c0;
        adam_update(w, m, v, g, alpha);
        a.W1[idx] = w;
        a.mW1[idx] = m;
        a.vW1[idx] = v;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        p += __shfl_xor_sync(0xffffffffu, p, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
      }
      if (lane == 0) {
        pq[warp][t][0] = p;
        pq[warp][t][1] = q;
      }
    }
    __syncthreads();
    if (tid < tmax) {
      float P = 0.f, Q = 0.f;
      for (int w = 0; w < nwarps; ++w) {
        P += pq[w][tid][0];
        Q += pq[w][tid][1];
      }
      const int64_t k = k0 + tid;
      const float dgamma = sc[tid][2] * P;
      const float dbeta = Q;
      float gm = a.gamma[k], m = a.m_gamma[k], v = a.v_gamma[k];
      adam_update(gm, m, v, dgamma, alpha);
      a.gamma[k] = gm;
      a.m_gamma[k] = m;
      a.v_gamma[k] = v;
      float bt = a.beta[k];
      m = a.m_beta[k];
      v = a.v_beta[k];
      adam_update(bt, m, v, dbeta, alpha);
      a.beta[k] = bt;
      a.m_beta[k] = m;
      a.v_beta[k] = v;
    }
    __syncthreads();
  }
}

static int block_threads(int H) { return H < 64 ? 64 : H; }

int l1_forward_simt(const L1Args& a, int n_partials, cudaStream_t s) {
  LOC_CHECK(a.H % 32 == 0 && a.H >= 32 && a.H <= 1024, "first layer (simt): width must be a multiple of 32 in [32, 1024]");
  const size_t smem = (size_t)kF1Chunk * (kMaxB + 1) * sizeof(float);
  k_l1_fwd_simt<<<n_partials, block_threads(a.H), smem, s>>>(a, n_partials);
  LOC_LAUNCHED();
  return 0;
}

int l1_backward_simt(const L1Args& a, int nblocks, cudaStream_t s) {
  LOC_CHECK(a.H % 32 == 0 && a.H >= 32 && a.H <= 1024, "first layer (simt): width must be a multiple of 32 in [32, 1024]");
  k_l1_bwd_simt<<<nblocks, block_threads(a.H), 0, s>>>(a);
  LOC_LAUNCHED();
  return 0;
}

}  // namespace loc
