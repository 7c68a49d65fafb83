// First layer on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), width H = 256.
//
// Reference: BatchNormalization + Dense(256) forward / backward + Adam inside model.fit,
// locator/locator.py:318-320,367-376; algebra in l1_simt.cu's header.  Both kernels are HBM-bound
// streams over W1 (and m, v); the tensor cores remove the 2*32*256 FMA per SNP from the CUDA cores.
//
// FORWARD  (k_l1_fwd_tc), one persistent CTA per SM, split over SNPs:
//   D[j, b] += W1[k, j]^T * xhat[k, b]      M = 128 (two halves of j), N = 32 (batch), K = 8 SNPs / MMA
//   A = W1 tile.  W1 (and Adam's m, v) live in HBM in a chunk-tiled, pre-swizzled layout
//       (model.cuh: w1_tiled_index) -- blocks of 8 SNPs x 256 columns = 8 KB, inside a block
//       [8 j-chunks][8 SNP rows][128 B] with the 128B/32B-atom swizzle -- which IS the canonical
//       MN-major tf32 operand image: a stage is one contiguous 32 KB cp.async.bulk, no tensor map,
//       no conversion pass (kind::tf32 reads the fp32 master weights' bits).
//   B = xhat tile [32 SNP rows][32 batch = 128 B], built in shared memory by the builder warps from
//       the 2-bit genotypes with the folded BatchNorm (x*inv + shift), rounded to tf32.
//   warp 0: bulk-copy producer | warp 1: TMEM alloc + MMA issue | warps 2-5: operand builders, epilogue.
//   5-stage mbarrier ring; accumulators (2 x 32 columns) stay in TMEM for the whole K range; the
//   epilogue writes one [32][256] partial tile per CTA (reduced in fixed order by k_hidden).
//
// BACKWARD (k_l1_bwd_tc), one persistent CTA per SM, split over SNPs, 64 SNPs per tile:
//   S[j, k] = sum_b dZ1[b, j] * (x[b, k] - mean_k)   M = 128 (two halves of j), N = 64 SNPs, K = 8 rows / MMA
//   A = dZ1 as hi + lo tf32 parts (MN-major, swizzled, built once per CTA), B = centred genotypes
//   (K-major, swizzled; exact in tf32 for a power-of-two batch) -> S is fp32-accurate.
//   W1, m, v never touch the load/store units' global path: a load thread streams 8-SNP chunks
//   (3 x 8 KB, contiguous rows, L2 evict_first) into a 5-stage shared-memory ring with cp.async.bulk +
//   mbarrier, the epilogue warps (accumulator row j = TMEM lane, so a warp reads/writes 128 contiguous
//   bytes of a row: conflict-free) apply Adam in place, and a store thread writes the chunk back with
//   cp.async.bulk; dW1 never exists in memory.  P_k, Q_k (for dgamma, dbeta) are reduced with a
//   butterfly transpose across the warp and summed across warps in fixed order.
//   (A 6-stage ring with a single-pass tf32 dZ1 was measured: no faster, so the hi/lo split stays.)
//   Odd steps walk each CTA's tiles downwards: the tail of the previous step's updates is still in L2.
//   Fused runs (L1Args::fuse_next) also compute the NEXT step's forward partial tile from every freshly
//   updated chunk while it is in shared memory (two forward warps, own TMEM columns).
//   warps 0-15: epilogue (two groups alternating chunks) | 16-17: genotype unpack / BN statistics /
//   gamma-beta Adam (unfused runs), MMA issue | 18: bulk loads | 19: bulk stores | 20-21: forward warps.
#include <stdlib.h>

#include "l1_common.cuh"

namespace loc {
namespace tc {

constexpr int kH = 256;

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// generic-proxy shared-memory writes -> visible to the async proxy (tensor core / TMA)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// D[tmem] (+)= A[smem] * B[smem], kind::tf32 (fp32 bits in shared memory, fp32 accumulate).
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once every tcgen05.mma issued so far by this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout).
//   kLayoutSw128    : K-major operands, 16-byte chunks XOR (row & 7) within 128-byte rows
//   kLayoutSw128B32 : MN-major tf32 operands -- the only swizzle the tensor core accepts for them:
//                     32-byte chunks XOR (row & 3) within 128-byte rows (TMA: SWIZZLE_128B_ATOM_32B);
//                     LBO = bytes between 32-element MN chunks, SBO = bytes between 4-row K groups
constexpr uint32_t kLayoutSw128 = 2, kLayoutSw128B32 = 1;
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  d |= (uint64_t)layout << 61;
  return d;
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): tf32 x tf32 -> f32.
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void tmem_ld_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// One lane of a converged warp (elect.sync): the compiler then emits the uniform-datapath
// tcgen05 / bulk-copy instructions directly instead of a per-active-lane loop around each of them.
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

// Row r of a swizzled [rows][128 B] tile, logical 16-byte chunk c:
//   swz   (K-major SWIZZLE_128B):            chunk c lives at c ^ (r & 7)
//   swz32 (MN-major SWIZZLE_128B, 32B atom): the 32-byte pair (c >> 1) lives at (c >> 1) ^ (r & 3)
__device__ __forceinline__ uint32_t swz(int r, int c) { return (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }
__device__ __forceinline__ uint32_t swz32(int r, int c) {
  return (uint32_t)(r * 128 + (((((c >> 1) ^ (r & 3)) << 1) | (c & 1)) << 4));
}

// Split of the 64-SNP tiles over the CTAs of a first-layer kernel: the first (ntiles % grid) CTAs take one tile
// more than the others.  The CTAs with the smaller share are the LAST ones: in a chained step (model.cu:
// train_step) the hidden stack still holds 16 SMs when the backward is launched, and the CTAs that have to wait
// for those SMs -- the last ones the block scheduler hands out -- then finish no later than the rest.
__device__ __forceinline__ void tile_range(int64_t ntiles, int64_t& t_begin, int64_t& t_end) {
#if LOC_SPLIT_INTERLEAVED  // A/B: the shares of q and q + 1 tiles interleaved over the CTAs
  t_begin = ntiles * blockIdx.x / gridDim.x;
  t_end = ntiles * (blockIdx.x + 1) / gridDim.x;
#else
  const int64_t q = ntiles / gridDim.x, rem = ntiles % gridDim.x, b = blockIdx.x;
  t_begin = b * q + (b < rem ? b : rem);
  t_end = t_begin + q + (b < rem ? 1 : 0);
#endif
}

// ---------------------------------------------------------------------------------------------
// Forward
// ---------------------------------------------------------------------------------------------
constexpr int F_KT = 32;                              // SNPs per stage
constexpr int F_STAGES = 6;
constexpr int F_THREADS = 192;                        // 6 warps
constexpr int F_WBYTES = F_KT * kH * 4;               // 32 KB: 4 blocks of [8 j-chunks][8 rows][128 B]
constexpr int F_CHUNK = F_KT * 128;                   // bytes between j-chunks (LBO)
constexpr int F_XBYTES = F_KT * 128;                  // 4 KB:  [32 rows][32 batch]
constexpr int F_SMEM = F_STAGES * (F_WBYTES + F_XBYTES) + 4 * 32 * 8 + 256 + 1024;  // + bits scratch + barriers + align

__global__ void __launch_bounds__(F_THREADS, 1) k_l1_fwd_tc(L1Args a, int64_t ntiles) {
  if (a.gated && a.st->stopped) return;
  if (threadIdx.x == 0 && blockIdx.x == 0) tl_mark(a.tl, 7u, (unsigned)a.tl_id);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* sW = sm;
  uint8_t* sX = sW + F_STAGES * F_WBYTES;
  uint32_t* sBits = (uint32_t*)(sX + F_STAGES * F_XBYTES);  // [4 warps][32 rows][2 words]
  uint64_t* bars = (uint64_t*)(sBits + 4 * 32 * 2);
  uint64_t* full_w = bars;
  uint64_t* full_x = bars + F_STAGES;
  uint64_t* empty = bars + 2 * F_STAGES;
  uint64_t* done = bars + 3 * F_STAGES;
  uint32_t* tmem_slot = (uint32_t*)(bars + 3 * F_STAGES + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nb = a.src.nb;
  // ntiles counts 64-SNP tiles (the backward kernel's unit) so both kernels split K identically
  int64_t t_begin, t_end;
  tile_range(ntiles, t_begin, t_end);
  t_begin *= 2;  // 32-SNP stages
  t_end *= 2;
  const int nloc = (int)(t_end - t_begin);

  if (threadIdx.x == 0) {
    for (int s = 0; s < F_STAGES; ++s) {
      mbar_init(&full_w[s], 1);
      mbar_init(&full_x[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(done, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 64);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ---- TMA producer ----
    if (elect_one()) {
      for (int li = 0; li < nloc; ++li) {
        const int s = li % F_STAGES;
        const uint32_t ph = (uint32_t)(li / F_STAGES) & 1u;
        mbar_wait(&empty[s], ph ^ 1u);
        mbar_arrive_expect_tx(&full_w[s], F_WBYTES);
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         smem_u32(sW + s * F_WBYTES)),
                     "l"(a.W1 + (t_begin + li) * (int64_t)(F_KT * kH)), "r"((uint32_t)F_WBYTES), "r"(smem_u32(&full_w[s]))
                     : "memory");
      }
    }
  } else if (warp == 1) {
    // ---- MMA issuer ----
    constexpr uint32_t idesc = make_idesc(128, 32, 1, 1);
    if (elect_one()) {
      for (int li = 0; li < nloc; ++li) {
        const int s = li % F_STAGES;
        const uint32_t ph = (uint32_t)(li / F_STAGES) & 1u;
        mbar_wait(&full_w[s], ph);
        mbar_wait(&full_x[s], ph);
        tc_fence_after();
        const uint32_t wbase = smem_u32(sW + s * F_WBYTES), xbase = smem_u32(sX + s * F_XBYTES);
#pragma unroll
        for (int ks = 0; ks < F_KT / 8; ++ks) {
          const uint64_t bdesc = smem_desc(xbase + ks * 1024, F_CHUNK, 512, kLayoutSw128B32);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const uint64_t adesc = smem_desc(wbase + ks * 8192 + h * 4096, 1024, 512, kLayoutSw128B32);
            umma_tf32(tmem + h * 32, adesc, bdesc, idesc, (li > 0 || ks > 0) ? 1u : 0u);
          }
        }
        umma_commit(&empty[s]);
      }
      umma_commit(done);
    }
  } else {
    // ---- operand builders (warps 2..5), then epilogue ----
    const int wi = warp - 2;
    uint32_t* bits = sBits + wi * 64;
    const int64_t my_row = lane < nb ? row_of(a.src, a.st, lane) : 0;
    const uint32_t* my_ptr = a.packed + my_row * a.row_words;
    // the global loads of a stage -- lane <-> batch row: the row's 32 genotypes of the tile (2 words); lane <-> SNP: the
    // SNP's parameters -- are requested one of the warp's stages ahead (they sat on its critical path once per stage)
    struct StageIn {
      uint2 w2;
      float gamma, beta, mm, mv;
    };
    auto stage_in = [&](int li) {
      StageIn r;
      const int64_t tile = t_begin + li;
      r.w2 = make_uint2(0u, 0u);
      if (lane < nb && tile * 2 + 1 < a.row_words) r.w2 = __ldg(reinterpret_cast<const uint2*>(my_ptr + tile * 2));
      const int64_t k = tile * F_KT + lane;
      r.gamma = r.beta = r.mm = 0.f;
      r.mv = 1.f;
      if (k < a.K) {
        r.gamma = a.gamma[k];
        r.beta = a.beta[k];
        r.mm = a.mmean[k];  // (read before this thread's own update of the same element below; nobody else touches it)
        r.mv = a.mvar[k];
      }
      return r;
    };
    StageIn nxt;
    if (wi < nloc) nxt = stage_in(wi);
    for (int li = wi; li < nloc; li += 4) {
      const int s = li % F_STAGES;
      const uint32_t ph = (uint32_t)(li / F_STAGES) & 1u;
      const int64_t tile = t_begin + li;
      const StageIn cur = nxt;
      if (li + 4 < nloc) nxt = stage_in(li + 4);
      const uint2 w2 = cur.w2;
      const int64_t k = tile * F_KT + lane;
      const bool valid = k < a.K;
      const float gamma = cur.gamma, beta = cur.beta, mm = cur.mm, mv = cur.mv;
      bits[lane * 2] = w2.x;
      bits[lane * 2 + 1] = w2.y;
      __syncwarp();
      const int wsel = lane >> 4, sh = 2 * (lane & 15);
      unsigned long long g = 0ull;
      int n1 = 0, n2 = 0;
#pragma unroll
      for (int b = 0; b < kMaxB; ++b) {
        const unsigned x = (bits[b * 2 + wsel] >> sh) & 3u;  // rows >= nb hold zeros
        g |= (unsigned long long)x << (2 * b);
        n1 += (x == 1u);
        n2 += (x == 2u);
      }
      __syncwarp();
      float mean, var;
      float miss = 0.f;  // x = 3 (missing call or absent site of a query, never in training): xhat = beta
      if (a.training) {
        moments_from_counts(n1, n2, nb, mean, var);
        if (valid) {
          a.mmean[k] = mm * kBnMom + mean * kBnOneMinusMom;
          a.mvar[k] = mv * kBnMom + var * kBnOneMinusMom;
        }
      } else {
        mean = mm;
        var = mv;
        miss = valid ? to_tf32(beta) : 0.f;
      }
      const float inv = rsqrtf(var + kBnEps) * gamma;
      const float shift = beta - mean * inv;
      float lut[3];
      lut[0] = valid ? to_tf32(shift) : 0.f;
      lut[1] = valid ? to_tf32(inv + shift) : 0.f;
      lut[2] = valid ? to_tf32(2.f * inv + shift) : 0.f;
      mbar_wait(&empty[s], ph ^ 1u);
      uint8_t* xrow = sX + s * F_XBYTES;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int b = 4 * c + e;
          const unsigned x = (unsigned)((g >> (2 * b)) & 3ull);
          // branch-free select (the lanes of a warp hold different genotypes)
          const float val = (x & 2u) ? ((x & 1u) ? miss : lut[2]) : ((x & 1u) ? lut[1] : lut[0]);
          v[e] = b < nb ? val : 0.f;
        }
        *reinterpret_cast<float4*>(xrow + swz32(lane, c)) = make_float4(v[0], v[1], v[2], v[3]);
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full_x[s]);
    }
    // ---- epilogue: accumulator row = j (TMEM lane), column = batch row ----
    mbar_wait(done, 0);
    tc_fence_after();
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    float* out = a.partials + (int64_t)blockIdx.x * kMaxB * kH;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint32_t r[32];
      tmem_ld_x32(tmem + ((uint32_t)(32 * q) << 16) + (uint32_t)(h * 32), r);
      tmem_ld_wait();
      const int j = h * 128 + 32 * q + lane;
#pragma unroll
      for (int b = 0; b < kMaxB; ++b) out[b * kH + j] = __uint_as_float(r[b]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 64);
  if (threadIdx.x == 0 && blockIdx.x == 0) tl_mark(a.tl, 8u, (unsigned)a.tl_id);
}


// ---------------------------------------------------------------------------------------------
// Wide inference forward (validation / prediction / jacknife sweeps): up to 256 rows per pass over W1
// ---------------------------------------------------------------------------------------------
// model.predict / the validation pass of model.fit (locator.py:374,414,441) only need Z1 = xhat * W1 with the
// moving statistics; the reference runs them at batch 32 and so did this library: one full stream of W1 per 32
// rows.  Here the batch axis of the MMA is N = 32..256 (D[j, b], M = 128 x 2 halves, K = 8 SNPs per MMA, both
// accumulators of N columns in TMEM: 512 columns at N = 256), so W1 is streamed ONCE per 256 rows: 8 builder
// warps each turn one 32-row chunk of the packed genotypes into its [32 SNPs][32 rows] slice of the MN-major
// B operand (chunks are LBO = 4 KB apart), per 32-SNP stage.  At N = 256 a stage is 8 MMAs of 128 x 256 x 8
// (about 1,024 tensor-core cycles) against 32 KB of W1 (about 1,400 cycles of this SM's share of HBM): the
// sweep sits at the crossover of the two rooflines instead of 8x under the memory one.
constexpr int W_STAGES = 3;
constexpr int W_XBYTES = 8 * F_XBYTES;           // 32 KB: [8 chunks of 32 rows][32 SNP rows][128 B]
constexpr int W_BUILD = 8;                        // builder warps = max 32-row chunks
constexpr int W_THREADS = (2 + W_BUILD) * 32;     // producer, MMA issuer, builders (also the epilogue)
constexpr int W_SMEM = W_STAGES * (F_WBYTES + W_XBYTES) + W_BUILD * 32 * 16 + 256 + 1024;

__global__ void __launch_bounds__(W_THREADS, 1) k_l1_fwd_wide(L1Args a, int64_t ntiles, int nrows, float* __restrict__ out) {
  if (a.gated && a.st->stopped) return;
  if (threadIdx.x == 0 && blockIdx.x == 0) tl_mark(a.tl, 9u, (unsigned)a.tl_id);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* sW = sm;
  uint8_t* sX = sW + W_STAGES * F_WBYTES;
  uint32_t* sBits = (uint32_t*)(sX + W_STAGES * W_XBYTES);  // [8 warps][32 SNPs][4 floats]: per-SNP value tables
  uint64_t* bars = (uint64_t*)(sBits + W_BUILD * 32 * 4);
  uint64_t* full_w = bars;
  uint64_t* full_x = bars + W_STAGES;
  uint64_t* empty = bars + 2 * W_STAGES;
  uint64_t* done = bars + 3 * W_STAGES;
  uint32_t* tmem_slot = (uint32_t*)(bars + 3 * W_STAGES + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int NC = (nrows + 31) >> 5, N = NC * 32;  // 32-row chunks, MMA N
  int64_t t_begin, t_end;
  tile_range(ntiles, t_begin, t_end);
  t_begin *= 2;  // 32-SNP stages
  t_end *= 2;
  const int nloc = (int)(t_end - t_begin);

  if (threadIdx.x == 0) {
    for (int s = 0; s < W_STAGES; ++s) {
      mbar_init(&full_w[s], 1);
      mbar_init(&full_x[s], (uint32_t)NC);
      mbar_init(&empty[s], 1);
    }
    mbar_init(done, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      for (int li = 0; li < nloc; ++li) {
        const int s = li % W_STAGES;
        const uint32_t ph = (uint32_t)(li / W_STAGES) & 1u;
        mbar_wait(&empty[s], ph ^ 1u);
        mbar_arrive_expect_tx(&full_w[s], F_WBYTES);
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         smem_u32(sW + s * F_WBYTES)),
                     "l"(a.W1 + (t_begin + li) * (int64_t)(F_KT * kH)), "r"((uint32_t)F_WBYTES), "r"(smem_u32(&full_w[s]))
                     : "memory");
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = make_idesc(128, N, 1, 1);
    if (elect_one()) {
      for (int li = 0; li < nloc; ++li) {
        const int s = li % W_STAGES;
        const uint32_t ph = (uint32_t)(li / W_STAGES) & 1u;
        mbar_wait(&full_w[s], ph);
        mbar_wait(&full_x[s], ph);
        tc_fence_after();
        const uint32_t wbase = smem_u32(sW + s * F_WBYTES), xbase = smem_u32(sX + s * W_XBYTES);
#pragma unroll
        for (int ks = 0; ks < F_KT / 8; ++ks) {
          // B: MN-major, N = NC chunks of 32 rows, F_CHUNK (4 KB) apart; 8 SNP rows of this k-step at ks * 1 KB
          const uint64_t bdesc = smem_desc(xbase + ks * 1024, F_CHUNK, 512, kLayoutSw128B32);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const uint64_t adesc = smem_desc(wbase + ks * 8192 + h * 4096, 1024, 512, kLayoutSw128B32);
            umma_tf32(tmem + (uint32_t)(h * N), adesc, bdesc, idesc, (li > 0 || ks > 0) ? 1u : 0u);
          }
        }
        umma_commit(&empty[s]);
      }
      umma_commit(done);
    }
  } else {
    // ---- builders: warp wi owns the 32-row chunk wi (rows 32 wi .. 32 wi + 31 of this pass) ----
    const int wi = warp - 2;
    if (wi < NC) {
      float4* lutw = reinterpret_cast<float4*>(sBits) + wi * 32;  // this warp's table: [32 SNPs]{x = 0, 1, 2, -}
      const int b_row = wi * 32 + lane;             // row of the pass this lane loads
      const bool row_ok = b_row < nrows;
      const int nb_chunk = nrows - wi * 32 < 32 ? nrows - wi * 32 : 32;
      const int64_t my_row = row_ok ? row_of(a.src, a.st, b_row) : 0;
      const uint32_t* my_ptr = a.packed + my_row * a.row_words;
      // One warp builds every stage of its chunk, so the global loads of a stage (the row's 32 genotypes, the SNPs'
      // parameters) would sit on its critical path once per stage: they are requested one stage ahead.
      struct StageIn {
        uint2 w2;
        float gamma, beta, mm, mv;
      };
      auto stage_in = [&](int li) {
        StageIn r;
        const int64_t tile = t_begin + li;
        r.w2 = make_uint2(0u, 0u);
        if (row_ok && tile * 2 + 1 < a.row_words) r.w2 = __ldg(reinterpret_cast<const uint2*>(my_ptr + tile * 2));
        const int64_t k = tile * F_KT + lane;
        r.gamma = r.beta = r.mm = 0.f;
        r.mv = 1.f;
        if (k < a.K) {
          r.gamma = __ldg(a.gamma + k);
          r.beta = __ldg(a.beta + k);
          r.mm = __ldg(a.mmean + k);
          r.mv = __ldg(a.mvar + k);
        }
        return r;
      };
      StageIn nxt = stage_in(0);
      for (int li = 0; li < nloc; ++li) {
        const int s = li % W_STAGES;
        const uint32_t ph = (uint32_t)(li / W_STAGES) & 1u;
        const int64_t tile = t_begin + li;
        const StageIn cur = nxt;
        if (li + 1 < nloc) nxt = stage_in(li + 1);
        const uint2 w2 = cur.w2;
        const int64_t k = tile * F_KT + lane;
        const bool valid = k < a.K;
        const float gamma = cur.gamma, beta = cur.beta, mm = cur.mm, mv = cur.mv;
        // lane <-> SNP: the three values a genotype of this SNP can take, shared through a per-warp table; then
        // lane <-> batch row: every lane walks its own row's 32 genotypes (they are in its registers) and writes one
        // element per SNP row of the operand tile -- a 128-byte row per store instruction, conflict-free.  (The first
        // version transposed the genotypes through shared memory instead, 32 loads + ~130 integer instructions per
        // lane and stage: 23 % of the kernel's samples.)
        const float inv = rsqrtf(mv + kBnEps) * gamma;  // inference: moving statistics
        // fused as it always was: beta's use in the code-3 slot below would otherwise leave it a multiply and a
        // subtraction, and move the tf32 images of the three genotype values
        const float shift = fmaf(-mm, inv, beta);
        __syncwarp();  // the previous stage's table has been read by every lane
        // x = 3 (missing call or absent site of a query): xhat = beta, BatchNorm's output at the moving mean
        lutw[lane] = make_float4(valid ? to_tf32(shift) : 0.f, valid ? to_tf32(inv + shift) : 0.f,
                                 valid ? to_tf32(2.f * inv + shift) : 0.f, valid ? to_tf32(beta) : 0.f);
        __syncwarp();
        mbar_wait(&empty[s], ph ^ 1u);
        uint8_t* xrow = sX + s * W_XBYTES + wi * F_CHUNK + (lane & 3) * 4;
        const float* lutf = reinterpret_cast<const float*>(lutw);
        const bool row_on = lane < nb_chunk;
        uint32_t off4[4];  // swz32(k, lane >> 2) - 128 k only depends on k & 3
#pragma unroll
        for (int q = 0; q < 4; ++q) off4[q] = swz32(q, lane >> 2) - 128u * q;
        // (all table reads first, then all stores: through these generic pointers the compiler must keep a store and
        // the next load in order, and 32 dependent load -> store round trips cost a microsecond per stage)
        float vals[F_KT];
#pragma unroll
        for (int k = 0; k < F_KT; ++k) {
          const unsigned x = ((k < 16 ? w2.x : w2.y) >> (2 * (k & 15))) & 3u;
          vals[k] = lutf[4 * k + x];
        }
#pragma unroll
        for (int k = 0; k < F_KT; ++k) *reinterpret_cast<float*>(xrow + 128 * k + off4[k & 3]) = row_on ? vals[k] : 0.f;
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&full_x[s]);
      }
    }
    // ---- epilogue: warps 2-5 take half 0, warps 6-9 half 1; accumulator row = j (TMEM lane), column = row of the pass
    mbar_wait(done, 0);
    tc_fence_after();
    const int q = warp & 3, h = wi >> 2;
    float* o = out + (int64_t)blockIdx.x * N * kH + (h * 128 + 32 * q + lane);
    for (int c = 0; c < NC; ++c) {
      uint32_t r[32];
      tmem_ld_x32(tmem + ((uint32_t)(32 * q) << 16) + (uint32_t)(h * N + c * 32), r);
      tmem_ld_wait();
#pragma unroll
      for (int b = 0; b < 32; ++b) o[(int64_t)(c * 32 + b) * kH] = __uint_as_float(r[b]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
  if (threadIdx.x == 0 && blockIdx.x == 0) tl_mark(a.tl, 10u, (unsigned)a.tl_id);
}

// ---------------------------------------------------------------------------------------------
// Backward + Adam
// ---------------------------------------------------------------------------------------------
#ifndef LOC_SPLIT_INTERLEAVED
#define LOC_SPLIT_INTERLEAVED 0
#endif
#ifndef LOC_FWD_WARPS
#define LOC_FWD_WARPS 4  // forward warps of the fused backward (2 or 4): each takes every LOC_FWD_WARPS-th chunk
#endif
constexpr int B_NT = 64;                       // SNPs per tile (one accumulator buffer)
constexpr int B_CH = 8;                        // SNPs per streamed chunk (one W/m/v stage)
constexpr int B_STAGES = 5;
constexpr int B_RING = 2 * B_STAGES;             // barrier ring: one per (epilogue group, stage)
constexpr int B_EPI_WARPS = 16;                // two groups of 8: group g owns the chunks with index % 2 == g
constexpr int B_NFW = LOC_FWD_WARPS;            // forward warps (fused runs)
constexpr int B_THREADS = (B_EPI_WARPS + 4 + B_NFW) * 32;  // + 2 builder warps, load warp, store warp, forward warps
// warp roles after the epilogue warps and the two builder warps; the forward warps land on different schedulers
constexpr int W_LOAD = B_EPI_WARPS + 2, W_STORE = B_EPI_WARPS + 3, W_FWD0 = B_EPI_WARPS + 4;
static_assert(B_NFW == 2 || B_NFW == 4, "forward warps: 2 or 4 (TMEM columns 256 + 64 per warp)");
constexpr int B_DZ = kMaxB * kH * 4;           // 32 KB: [8 chunks][32 rows (b)][128 B]
constexpr int B_DZ_CHUNK = kMaxB * 128;        // 4096
constexpr int B_X = B_NT * 128;                // 8 KB: [64 rows (SNP)][32 batch]
constexpr int B_ARR = B_CH * kH * 4;           // 8 KB: one array's rows of a chunk
constexpr int B_STAGE = 3 * B_ARR;             // 24 KB: W | m | v
constexpr int B_XF = 8 * 128;                  // 1 KB: next batch's xhat rows of one chunk [8 SNP rows][32 batch]
constexpr int B_SMEM = 2 * B_DZ + 2 * B_X + B_STAGES * (B_STAGE + B_XF) + 2 * B_NT * 16 + 2 * 8 * B_NT * 8 + 2 * 32 * 8 + 512 + 1024;

// Keras Adam with hardware approximations for the root and the quotient (both ~1 ulp of fp32:
// far below the tf32 rounding of the gradient products; the IEEE sqrt was 27% of this kernel's
// instruction stream)
__device__ __forceinline__ void adam_update_fast(float& w, float& m, float& v, float g, float alpha) {
  m = m + (g - m) * kAdam1mB1;
  v = v + (g * g - v) * kAdam1mB2;
  float rt;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(rt) : "f"(v));
  w = w - __fdividef(m * alpha, rt + kAdamEps);
}

// L2 evict_first as the 64-bit cache-policy operand of the bulk copies (the value
// createpolicy.fractional.L2::evict_first produces for fraction 1.0)
constexpr uint64_t kL2EvictFirst = 0x12F0000000000000ull;

__device__ __forceinline__ void bulk_load(uint32_t smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar, uint64_t pol) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                   smem_dst),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void bulk_store(void* gdst, uint32_t smem_src, uint32_t bytes, uint64_t pol) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(gdst), "r"(smem_src),
               "r"(bytes), "l"(pol)
               : "memory");
}

__global__ void __launch_bounds__(B_THREADS, 1) k_l1_bwd_tc(L1Args a, int64_t ntiles) {
  // programmatic dependent launch: a kernel queued behind this one with the programmatic-serialization
  // attribute (the small-layer update of the ring schedule) may be scheduled as soon as every CTA is running
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (a.gated && a.st->stopped) {  // past the stopping epoch: a no-op that still keeps the hand-over counter in step
    if (threadIdx.x == 0) atomicAdd(&a.st->bwd_cnt, 1u);
    return;
  }
  if (threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1)) tl_mark(a.tl, blockIdx.x ? 17u : 1u, (unsigned)a.tl_id);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* sDZhi = sm;
  uint8_t* sDZlo = sDZhi + B_DZ;
  uint8_t* sXhi = sDZlo + B_DZ;                  // [2][B_X]
  uint8_t* sStage = sXhi + 2 * B_X;              // [B_STAGES][W | m | v][8 rows][256]
  uint8_t* sXf = sStage + B_STAGES * B_STAGE;    // [B_STAGES][1 KB] forward B operand of the chunk in the stage
  float4* sSc = (float4*)(sXf + B_STAGES * B_XF);  // [2][64] (inv, beta, rs, -)
  float2* sRed = (float2*)(sSc + 2 * B_NT);      // [2][8 warps][64] (P, Q) partial sums
  uint32_t* sBits = (uint32_t*)(sRed + 2 * 8 * B_NT);  // [2 builder warps][32 rows][2 words]
  uint64_t* bars = (uint64_t*)(sBits + 2 * 32 * 2);
  uint64_t* tmem_full = bars;                    // [2]  MMA of a tile done
  uint64_t* tmem_empty = bars + 2;               // [2]  all 16 epilogue warps done with a tile
  // st_full / st_done are indexed by chunk % B_RING (= stage and epilogue group together): the waiters of a
  // chunk alternate between the two epilogue groups / forward warps, and B_STAGES is odd, so a barrier per
  // stage would be waited on by a warp that never observed the stage's previous phase -- a parity wait then
  // passes while that previous use is still in flight.  With one barrier per (group, stage) every waiter
  // sees every phase of its barriers in order.
  uint64_t* st_full = bars + 4;                  // [B_RING] W/m/v chunk landed
  uint64_t* st_done = st_full + B_RING;          // [B_RING] chunk updated in place (8 warps)
  uint64_t* st_free = st_done + B_RING;          // [B_STAGES] chunk written back, stage reusable (load warp, in order)
  uint64_t* fwd_done = st_free + B_STAGES;       // forward accumulators complete (fused runs)
  uint64_t* fwd_tile = fwd_done + 1;             // [2] both forward warps have read a tile's scales / row sums
  uint32_t* tmem_slot = (uint32_t*)(fwd_tile + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nb = a.src.nb;
  const bool fuse = a.fuse_next != 0;  // also run the NEXT step's forward on the freshly updated chunks
  int64_t t_begin, t_end;
  tile_range(ntiles, t_begin, t_end);
  const int nloc = (int)(t_end - t_begin);
  const int nchunks = nloc * (B_NT / B_CH);
  // odd steps walk the tiles downwards (L1Args::rev); chunks inside a tile keep their order
  auto tile_of = [&](int li) -> int64_t { return t_begin + (a.rev ? nloc - 1 - li : li); };

  if (threadIdx.x == 0) {
    mbar_init(&tmem_full[0], 1);
    mbar_init(&tmem_full[1], 1);
    mbar_init(&tmem_empty[0], B_EPI_WARPS);
    mbar_init(&tmem_empty[1], B_EPI_WARPS);
    for (int s = 0; s < B_RING; ++s) {
      mbar_init(&st_full[s], 1);
      mbar_init(&st_done[s], 8);
    }
    for (int s = 0; s < B_STAGES; ++s) mbar_init(&st_free[s], fuse ? 2 : 1);  // written back (+ consumed by the forward MMA)
    mbar_init(fwd_done, B_NFW);  // one commit per forward warp
    mbar_init(&fwd_tile[0], B_NFW);
    mbar_init(&fwd_tile[1], B_NFW);
    fence_barrier_init();
  }
  if (warp == B_EPI_WARPS) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();  // barriers and TMEM are ready: the load warp starts streaming W1 | m | v right away ...
  tc_fence_after();
  if (warp != W_LOAD) {
    // Launched ahead of this step's hidden stack (programmatic dependent launch: the set-up above and the first
    // ring stages of W1 | m | v run in its shadow): dZ1, alpha and the loss only exist once it has published.
    if (a.wait_hid != 0) {
      // ONE poller per CTA (2,700 polling warps on one L2 line slowed the very hidden stack they were waiting for)
      if (threadIdx.x == 0) wait_counter(&a.st->hid_seq, a.wait_hid, &a.st->chain_timeout);
      asm volatile("bar.sync 4, %0;" ::"n"(B_THREADS - 32) : "memory");  // everyone but the load warp
    }
    // ... while everybody else stages dZ1 -> hi/lo tf32 operands, [chunk = j/32][row = b][swizzled 32 j]
    // (all of a thread's loads first: one L2 round trip instead of three)
    constexpr int kIters = (kMaxB * kH / 4 + B_THREADS - 33) / (B_THREADS - 32);
    const int t = threadIdx.x < W_LOAD * 32 ? threadIdx.x : threadIdx.x - 32;  // skip the load warp
    float4 v[kIters];
#pragma unroll
    for (int it = 0; it < kIters; ++it) {
      const int i = t + it * (B_THREADS - 32);
      const int b = i / (kH / 4), j4 = (i % (kH / 4)) * 4;
      v[it] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < kMaxB * kH / 4 && b < nb) v[it] = __ldcg(reinterpret_cast<const float4*>(a.dZ1 + b * kH + j4));
    }
#pragma unroll
    for (int it = 0; it < kIters; ++it) {
      const int i = t + it * (B_THREADS - 32);
      if (i >= kMaxB * kH / 4) break;
      const int b = i / (kH / 4), j4 = (i % (kH / 4)) * 4;
      const float4 hi = make_float4(to_tf32(v[it].x), to_tf32(v[it].y), to_tf32(v[it].z), to_tf32(v[it].w));
      const float4 lo = make_float4(to_tf32(v[it].x - hi.x), to_tf32(v[it].y - hi.y), to_tf32(v[it].z - hi.z),
                                    to_tf32(v[it].w - hi.w));
      const uint32_t off = (uint32_t)((j4 >> 5) * B_DZ_CHUNK) + swz32(b, (j4 & 31) >> 2);
      *reinterpret_cast<float4*>(sDZhi + off) = hi;
      *reinterpret_cast<float4*>(sDZlo + off) = lo;
    }
    fence_proxy_async();
    asm volatile("bar.sync 3, %0;" ::"n"(B_THREADS - 32) : "memory");  // everyone but the load warp
  }
  const uint32_t tmem = *tmem_slot;
  const float alpha = a.st->alpha;
  if (warp < B_EPI_WARPS) {
    // =========================== epilogue warps ===========================
    const int grp = warp >> 3, w8 = warp & 7;
    const int h = w8 >> 2, q = w8 & 3;
    const int j = h * 128 + q * 32 + lane;
    float c0 = 0.f;
    {  // all loads in flight at once; summed in row order
      float dz[kMaxB];
#pragma unroll
      for (int b = 0; b < kMaxB; ++b) dz[b] = b < nb ? __ldcg(a.dZ1 + b * kH + j) : 0.f;
#pragma unroll
      for (int b = 0; b < kMaxB; ++b) c0 += dz[b];
    }
    for (int c = grp; c < nchunks; c += 2) {
      const int li = c >> 3, cc = c & 7;
      const int buf = li & 1;
      const int s = c % B_STAGES;
      if (cc < 2) {  // first chunk of the tile for this group
        mbar_wait(&tmem_full[buf], (uint32_t)(li >> 1) & 1u);
        tc_fence_after();
      }
      uint32_t gr[8];
      tmem_ld_x8(tmem + ((uint32_t)(32 * q) << 16) + (uint32_t)(buf * 128 + h * 64 + cc * 8), gr);
      mbar_wait(&st_full[c % B_RING], (uint32_t)(c / B_RING) & 1u);
      // element (row r, column j) of a chunk block: [j/32][r][32B atoms XOR (r & 3)] (w1_tiled_index)
      float* stw = reinterpret_cast<float*>(sStage + s * B_STAGE) + ((j >> 5) << 8) + (j & 7);
      const int j8 = (j & 31) >> 3;
      float w[8], m[8], v[8];
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const int o = (r << 5) + ((j8 ^ (r & 3)) << 3);
        w[r] = stw[o];
        m[r] = stw[B_ARR / 4 + o];
        v[r] = stw[2 * (B_ARR / 4) + o];
      }
      tmem_ld_wait();
      float pq[16];
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const float4 sc = sSc[buf * B_NT + cc * 8 + r];
        const float S = __uint_as_float(gr[r]);
        const float g = sc.x * S + sc.y * c0;
        pq[r] = w[r] * S;  // padding rows (k >= K) hold zeros and stay zero
        pq[8 + r] = w[r] * c0;
        adam_update_fast(w[r], m[r], v[r], g, alpha);
      }
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const int o = (r << 5) + ((j8 ^ (r & 3)) << 3);
        stw[o] = w[r];
        stw[B_ARR / 4 + o] = m[r];
        stw[2 * (B_ARR / 4) + o] = v[r];
      }
      fence_proxy_async();  // the bulk store reads these rows through the async proxy
      // butterfly transpose-reduce: lane l ends with the warp total of pq[l & 15]
#pragma unroll
      for (int o = 8; o >= 1; o >>= 1) {
        const bool up = (lane & o) != 0;
#pragma unroll
        for (int i = 0; i < o; ++i) {
          const float send = up ? pq[i] : pq[i + o];
          const float keep = up ? pq[i + o] : pq[i];
          pq[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
      }
      pq[0] += __shfl_xor_sync(0xffffffffu, pq[0], 16);
      if (lane < 16) {
        float* dst = reinterpret_cast<float*>(&sRed[(buf * 8 + w8) * B_NT + cc * 8 + (lane & 7)]);
        dst[lane >> 3] = pq[0];
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&st_done[c % B_RING]);
      if (cc >= 6) {  // last chunk of the tile for this group
        tc_fence_before();
        if (lane == 0) mbar_arrive(&tmem_empty[buf]);
      }
    }
    if (fuse && grp == 0) {  // next step's split-K partial tile of Z1: accumulator row = j, column = batch row
      mbar_wait(fwd_done, 0);
      tc_fence_after();
      // the forward warps accumulated into their own TMEM columns: added here in warp order
      float acc[32];
#pragma unroll
      for (int w = 0; w < B_NFW; ++w) {
        uint32_t r32[32];
        tmem_ld_x32(tmem + ((uint32_t)(32 * q) << 16) + (uint32_t)(256 + w * 64 + h * 32), r32);
        tmem_ld_wait();
#pragma unroll
        for (int b = 0; b < kMaxB; ++b) acc[b] = w == 0 ? __uint_as_float(r32[b]) : acc[b] + __uint_as_float(r32[b]);
      }
      float* out = a.partials + (int64_t)blockIdx.x * kMaxB * kH + j;
#pragma unroll
      for (int b = 0; b < kMaxB; ++b) out[b * kH] = acc[b];
    }
  } else if (warp == W_LOAD) {
    // =========================== load warp: W, m, v chunk -> stage ===========================
    if (elect_one()) {
      // chained step: this CTA may have been placed on an SM that ANOTHER CTA of the model's previous backward
      // just left, while the CTA that owns these tiles there is still updating them
      if (a.wait_hid != 0) wait_counter(&a.st->bwd_cnt, a.wait_bwd, &a.st->chain_timeout);
      for (int c = 0; c < nchunks; ++c) {
        const int s = c % B_STAGES;
        mbar_wait(&st_free[s], ((uint32_t)(c / B_STAGES) & 1u) ^ 1u);
        uint64_t* full = &st_full[c % B_RING];
        mbar_arrive_expect_tx(full, B_STAGE);
        const int64_t off = (tile_of(c >> 3) * B_NT + (int64_t)(c & 7) * B_CH) * kH;  // chunk blocks are contiguous 8 KB
        const uint32_t dst = smem_u32(sStage + s * B_STAGE);
        // the chunks stream through L2 once per step: evict_first on the loads and the stores measured 7% faster
        // (B200, cfg2) than the default policy
        bulk_load(dst, a.W1 + off, B_ARR, full, kL2EvictFirst);
        bulk_load(dst + B_ARR, a.mW1 + off, B_ARR, full, kL2EvictFirst);
        bulk_load(dst + 2 * B_ARR, a.vW1 + off, B_ARR, full, kL2EvictFirst);
      }
    }
  } else if (warp == W_STORE) {
    // =========================== store warp: updated chunk -> W, m, v ===========================
    // two bulk-store groups in flight: a stage is released once the store issued before the latest
    // one has finished reading shared memory
    if (elect_one()) {
      for (int c = 0; c < nchunks; ++c) {
        const int s = c % B_STAGES;
        mbar_wait(&st_done[c % B_RING], (uint32_t)(c / B_RING) & 1u);
        const int64_t off = (tile_of(c >> 3) * B_NT + (int64_t)(c & 7) * B_CH) * kH;
        const uint32_t src = smem_u32(sStage + s * B_STAGE);
        bulk_store(a.W1 + off, src, B_ARR, kL2EvictFirst);
        bulk_store(a.mW1 + off, src + B_ARR, B_ARR, kL2EvictFirst);
        bulk_store(a.vW1 + off, src + 2 * B_ARR, B_ARR, kL2EvictFirst);
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        if (c > 0) {
          asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
          mbar_arrive(&st_free[(c - 1) % B_STAGES]);
        }
      }
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      mbar_arrive(&st_free[(nchunks - 1) % B_STAGES]);
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
  } else if (warp >= W_FWD0) {
    // ====== forward warps (fused runs), alternating chunks: per chunk, gamma/beta Adam, the next batch's
    //        BN statistics and xhat rows, and the forward MMA on the chunk of W1 just updated in the stage.
    //        Each warp accumulates into its own TMEM columns; the epilogue adds the two. ======
    if (fuse) {
      constexpr uint32_t idesc_f = make_idesc(128, 32, 1, 1);
      const int fw = warp - W_FWD0;
      const int nbn = a.src_next.nb;
      const int64_t nrow = lane < nbn ? row_of(a.src_next, a.st, lane) : 0;
      const uint32_t* nptr = a.packed + nrow * a.row_words;
      const int r = lane & 7;  // SNP of the chunk this lane does the scalar work for (lanes 8.. replicate)
      struct Pre {
        uint32_t word;
        float gm, bt, mg, vg, mb, vb, mm, mv;
      };
      auto prefetch = [&](int c) {
        Pre p = {0u, 1.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 1.f};
        if (c >= nchunks) return p;
        const int64_t k0 = tile_of(c >> 3) * B_NT + (int64_t)(c & 7) * B_CH;
        const int64_t k = k0 + r;
        if (lane < nbn && (k0 >> 4) < a.row_words) p.word = __ldg(nptr + (k0 >> 4));
        if (k < a.K) {
          p.gm = a.gamma[k];
          p.bt = a.beta[k];
          p.mg = a.m_gamma[k];
          p.vg = a.v_gamma[k];
          p.mb = a.m_beta[k];
          p.vb = a.v_beta[k];
          p.mm = a.mmean[k];
          p.mv = a.mvar[k];
        }
        return p;
      };
      Pre cur = prefetch(fw);
      for (int c = fw; c < nchunks; c += B_NFW) {
        const Pre nxt = prefetch(c + B_NFW);  // one chunk of this warp ahead: hides the global-load latency
        const int li = c >> 3, cc = c & 7, buf = li & 1, s = c % B_STAGES;
        const int64_t k0 = tile_of(c >> 3) * B_NT + (int64_t)(c & 7) * B_CH;
        const int64_t k = k0 + r;
        const bool valid = k < a.K;
        // next batch: genotype of (row = lane, SNP r8), per-SNP counts by ballot, statistics -- all of
        // it independent of this chunk's epilogue
        const int sh0 = 2 * (int)(k0 & 15);
        unsigned xs[8];
        int n1 = 0, n2 = 0;
#pragma unroll
        for (int r8 = 0; r8 < 8; ++r8) {
          const unsigned x = (cur.word >> (sh0 + 2 * r8)) & 3u;  // rows >= nbn hold zeros
          xs[r8] = x;
          const unsigned m1 = __ballot_sync(0xffffffffu, x == 1u), m2 = __ballot_sync(0xffffffffu, x == 2u);
          if (r == r8) {
            n1 = __popc(m1);
            n2 = __popc(m2);
          }
        }
        float mean, var;
        moments_from_counts(n1, n2, nbn, mean, var);
        const float rsn = rsqrtf(var + kBnEps);
        mbar_wait(&st_done[c % B_RING], (uint32_t)(c / B_RING) & 1u);
        float P = 0.f, Q = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
          const float2 pr = sRed[(buf * 8 + w) * B_NT + cc * 8 + r];
          P += pr.x;
          Q += pr.y;
        }
        const float rs = sSc[buf * B_NT + cc * 8 + r].z;
        if (cc >= 8 - B_NFW) {  // this warp's last chunk of the tile: its sSc / sRed reads are done
          __syncwarp();
          if (lane == 0) mbar_arrive(&fwd_tile[buf]);
        }
        float gm = cur.gm, mg = cur.mg, vg = cur.vg, bt = cur.bt, mb = cur.mb, vb = cur.vb;
        adam_update_fast(gm, mg, vg, rs * P, alpha);
        adam_update_fast(bt, mb, vb, Q, alpha);
        const float inv = rsn * gm;
        const float shift = bt - mean * inv;
        const float l0 = valid ? to_tf32(shift) : 0.f;
        const float l1 = valid ? to_tf32(inv + shift) : 0.f;
        const float l2 = valid ? to_tf32(2.f * inv + shift) : 0.f;
        uint8_t* xf = sXf + s * B_XF;
#pragma unroll
        for (int r8 = 0; r8 < 8; ++r8) {
          const float a0 = __shfl_sync(0xffffffffu, l0, r8), a1 = __shfl_sync(0xffffffffu, l1, r8),
                      a2 = __shfl_sync(0xffffffffu, l2, r8);
          float val = a0;
          val = xs[r8] == 1u ? a1 : val;
          val = xs[r8] == 2u ? a2 : val;
          if (lane >= nbn) val = 0.f;
          *reinterpret_cast<float*>(xf + r8 * 128 + ((((lane >> 3) ^ (r8 & 3))) << 5) + ((lane & 7) << 2)) = val;
        }
        fence_proxy_async();
        __syncwarp();
        if (elect_one()) {
          tc_fence_after();
          const uint32_t wbs = smem_u32(sStage + s * B_STAGE);
          const uint64_t bdesc = smem_desc(smem_u32(xf), 1024, 512, kLayoutSw128B32);
#pragma unroll
          for (int hh = 0; hh < 2; ++hh)
            umma_tf32(tmem + (uint32_t)(256 + fw * 64 + hh * 32), smem_desc(wbs + hh * 4096, 1024, 512, kLayoutSw128B32),
                      bdesc, idesc_f, c > fw ? 1u : 0u);
          umma_commit(&st_free[s]);
          if (c + B_NFW >= nchunks) umma_commit(fwd_done);
        }
        __syncwarp();
        if (valid && lane < 8) {  // off the stage's critical path
          a.gamma[k] = gm;
          a.m_gamma[k] = mg;
          a.v_gamma[k] = vg;
          a.beta[k] = bt;
          a.m_beta[k] = mb;
          a.v_beta[k] = vb;
          a.mmean[k] = cur.mm * kBnMom + mean * kBnOneMinusMom;  // the next step's forward is a training forward
          a.mvar[k] = cur.mv * kBnMom + var * kBnOneMinusMom;
        }
        cur = nxt;
      }
    }
  } else {
    // =========================== builder warps (2 x 32 SNPs per tile) ===========================
    constexpr uint32_t idesc = make_idesc(128, B_NT, 1, 0);
    const int wb = warp - B_EPI_WARPS;  // 0 / 1: which half of the tile's SNPs
    uint32_t* bits = sBits + wb * 64;
    const int64_t my_row = lane < nb ? row_of(a.src, a.st, lane) : 0;
    const uint32_t* my_ptr = a.packed + my_row * a.row_words;
    // per-SNP state of the two tiles in flight (this lane's SNP): for the gamma/beta update
    float rs_[2] = {0.f, 0.f}, gam_[2] = {0.f, 0.f}, bet_[2] = {0.f, 0.f}, mg_[2] = {0.f, 0.f}, vg_[2] = {0.f, 0.f},
          mb_[2] = {0.f, 0.f}, vb_[2] = {0.f, 0.f};
    auto finalize = [&](int li) {
      // gamma/beta Adam of tile li once its epilogue has left P, Q in shared memory
      const int buf = li & 1;
      mbar_wait(&tmem_empty[buf], (uint32_t)(li >> 1) & 1u);
      if (fuse) {
        // the forward warps update gamma / beta chunk by chunk -- and read this tile's scales (sSc) and row
        // sums (sRed) a little after the epilogue is done with it: the buffers may only be rebuilt once
        // both of them have passed the tile's last chunk
        mbar_wait(&fwd_tile[buf], (uint32_t)(li >> 1) & 1u);
        return;
      }
      const int64_t k = tile_of(li) * B_NT + wb * 32 + lane;
      float P = 0.f, Q = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) {
        const float2 r = sRed[(buf * 8 + w) * B_NT + wb * 32 + lane];
        P += r.x;
        Q += r.y;
      }
      if (k < a.K) {
        float gm = gam_[buf], m = mg_[buf], v = vg_[buf];
        adam_update_fast(gm, m, v, rs_[buf] * P, alpha);
        a.gamma[k] = gm;
        a.m_gamma[k] = m;
        a.v_gamma[k] = v;
        float bt = bet_[buf];
        m = mb_[buf];
        v = vb_[buf];
        adam_update_fast(bt, m, v, Q, alpha);
        a.beta[k] = bt;
        a.m_beta[k] = m;
        a.v_beta[k] = v;
      }
    };
    for (int li = 0; li < nloc; ++li) {
      const int buf = li & 1;
      const int64_t tile = tile_of(li);
      // lane <-> batch row: the 32 genotypes of this builder warp's half tile
      uint2 w2 = make_uint2(0u, 0u);
      const int64_t wofs = tile * 4 + wb * 2;
      if (lane < nb && wofs + 1 < a.row_words) w2 = __ldg(reinterpret_cast<const uint2*>(my_ptr + wofs));
      const int64_t k = tile * B_NT + wb * 32 + lane;
      const bool valid = k < a.K;
      float gm = 0.f, bt = 0.f, mg = 0.f, vg = 0.f, mb = 0.f, vb = 0.f;
      if (valid) {
        gm = a.gamma[k];
        bt = a.beta[k];
        mg = a.m_gamma[k];
        vg = a.v_gamma[k];
        mb = a.m_beta[k];
        vb = a.v_beta[k];
      }
      // the buffers of tile li-2 must be drained (and its gamma/beta update done) before reuse
      if (li >= 2) finalize(li - 2);
      bits[lane * 2] = w2.x;
      bits[lane * 2 + 1] = w2.y;
      __syncwarp();
      const int wsel = lane >> 4, sh = 2 * (lane & 15);
      unsigned long long g = 0ull;
      int n1 = 0, n2 = 0;
#pragma unroll
      for (int b = 0; b < kMaxB; ++b) {
        const unsigned x = (bits[b * 2 + wsel] >> sh) & 3u;
        g |= (unsigned long long)x << (2 * b);
        n1 += (x == 1u);
        n2 += (x == 2u);
      }
      __syncwarp();
      float mean, var;
      moments_from_counts(n1, n2, nb, mean, var);
      const float rs = rsqrtf(var + kBnEps);
      rs_[buf] = rs;
      gam_[buf] = gm;
      bet_[buf] = bt;
      mg_[buf] = mg;
      vg_[buf] = vg;
      mb_[buf] = mb;
      vb_[buf] = vb;
      sSc[buf * B_NT + wb * 32 + lane] = make_float4(valid ? rs * gm : 0.f, valid ? bt : 0.f, valid ? rs : 0.f, 0.f);
      // centred genotypes are multiples of 1/nb: exact in tf32 for a power-of-two batch (the usual 32);
      // a ragged last batch rounds them to tf32 (10-bit mantissa), like every other tf32 product here
      float chi[3];
#pragma unroll
      for (int x = 0; x < 3; ++x) chi[x] = to_tf32(valid ? (float)x - mean : 0.f);
      const int r = wb * 32 + lane;
      uint8_t* xh = sXhi + buf * B_X;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float vh[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int b = 4 * c + e;
          const unsigned x = (unsigned)((g >> (2 * b)) & 3ull);
          float h = chi[0];  // branch-free select
          h = x == 1u ? chi[1] : h;
          h = x == 2u ? chi[2] : h;
          vh[e] = b < nb ? h : 0.f;
        }
        *reinterpret_cast<float4*>(xh + swz(r, c)) = make_float4(vh[0], vh[1], vh[2], vh[3]);
      }
      fence_proxy_async();
      asm volatile("bar.sync 1, 64;" ::: "memory");  // both builder warps have written their half
      if (wb == 0 && lane == 0) {
        tc_fence_after();
        const uint32_t xhb = smem_u32(xh);
        const uint32_t dhi = smem_u32(sDZhi), dlo = smem_u32(sDZlo);
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const uint32_t d = tmem + (uint32_t)(buf * 128 + hh * 64);
          uint32_t acc = 0u;
#pragma unroll
          for (int ks = 0; ks < kMaxB / 8; ++ks) {
            const uint64_t a_hi = smem_desc(dhi + hh * 4 * B_DZ_CHUNK + ks * 1024, B_DZ_CHUNK, 512, kLayoutSw128B32);
            const uint64_t a_lo = smem_desc(dlo + hh * 4 * B_DZ_CHUNK + ks * 1024, B_DZ_CHUNK, 512, kLayoutSw128B32);
            const uint64_t b_hi = smem_desc(xhb + ks * 32, 16, 1024, kLayoutSw128);
            umma_tf32(d, a_hi, b_hi, idesc, acc);
            acc = 1u;
            umma_tf32(d, a_lo, b_hi, idesc, acc);
          }
        }
        umma_commit(&tmem_full[buf]);
      }
    }
    if (nloc >= 2) finalize(nloc - 2);
    if (nloc >= 1) finalize(nloc - 1);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == B_EPI_WARPS) tmem_dealloc(tmem, 512);
  if (threadIdx.x == 0) {
    // everything this CTA wrote (updated chunks: the bulk stores have completed; gamma / beta; the next step's
    // partial tile) is visible before the counter moves: the next hidden stack may already be spinning on it
    __threadfence();
    atomicAdd(&a.st->bwd_cnt, 1u);
    tl_mark(a.tl, blockIdx.x == gridDim.x - 1 ? 18u : (blockIdx.x ? 25u : 2u), (unsigned)a.tl_id);  // 25: any other block
  }
}

}  // namespace tc

// ---------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------
bool l1_tc_supported(int64_t K, int H) {
  if (H != tc::kH || K < 1) return false;
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return false;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  return major == 10;
}

int l1_tc_partials(int64_t K) {
  const int64_t ntiles = cdiv(K, tc::B_NT);
  return (int)(ntiles < sm_count() ? ntiles : sm_count());
}

int l1_forward_tc(const L1Args& a, int n_partials, cudaStream_t s) {
  static bool attr_set = false;
  if (!attr_set) {
    LOC_CUDA(cudaFuncSetAttribute(tc::k_l1_fwd_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::F_SMEM));
    attr_set = true;
  }
  const int64_t ntiles = cdiv(a.K, tc::B_NT);
  tc::k_l1_fwd_tc<<<n_partials, tc::F_THREADS, tc::F_SMEM, s>>>(a, ntiles);
  LOC_LAUNCHED();
  return 0;
}

int l1_forward_wide_tc(const L1Args& a, int n_partials, int nrows, float* out, cudaStream_t s) {
  LOC_CHECK(nrows >= 1 && nrows <= 256, "wide forward: 1..256 rows per pass");
  static bool attr_set = false;
  if (!attr_set) {
    LOC_CUDA(cudaFuncSetAttribute(tc::k_l1_fwd_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::W_SMEM));
    attr_set = true;
  }
  const int64_t ntiles = cdiv(a.K, tc::B_NT);
  tc::k_l1_fwd_wide<<<n_partials, tc::W_THREADS, tc::W_SMEM, s>>>(a, ntiles, nrows, out);
  LOC_LAUNCHED();
  return 0;
}

int l1_backward_tc(const L1Args& a, int nblocks, cudaStream_t s, bool overlap_previous) {
  static bool attr_set = false;
  if (!attr_set) {
    LOC_CUDA(cudaFuncSetAttribute(tc::k_l1_bwd_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::B_SMEM));
    attr_set = true;
  }
  const int64_t ntiles = cdiv(a.K, tc::B_NT);
  // exactly nblocks CTAs: the caller's mirror of DevState::bwd_cnt counts them (fewer than SMs: loc_model_set_l1_ctas
  // leaves SMs to a concurrent hidden stack)
  LOC_CHECK(nblocks >= 1 && nblocks <= ntiles && nblocks <= sm_count(),
            "first-layer backward: CTA count must be in [1, min(tiles, SMs)]");
  // overlap_previous: programmatic dependent launch -- the kernel starts once every CTA of the previous
  // kernel in the stream is running (it never waits for that kernel's results: the ring schedule puts
  // another model's hidden stack there), instead of after its completion
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)nblocks);
  cfg.blockDim = dim3(tc::B_THREADS);
  cfg.dynamicSmemBytes = tc::B_SMEM;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = overlap_previous ? 1 : 0;
  LOC_CUDA(cudaLaunchKernelEx(&cfg, tc::k_l1_bwd_tc, a, ntiles));
  loc::g_launches.fetch_add(1);
  return 0;
}

}  // namespace loc
