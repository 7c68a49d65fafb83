// K1/K2: genotype filter, 2-bit pack, row/column gathers, jacknife column replacement.
// Integer, HBM-bound, bit-exact against oracle/ingest_ref.py.
//
// Reference semantics (locator/locator.py): filter_snps :265-281 (allel count_alleles /
// is_biallelic / to_allele_counts()[:, :, 1]), split_train_test :303-307, bootstrap gather
// :651-653, jacknife replace :726-727, replace_md :258-261.
#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"

namespace loc {
thread_local std::string g_err;
std::atomic<long long> g_launches{0};

// ---------------------------------------------------------------------------------------------
// Site statistics: one warp per site.  The row (N calls = 2N bytes) is read as 16-byte vectors from
// its first 16-byte boundary on (4 independent loads per lane in flight); the few calls before /
// after the vector body go through the scalar path, so any N and any row offset work.  Per 32-bit
// vector whose alleles are all in {-1, 0, 1} the counts come from two dp4a dot products per word; other vectors
// take exact zero-byte tests in plain integer logic (the __vcmp*4 intrinsics are emulated on this part).
// ---------------------------------------------------------------------------------------------
struct SiteAcc {
  unsigned seen[4];  // allele indices 0..127
  int alt, miss;
};

// allele a in [0, 127] -> bitmap (select instead of a dynamic register index)
__device__ __forceinline__ void mark(SiteAcc& s, int a) {
  const unsigned bit = 1u << (a & 31);
#pragma unroll
  for (int q = 0; q < 4; ++q) s.seen[q] |= (a >> 5) == q ? bit : 0u;
}

__device__ __forceinline__ void acc_call(SiteAcc& s, int a0, int a1) {
  if (a0 >= 0) mark(s, a0);
  if (a1 >= 0) mark(s, a1);
  s.alt += (a0 == 1) + (a1 == 1);
  s.miss += (a0 < 0) | (a1 < 0);
}

// 0x80 in every byte of x that is zero (exact per byte: no borrow crosses a byte)
__device__ __forceinline__ uint32_t zero_bytes(uint32_t x) {
  return ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u;
}

// Running masks of one lane over a row; w = bytes (a0, a1) of call A | (a0, a1) of call B.
struct WordAcc {
  uint32_t any0, any1;  // some allele was 0 / 1
  int alt, miss;
};

// returns the bytes (0x80 flags) that hold an allele >= 2: the caller bitmaps those one by one (rare)
__device__ __forceinline__ uint32_t acc_word(WordAcc& s, uint32_t w) {
  const uint32_t z1 = zero_bytes(w ^ 0x01010101u);  // allele 1
  const uint32_t z0 = zero_bytes(w);                // allele 0
  const uint32_t neg = w & 0x80808080u;             // sign bits: missing alleles
  s.alt += __popc(z1);
  s.any0 |= z0;
  s.any1 |= z1;
  s.miss += __popc((neg | (neg >> 8)) & 0x00800080u);  // a call is missing if either allele is
  return ~(z0 | z1 | w) & 0x80808080u;
}

__device__ __forceinline__ void mark_others(SiteAcc& s, uint32_t w, uint32_t other) {
  if (other) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int a = (int)(int8_t)(w >> (8 * i));
      if (a >= 2) mark(s, a);
    }
  }
}

// 16-byte loads in flight per lane (8 measured slower than 4: the scan is bound by the integer pipe, not by latency)
#ifndef LOC_STAT_LOADS
#define LOC_STAT_LOADS 4
#endif
constexpr int kStatLoads = LOC_STAT_LOADS;

__global__ void __launch_bounds__(256, 4) k_site_stats(const int8_t* __restrict__ gt, int64_t nvar, int64_t nsamp,
                                                    int min_mac, int32_t* __restrict__ n_alleles,
                                                    int32_t* __restrict__ alt_count, int32_t* __restrict__ n_missing,
                                                    uint8_t* __restrict__ keep) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t nbytes = nsamp * 2;
  for (int64_t v = warp; v < nvar; v += nwarps) {
    const int8_t* row = gt + v * nbytes;
    SiteAcc s = {{0u, 0u, 0u, 0u}, 0, 0};
    // calls before the first 16-byte boundary (the whole row if it starts at an odd address)
    const uintptr_t addr = reinterpret_cast<uintptr_t>(row);
    int64_t head = (addr & 1) ? nbytes : (int64_t)((16 - (addr & 15)) & 15);
    if (head > nbytes) head = nbytes;
    for (int64_t c = lane; c < head / 2; c += 32) acc_call(s, row[2 * c], row[2 * c + 1]);
    // vector body
    const uint4* vp = reinterpret_cast<const uint4*>(row + head);
    const int64_t nvec = (nbytes - head) >> 4;
    // Fast path (ncu: the byte-wise zero tests made the scan integer-pipe bound -- 114 warp instructions per 512 bytes,
    // math-pipe throttle the top stall -- at 0.50 of the HBM peak).  A vector whose 16 alleles are all in {-1, 0, 1}
    // (every vector of a biallelic site) only feeds two dot products per word: S1 = sum a, S2 = sum a^2, from which
    // #(a == 1) = (S2 + S1) / 2 and #(a == -1) = (S2 - S1) / 2; missing CALLS = missing alleles - calls with both
    // alleles missing.  Anything else (allele >= 2, a negative value other than -1) sends the vector down the exact
    // byte-by-byte path.
    int s1 = 0, s2 = 0, both = 0, nfast = 0;
    WordAcc wa = {0u, 0u, 0, 0};
    for (int64_t i = lane; i < nvec; i += 32 * kStatLoads) {
      uint4 q[kStatLoads];
#pragma unroll
      for (int u = 0; u < kStatLoads; ++u)
        if (i + 32 * u < nvec) q[u] = __ldcs(vp + i + 32 * u);
#pragma unroll
      for (int u = 0; u < kStatLoads; ++u)
        if (i + 32 * u < nvec) {
          const uint32_t w[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
          uint32_t odd = 0u;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const uint32_t neg = w[e] & 0x80808080u;
            const uint32_t m = (neg >> 7) * 0xFFu;             // 0xFF in every negative byte
            odd |= (w[e] ^ m) & (m | 0xFEFEFEFEu);            // non-negative byte > 1, or negative byte != -1
          }
          if (odd == 0u) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              s1 = __dp4a((int)w[e], 0x01010101, s1);
              s2 = __dp4a((int)w[e], (int)w[e], s2);
              const uint32_t neg = w[e] & 0x80808080u;
              both += __popc(neg & (neg >> 8) & 0x00800080u);
            }
            nfast += 16;
          } else {
            const uint32_t ox = acc_word(wa, w[0]), oy = acc_word(wa, w[1]);
            const uint32_t oz = acc_word(wa, w[2]), ow = acc_word(wa, w[3]);
            mark_others(s, w[0], ox);
            mark_others(s, w[1], oy);
            mark_others(s, w[2], oz);
            mark_others(s, w[3], ow);
          }
        }
    }
    {
      const int n1 = (s2 + s1) >> 1, nm = (s2 - s1) >> 1;  // alleles equal to 1 / to -1 in the fast vectors
      const int n0 = nfast - n1 - nm;
      s.seen[0] |= ((wa.any0 || n0 > 0) ? 1u : 0u) | ((wa.any1 || n1 > 0) ? 2u : 0u);
      s.alt += wa.alt + n1;
      s.miss += wa.miss + nm - both;
    }
    // calls after the last whole vector (< 8)
    const int8_t* tail = row + head + nvec * 16;
    const int64_t tail_calls = (nbytes - head - nvec * 16) / 2;
    if (lane < tail_calls) acc_call(s, tail[2 * lane], tail[2 * lane + 1]);

    int na = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) na += __popc(__reduce_or_sync(0xffffffffu, s.seen[q]));
    const int alt = __reduce_add_sync(0xffffffffu, s.alt);
    const int miss = __reduce_add_sync(0xffffffffu, s.miss);
    if (lane == 0) {
      if (n_alleles) n_alleles[v] = na;
      if (alt_count) alt_count[v] = alt;
      if (n_missing) n_missing[v] = miss;
      if (keep) keep[v] = (na == 2 && (min_mac == 1 || alt >= min_mac)) ? 1 : 0;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Pack: a block turns 256 kept sites x (32 * CALLS) samples into 16 packed words per sample.
// A lane owns CALLS = VB / 2 consecutive samples and reads them with one VB-byte load per site (a warp
// reads 32 * VB contiguous bytes of the site's row; 16 loads in flight per lane); the 2-bit counts of a
// 16-site word come from byte-wise SIMD compares.  A padded shared-memory tile turns the per-lane words
// into 64 contiguous bytes per sample for the write.  Blocks that are adjacent in x cover one set of
// sites across all samples, so concurrently running blocks read whole rows.
// The host picks the widest VB for which every load is aligned (VB | 2N and the base pointer).
// ---------------------------------------------------------------------------------------------
template <int VB>
__device__ __forceinline__ void load_calls(const int8_t* p, uint32_t (&w)[(VB + 3) / 4]) {
  if constexpr (VB == 16) {
    const uint4 q = __ldcs(reinterpret_cast<const uint4*>(p));
    w[0] = q.x, w[1] = q.y, w[2] = q.z, w[3] = q.w;
  } else if constexpr (VB == 8) {
    const uint2 q = __ldcs(reinterpret_cast<const uint2*>(p));
    w[0] = q.x, w[1] = q.y;
  } else if constexpr (VB == 4) {
    w[0] = __ldcs(reinterpret_cast<const uint32_t*>(p));
  } else {
    w[0] = __ldcs(reinterpret_cast<const unsigned short*>(p));  // one call; the upper bytes read as allele 0
  }
}

constexpr int kPackWords = 16;  // packed words (of 16 sites) per block
constexpr int kPackPitch = kPackWords + 1;

template <int VB>
__global__ void __launch_bounds__(256) k_pack_sites(const int8_t* __restrict__ gt, int64_t nsamp,
                                                    const int64_t* __restrict__ site_idx, int64_t K,
                                                    uint32_t* __restrict__ packed, int64_t row_words) {
  constexpr int CALLS = VB / 2;
  constexpr int S = 32 * CALLS;
  constexpr int NW = (VB + 3) / 4;
  __shared__ uint32_t tile[S * kPackPitch];  // [call c of the lane][lane][word], pitch 17: conflict-free writes
  const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
  const int64_t s0 = (int64_t)blockIdx.x * S;
  const int64_t w0 = ((int64_t)blockIdx.z * gridDim.y + blockIdx.y) * kPackWords;  // z: slabs beyond 65535 word groups
  const int64_t sb = s0 + (int64_t)lane * CALLS;  // first sample of this lane (N % CALLS == 0: all or none in range)
#pragma unroll
  for (int jw = 0; jw < 2; ++jw) {
    const int wl = 2 * wi + jw;
    const int64_t k0 = (w0 + wl) * 16;
    uint32_t raw[16][NW];
#pragma unroll
    for (int q = 0; q < 16; ++q) {
#pragma unroll
      for (int e = 0; e < NW; ++e) raw[q][e] = 0u;
      if (k0 + q < K && sb < nsamp) load_calls<VB>(gt + (__ldg(site_idx + k0 + q) * nsamp + sb) * 2, raw[q]);
    }
    uint32_t acc[CALLS];
#pragma unroll
    for (int c = 0; c < CALLS; ++c) acc[c] = 0u;
#pragma unroll
    for (int q = 0; q < 16; ++q) {
#pragma unroll
      for (int e = 0; e < NW; ++e) {
        const uint32_t e1 = zero_bytes(raw[q][e] ^ 0x01010101u) >> 7;         // 1 where the allele is 1
        const uint32_t g2 = (e1 + (e1 >> 8)) & 0x00030003u;                   // count of call A | call B << 16
        acc[2 * e] |= (g2 & 3u) << (2 * q);
        if constexpr (CALLS > 1) acc[2 * e + 1] |= (g2 >> 16) << (2 * q);
      }
    }
#pragma unroll
    for (int c = 0; c < CALLS; ++c) tile[(c * 32 + lane) * kPackPitch + wl] = acc[c];
  }
  __syncthreads();
  const int quarter = threadIdx.x & 3;
  const int64_t w = w0 + 4 * quarter;
  if (w < row_words) {
    for (int sl = threadIdx.x >> 2; sl < S; sl += 64) {
      const int64_t ss = s0 + sl;
      if (ss >= nsamp) break;
      const uint32_t* t = tile + ((sl % CALLS) * 32 + sl / CALLS) * kPackPitch + 4 * quarter;
      *reinterpret_cast<uint4*>(packed + ss * row_words + w) = make_uint4(t[0], t[1], t[2], t[3]);
    }
  }
}

__global__ void k_patch_calls(uint32_t* __restrict__ packed, int64_t row_words, const int64_t* __restrict__ ks,
                              const int64_t* __restrict__ samp, const uint8_t* __restrict__ val, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t k = ks[i];
  uint32_t* wp = packed + samp[i] * row_words + (k >> 4);
  const int sh = 2 * (int)(k & 15);
  atomicAnd(wp, ~(3u << sh));
  atomicOr(wp, ((uint32_t)val[i] & 3u) << sh);
}

// uint8 [n][K] -> packed. One thread per (row, word).
__global__ void k_pack_counts(const uint8_t* __restrict__ counts, int64_t n, int64_t K,
                              uint32_t* __restrict__ packed, int64_t row_words) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t r = blockIdx.y;
  if (w >= row_words || r >= n) return;
  const uint8_t* src = counts + r * K + w * 16;
  uint32_t word = 0u;
  const int64_t rem = K - w * 16;
#pragma unroll
  for (int q = 0; q < 16; ++q)
    if (q < rem) word |= ((uint32_t)src[q] & 3u) << (2 * q);
  packed[r * row_words + w] = word;
}

__global__ void k_unpack_counts(const uint32_t* __restrict__ packed, int64_t n, int64_t K, int64_t row_words,
                                uint8_t* __restrict__ counts) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t r = blockIdx.y;
  if (k >= K || r >= n) return;
  counts[r * K + k] = (uint8_t)((packed[r * row_words + (k >> 4)] >> (2 * (k & 15))) & 3u);
}

__global__ void k_gather_rows(const uint4* __restrict__ in, int64_t row_vec, const int64_t* __restrict__ rows,
                              uint4* __restrict__ out) {
  const int64_t r = blockIdx.y;
  const uint4* src = in + rows[r] * row_vec;
  uint4* dst = out + r * row_vec;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < row_vec; i += (int64_t)gridDim.x * blockDim.x)
    dst[i] = src[i];
}

// out[r][k] = in[r][cols[k]]: one thread per output word (16 random 2-bit reads from one row,
// which stays L1/L2 resident: a row is K/4 bytes).
__global__ void __launch_bounds__(256) k_gather_cols(const uint32_t* __restrict__ in, int64_t row_words_in,
                                                     const int64_t* __restrict__ cols, int64_t K_out,
                                                     uint32_t* __restrict__ out, int64_t row_words_out) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t r = blockIdx.y;
  if (w >= row_words_out) return;
  const uint32_t* src = in + r * row_words_in;
  uint32_t word = 0u;
#pragma unroll 4
  for (int q = 0; q < 16; ++q) {
    const int64_t k = w * 16 + q;
    if (k < K_out) {
      const int64_t c = cols[k];
      word |= ((src[c >> 4] >> (2 * (c & 15))) & 3u) << (2 * q);
    }
  }
  out[r * row_words_out + w] = word;
}

__global__ void k_replace_cols(uint32_t* __restrict__ packed, int64_t n, int64_t row_words,
                               const int64_t* __restrict__ sites, int64_t nsites, const uint8_t* __restrict__ vals) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // sample row (fast -> coalesced vals)
  const int64_t i = blockIdx.y;
  if (r >= n || i >= nsites) return;
  const int64_t k = sites[i];
  uint32_t* wp = packed + r * row_words + (k >> 4);
  const int sh = 2 * (int)(k & 15);
  atomicAnd(wp, ~(3u << sh));
  atomicOr(wp, ((uint32_t)vals[i * n + r] & 3u) << sh);
}

// ---------------------------------------------------------------------------------------------
// Ordered compaction on the device (no host round trip of the masks): exclusive prefix sums over
// per-site counts in three launches -- per-block totals, one block scanning the totals, per-block
// rescan + scatter.  Values: keep flags (site filter) or missing calls per kept site (imputation).
// ---------------------------------------------------------------------------------------------
constexpr int kScanThreads = 256, kScanPer = 8, kScanBlock = kScanThreads * kScanPer;

struct ScanSrc {
  const uint8_t* keep;         // mode 0: value = keep[i]
  const int32_t* per_site;     // mode 1: value = per_site[site_idx[i]]
  const int64_t* site_idx;
};
__device__ __forceinline__ int scan_value(const ScanSrc& s, int64_t i, int64_t n) {
  if (i >= n) return 0;
  return s.keep != nullptr ? (int)(s.keep[i] != 0) : s.per_site[s.site_idx[i]];
}

// block-wide exclusive scan of one int per thread; returns the prefix, *total = block sum (all threads)
__device__ __forceinline__ long long block_exclusive(long long v, long long* total) {
  __shared__ long long wsum[kScanThreads / 32];
  __shared__ long long tot;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  long long inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  __syncthreads();  // wsum / tot of a previous call are no longer read
  if (lane == 31) wsum[w] = inc;
  __syncthreads();
  if (w == 0) {
    long long x = lane < kScanThreads / 32 ? wsum[lane] : 0;
    long long xi = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long t = __shfl_up_sync(0xffffffffu, xi, o);
      if (lane >= o) xi += t;
    }
    if (lane < kScanThreads / 32) wsum[lane] = xi - x;
    if (lane == 31) tot = xi;
  }
  __syncthreads();
  *total = tot;
  return wsum[w] + inc - v;
}

__global__ void __launch_bounds__(kScanThreads) k_scan_totals(ScanSrc src, int64_t n, long long* block_tot) {
  const int64_t base = (int64_t)blockIdx.x * kScanBlock + (int64_t)threadIdx.x * kScanPer;
  long long v = 0;
#pragma unroll
  for (int e = 0; e < kScanPer; ++e) v += scan_value(src, base + e, n);
  long long total;
  block_exclusive(v, &total);
  if (threadIdx.x == 0) block_tot[blockIdx.x] = total;
}

// one block: block_tot[b] -> exclusive prefix (in place), grand total to *count
__global__ void __launch_bounds__(kScanThreads) k_scan_blocks(long long* block_tot, int64_t nblocks, int64_t* count) {
  long long carry = 0;
  for (int64_t b0 = 0; b0 < nblocks; b0 += kScanThreads) {
    const int64_t b = b0 + threadIdx.x;
    const long long v = b < nblocks ? block_tot[b] : 0;
    long long total;
    const long long ex = block_exclusive(v, &total);
    if (b < nblocks) block_tot[b] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) *count = carry;
}

// mode 0: site_idx_out[prefix] = i for kept sites.
__global__ void __launch_bounds__(kScanThreads) k_compact_sites(ScanSrc src, int64_t n, const long long* block_off,
                                                                int64_t* __restrict__ out) {
  const int64_t base = (int64_t)blockIdx.x * kScanBlock + (int64_t)threadIdx.x * kScanPer;
  int f[kScanPer];
  long long v = 0;
#pragma unroll
  for (int e = 0; e < kScanPer; ++e) {
    f[e] = scan_value(src, base + e, n);
    v += f[e];
  }
  long long total;
  long long pos = block_off[blockIdx.x] + block_exclusive(v, &total);
#pragma unroll
  for (int e = 0; e < kScanPer; ++e)
    if (f[e]) out[pos++] = base + e;
}

// mode 1: offsets[i] = exclusive prefix of the missing calls of kept site i (offsets[K] is the total, written
// by the caller from *count).
__global__ void __launch_bounds__(kScanThreads) k_scan_offsets(ScanSrc src, int64_t n, const long long* block_off,
                                                               int64_t* __restrict__ offsets) {
  const int64_t base = (int64_t)blockIdx.x * kScanBlock + (int64_t)threadIdx.x * kScanPer;
  int f[kScanPer];
  long long v = 0;
#pragma unroll
  for (int e = 0; e < kScanPer; ++e) {
    f[e] = scan_value(src, base + e, n);
    v += f[e];
  }
  long long total;
  long long pos = block_off[blockIdx.x] + block_exclusive(v, &total);
#pragma unroll
  for (int e = 0; e < kScanPer; ++e) {
    if (base + e < n) offsets[base + e] = pos;
    pos += f[e];
  }
}

// One warp per kept site with missing calls: (k, sample) of every missing call in ascending sample order, at the
// site's offset -- np.nonzero(is_missing) in row-major (site, sample) order, the order replace_md draws in
// (locator.py:258-261) -- plus the site's allele frequency inputs are already in alt_count / n_missing.
__global__ void __launch_bounds__(256) k_missing_calls(const int8_t* __restrict__ gt, int64_t nsamp,
                                                       const int64_t* __restrict__ site_idx, int64_t K,
                                                       const int64_t* __restrict__ offsets, int64_t* __restrict__ out_k,
                                                       int64_t* __restrict__ out_samp) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t k = warp; k < K; k += nwarps) {
    const int64_t beg = offsets[k], end = offsets[k + 1];
    if (beg == end) continue;
    const int8_t* row = gt + site_idx[k] * nsamp * 2;
    int64_t pos = beg;
    for (int64_t s0 = 0; s0 < nsamp && pos < end; s0 += 32) {
      const int64_t sidx = s0 + lane;
      bool miss = false;
      if (sidx < nsamp) {
        const char2 c = *reinterpret_cast<const char2*>(row + 2 * sidx);
        miss = c.x < 0 || c.y < 0;
      }
      const unsigned m = __ballot_sync(0xffffffffu, miss);
      if (miss) {
        const int64_t o = pos + __popc(m & ((1u << lane) - 1u));
        out_k[o] = k;
        out_samp[o] = sidx;
      }
      pos += __popc(m);
    }
  }
}

// sums[k] = sum over all n rows of the packed counts of SNP k (jacknife allele frequencies, locator.py:714-717,
// with wide integers: the reference's pinned numpy promotes the uint8 row sums).  One thread per packed word
// (16 SNPs), rows in the loop: a warp reads 128 contiguous bytes per row.
__global__ void __launch_bounds__(128) k_site_sums(const uint32_t* __restrict__ packed, int64_t n, int64_t K,
                                                   int64_t row_words, int64_t* __restrict__ sums) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w * 16 >= K) return;
  // two 16 x 4-bit... plain counters: 16 ints per thread, rows split over blockIdx.y slabs and added atomically
  const int64_t r0 = n * blockIdx.y / gridDim.y, r1 = n * (blockIdx.y + 1) / gridDim.y;
  uint32_t lo[16];
#pragma unroll
  for (int q = 0; q < 16; ++q) lo[q] = 0u;
  for (int64_t r = r0; r < r1; ++r) {
    const uint32_t x = __ldg(packed + r * row_words + w);
#pragma unroll
    for (int q = 0; q < 16; ++q) lo[q] += (x >> (2 * q)) & 3u;
  }
#pragma unroll
  for (int q = 0; q < 16; ++q)
    if (w * 16 + q < K && lo[q]) atomicAdd(reinterpret_cast<unsigned long long*>(sums + w * 16 + q), (unsigned long long)lo[q]);
}

}  // namespace loc

using namespace loc;

extern "C" {

int loc_abi_version(void) { return LOC_ABI_VERSION; }
const char* loc_last_error(void) { return loc::g_err.c_str(); }
int64_t loc_launch_count(void) { return (int64_t)loc::g_launches.load(); }

int loc_site_stats(const int8_t* d_gt, int64_t nvar, int64_t nsamp, int32_t min_mac, int32_t* d_n_alleles,
                   int32_t* d_alt_count, int32_t* d_n_missing, uint8_t* d_keep, void* stream) {
  LOC_CHECK(nvar >= 0 && nsamp > 0, "loc_site_stats: bad shape");
  if (nvar == 0) return 0;
  LOC_CHECK(d_gt != nullptr, "loc_site_stats: null genotype pointer");
  const int warps_per_block = 8;
  int64_t blocks = cdiv(nvar, warps_per_block);
  static int wave = 0;  // one resident wave of blocks; the warps loop over the sites
  if (wave == 0) {
    int per_sm = 4;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_site_stats, 256, 0);
    wave = sm_count() * (per_sm > 0 ? per_sm : 1);
  }
  if (blocks > wave) blocks = wave;
  k_site_stats<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(d_gt, nvar, nsamp, min_mac, d_n_alleles,
                                                                 d_alt_count, d_n_missing, d_keep);
  LOC_LAUNCHED();
  return 0;
}


static int scan_launch(const ScanSrc& src, int64_t n, int64_t* d_count, long long** block_off_out, cudaStream_t st) {
  const int64_t nblocks = cdiv(n, kScanBlock);
  long long* block_off = nullptr;
  LOC_CUDA(cudaMallocAsync(&block_off, (size_t)(nblocks > 0 ? nblocks : 1) * sizeof(long long), st));
  if (nblocks > 0) {
    k_scan_totals<<<(unsigned)nblocks, kScanThreads, 0, st>>>(src, n, block_off);
    LOC_LAUNCHED();
  }
  k_scan_blocks<<<1, kScanThreads, 0, st>>>(block_off, nblocks, d_count);
  LOC_LAUNCHED();
  *block_off_out = block_off;
  return 0;
}

int loc_compact_sites(const uint8_t* d_keep, int64_t nvar, int64_t* d_site_idx, int64_t* d_count, void* stream) {
  LOC_CHECK(nvar >= 0 && d_count != nullptr, "loc_compact_sites: bad arguments");
  LOC_CHECK(nvar == 0 || (d_keep != nullptr && d_site_idx != nullptr), "loc_compact_sites: null pointer");
  LOC_CHECK(nvar <= (int64_t)kScanBlock * 0x7fffffff, "loc_compact_sites: too many sites");
  cudaStream_t st = (cudaStream_t)stream;
  ScanSrc src = {d_keep, nullptr, nullptr};
  long long* block_off = nullptr;
  if (scan_launch(src, nvar, d_count, &block_off, st)) return 1;
  if (nvar > 0) {
    k_compact_sites<<<(unsigned)cdiv(nvar, kScanBlock), kScanThreads, 0, st>>>(src, nvar, block_off, d_site_idx);
    LOC_LAUNCHED();
  }
  LOC_CUDA(cudaFreeAsync(block_off, st));
  return 0;
}

int loc_missing_calls(const int8_t* d_gt, int64_t nvar, int64_t nsamp, const int64_t* d_site_idx, int64_t K,
                      const int32_t* d_n_missing, int64_t* d_offsets, int64_t* d_k, int64_t* d_samp, void* stream) {
  (void)nvar;
  LOC_CHECK(K >= 0 && nsamp > 0 && d_offsets != nullptr, "loc_missing_calls: bad arguments");
  LOC_CHECK(K == 0 || (d_gt != nullptr && d_site_idx != nullptr && d_n_missing != nullptr), "loc_missing_calls: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  ScanSrc src = {nullptr, d_n_missing, d_site_idx};
  if (d_k == nullptr) {  // phase 1: offsets[0..K] (offsets[K] = number of missing calls)
    long long* block_off = nullptr;
    if (scan_launch(src, K, d_offsets + K, &block_off, st)) return 1;
    if (K > 0) {
      k_scan_offsets<<<(unsigned)cdiv(K, kScanBlock), kScanThreads, 0, st>>>(src, K, block_off, d_offsets);
      LOC_LAUNCHED();
    }
    LOC_CUDA(cudaFreeAsync(block_off, st));
    return 0;
  }
  LOC_CHECK(d_samp != nullptr, "loc_missing_calls: null output pointer");
  if (K == 0) return 0;
  int64_t blocks = cdiv(K, 8);
  if (blocks > 148 * 8) blocks = 148 * 8;
  k_missing_calls<<<(unsigned)blocks, 256, 0, st>>>(d_gt, nsamp, d_site_idx, K, d_offsets, d_k, d_samp);
  LOC_LAUNCHED();
  return 0;
}

int loc_site_sums(const uint32_t* d_packed, int64_t n, int64_t K, int64_t row_words, int64_t* d_sums, void* stream) {
  LOC_CHECK(n >= 0 && K >= 0 && row_words >= cdiv(K, 16), "loc_site_sums: bad shape");
  if (K == 0) return 0;
  LOC_CHECK(d_sums != nullptr && (n == 0 || d_packed != nullptr), "loc_site_sums: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  LOC_CUDA(cudaMemsetAsync(d_sums, 0, (size_t)K * sizeof(int64_t), st));
  if (n == 0) return 0;
  const int64_t words = cdiv(K, 16);
  int slabs = (int)(n < 16 ? n : 16);  // enough blocks to fill the SMs when K is small
  dim3 grid((unsigned)cdiv(words, 128), (unsigned)slabs);
  k_site_sums<<<grid, 128, 0, st>>>(d_packed, n, K, row_words, d_sums);
  LOC_LAUNCHED();
  return 0;
}

int loc_pack_sites(const int8_t* d_gt, int64_t nvar, int64_t nsamp, const int64_t* d_site_idx, int64_t K,
                   uint32_t* d_packed, int64_t row_words, void* stream) {
  (void)nvar;
  LOC_CHECK(nsamp > 0 && K >= 0, "loc_pack_sites: bad shape");
  LOC_CHECK(row_words >= cdiv(K, 16) && row_words % 4 == 0, "loc_pack_sites: row_words must be >= ceil(K/16) and a multiple of 4");
  if (row_words == 0) return 0;
  LOC_CHECK(d_gt != nullptr && d_packed != nullptr, "loc_pack_sites: null pointer");
  LOC_CHECK(reinterpret_cast<uintptr_t>(d_packed) % 16 == 0, "loc_pack_sites: packed rows must be 16-byte aligned");
  // widest aligned load: VB bytes = VB / 2 calls per lane
  const uintptr_t base = reinterpret_cast<uintptr_t>(d_gt);
  int vb = 16;
  while (vb > 2 && ((nsamp * 2) % vb != 0 || base % vb != 0)) vb >>= 1;
  LOC_CHECK(base % 2 == 0, "loc_pack_sites: genotype pointer must be 2-byte aligned");
  const int S = 32 * (vb / 2);
  const int64_t wgroups = cdiv(row_words, kPackWords);
  const int64_t gy = wgroups < 32768 ? wgroups : 32768;
  dim3 grid((unsigned)cdiv(nsamp, S), (unsigned)gy, (unsigned)cdiv(wgroups, gy));  // blocks past row_words write nothing
  LOC_CHECK(grid.z <= 65535, "loc_pack_sites: K too large for one launch");
  cudaStream_t st = (cudaStream_t)stream;
  switch (vb) {
    case 16: k_pack_sites<16><<<grid, 256, 0, st>>>(d_gt, nsamp, d_site_idx, K, d_packed, row_words); break;
    case 8: k_pack_sites<8><<<grid, 256, 0, st>>>(d_gt, nsamp, d_site_idx, K, d_packed, row_words); break;
    case 4: k_pack_sites<4><<<grid, 256, 0, st>>>(d_gt, nsamp, d_site_idx, K, d_packed, row_words); break;
    default: k_pack_sites<2><<<grid, 256, 0, st>>>(d_gt, nsamp, d_site_idx, K, d_packed, row_words); break;
  }
  LOC_LAUNCHED();
  return 0;
}

int loc_patch_calls(uint32_t* d_packed, int64_t row_words, const int64_t* d_k, const int64_t* d_samp,
                    const uint8_t* d_val, int64_t n, void* stream) {
  if (n <= 0) return 0;
  k_patch_calls<<<(unsigned)cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(d_packed, row_words, d_k, d_samp, d_val, n);
  LOC_LAUNCHED();
  return 0;
}

int loc_pack_counts(const uint8_t* d_counts, int64_t n, int64_t K, uint32_t* d_packed, int64_t row_words,
                    void* stream) {
  LOC_CHECK(row_words >= cdiv(K, 16) && row_words % 4 == 0, "loc_pack_counts: bad row_words");
  if (n <= 0 || row_words == 0) return 0;
  LOC_CHECK(n <= 65535, "loc_pack_counts: more than 65535 rows per call");
  dim3 grid((unsigned)cdiv(row_words, 256), (unsigned)n);
  k_pack_counts<<<grid, 256, 0, (cudaStream_t)stream>>>(d_counts, n, K, d_packed, row_words);
  LOC_LAUNCHED();
  return 0;
}

// Host matrix -> packed device matrix without a pageable cudaMemcpy of the whole thing: row blocks are copied
// into two pinned staging buffers by a few host threads (a single memcpy thread moves ~10 GB/s, the link several
// times that), sent with cudaMemcpyAsync and packed on the device while the next block is being staged.
namespace {
struct UploadStage {
  uint8_t* h[2] = {nullptr, nullptr};
  uint8_t* d[2] = {nullptr, nullptr};
  cudaEvent_t done[2] = {nullptr, nullptr};  // the block's pack kernel has finished (its buffers are reusable)
  size_t bytes = 0;
  int dev = -1;
};
UploadStage g_up;
std::mutex g_up_mu;

void parallel_copy(uint8_t* dst, const uint8_t* src, size_t bytes, int threads) {
  if (threads <= 1 || bytes < (size_t)4 << 20) {
    memcpy(dst, src, bytes);
    return;
  }
  std::vector<std::thread> ts;
  const size_t per = (bytes / threads + 4095) & ~(size_t)4095;
  for (int t = 0; t < threads; ++t) {
    const size_t o = (size_t)t * per;
    if (o >= bytes) break;
    const size_t nbytes = bytes - o < per ? bytes - o : per;
    ts.emplace_back([=] { memcpy(dst + o, src + o, nbytes); });
  }
  for (auto& t : ts) t.join();
}
}  // namespace

int loc_upload_pack_counts(const uint8_t* h_counts, int64_t n, int64_t K, uint32_t* d_packed, int64_t row_words,
                           void* stream) {
  LOC_CHECK(h_counts != nullptr && d_packed != nullptr, "loc_upload_pack_counts: null pointer");
  LOC_CHECK(row_words >= cdiv(K, 16) && row_words % 4 == 0, "loc_upload_pack_counts: bad row_words");
  if (n <= 0 || K <= 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  std::lock_guard<std::mutex> lk(g_up_mu);
  int dev = 0;
  LOC_CUDA(cudaGetDevice(&dev));
  const size_t kStageBytes = (size_t)16 << 20;
  const size_t want = (size_t)K > kStageBytes ? (size_t)K : kStageBytes;
  if (g_up.dev != dev || g_up.bytes < want) {
    for (int i = 0; i < 2; ++i) {
      if (g_up.h[i]) cudaFreeHost(g_up.h[i]);
      if (g_up.d[i]) cudaFree(g_up.d[i]);
      if (g_up.done[i]) cudaEventDestroy(g_up.done[i]);
      g_up.h[i] = g_up.d[i] = nullptr;
      g_up.done[i] = nullptr;
    }
    g_up.bytes = 0;
    for (int i = 0; i < 2; ++i) {
      LOC_CUDA(cudaMallocHost(&g_up.h[i], want));
      LOC_CUDA(cudaMalloc(&g_up.d[i], want));
      LOC_CUDA(cudaEventCreateWithFlags(&g_up.done[i], cudaEventDisableTiming));
    }
    g_up.bytes = want;
    g_up.dev = dev;
  }
  static const int threads = [] {
    const char* e = getenv("LOC_UPLOAD_THREADS");
    int v = e != nullptr ? atoi(e) : 4;
    return v < 1 ? 1 : (v > 16 ? 16 : v);
  }();
  int64_t rows_per = (int64_t)(g_up.bytes / (size_t)K);
  if (rows_per > 65535) rows_per = 65535;
  int blk = 0;
  for (int64_t r0 = 0; r0 < n; r0 += rows_per, ++blk) {
    const int64_t nr = n - r0 < rows_per ? n - r0 : rows_per;
    const int b = blk & 1;
    if (blk >= 2) LOC_CUDA(cudaEventSynchronize(g_up.done[b]));  // the block that used these buffers is packed
    parallel_copy(g_up.h[b], h_counts + r0 * K, (size_t)(nr * K), threads);
    LOC_CUDA(cudaMemcpyAsync(g_up.d[b], g_up.h[b], (size_t)(nr * K), cudaMemcpyHostToDevice, s));
    if (loc_pack_counts(g_up.d[b], nr, K, d_packed + r0 * row_words, row_words, stream)) return 1;
    LOC_CUDA(cudaEventRecord(g_up.done[b], s));
  }
  // the staging buffers are shared by later calls (possibly on other streams): drained before returning
  for (int b = 0; b < 2 && b < blk; ++b) LOC_CUDA(cudaEventSynchronize(g_up.done[b]));
  return 0;
}

int loc_unpack_counts(const uint32_t* d_packed, int64_t n, int64_t K, int64_t row_words, uint8_t* d_counts,
                      void* stream) {
  if (n <= 0 || K <= 0) return 0;
  LOC_CHECK(n <= 65535, "loc_unpack_counts: more than 65535 rows per call");
  dim3 grid((unsigned)cdiv(K, 256), (unsigned)n);
  k_unpack_counts<<<grid, 256, 0, (cudaStream_t)stream>>>(d_packed, n, K, row_words, d_counts);
  LOC_LAUNCHED();
  return 0;
}

int loc_gather_rows(const uint32_t* d_in, int64_t row_words, const int64_t* d_rows, int64_t n_out,
                    uint32_t* d_out, void* stream) {
  LOC_CHECK(row_words % 4 == 0, "loc_gather_rows: row_words must be a multiple of 4");
  if (n_out <= 0 || row_words == 0) return 0;
  LOC_CHECK(n_out <= 65535, "loc_gather_rows: more than 65535 rows per call");
  const int64_t row_vec = row_words / 4;
  dim3 grid((unsigned)(cdiv(row_vec, 256) > 64 ? 64 : cdiv(row_vec, 256)), (unsigned)n_out);
  k_gather_rows<<<grid, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const uint4*>(d_in), row_vec, d_rows,
                                                        reinterpret_cast<uint4*>(d_out));
  LOC_LAUNCHED();
  return 0;
}

int loc_gather_cols(const uint32_t* d_in, int64_t n, int64_t row_words_in, const int64_t* d_cols, int64_t K_out,
                    uint32_t* d_out, int64_t row_words_out, void* stream) {
  LOC_CHECK(row_words_out >= cdiv(K_out, 16) && row_words_out % 4 == 0, "loc_gather_cols: bad row_words_out");
  if (n <= 0 || row_words_out == 0) return 0;
  LOC_CHECK(n <= 65535, "loc_gather_cols: more than 65535 rows per call");
  dim3 grid((unsigned)cdiv(row_words_out, 256), (unsigned)n);
  k_gather_cols<<<grid, 256, 0, (cudaStream_t)stream>>>(d_in, row_words_in, d_cols, K_out, d_out, row_words_out);
  LOC_LAUNCHED();
  return 0;
}

int loc_replace_cols(uint32_t* d_packed, int64_t n, int64_t row_words, const int64_t* d_sites, int64_t nsites,
                     const uint8_t* d_vals, void* stream) {
  if (n <= 0 || nsites <= 0) return 0;
  LOC_CHECK(nsites <= 65535 * 32, "loc_replace_cols: too many sites per call");
  // grid.y is limited to 65535: loop in slabs.
  for (int64_t off = 0; off < nsites; off += 65535) {
    const int64_t cnt = (nsites - off) < 65535 ? (nsites - off) : 65535;
    dim3 grid((unsigned)cdiv(n, 128), (unsigned)cnt);
    k_replace_cols<<<grid, 128, 0, (cudaStream_t)stream>>>(d_packed, n, row_words, d_sites + off, cnt,
                                                           d_vals + off * n);
    LOC_LAUNCHED();
  }
  return 0;
}

}  // extern "C"
