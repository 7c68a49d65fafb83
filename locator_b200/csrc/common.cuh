// Shared helpers for the locator_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <string>

#include "../../include/locator_b200.h"

namespace loc {

extern thread_local std::string g_err;
extern std::atomic<long long> g_launches;

inline int fail(const char* what, const char* file, int line) {
  char buf[512];
  snprintf(buf, sizeof(buf), "%s (%s:%d)", what, file, line);
  g_err = buf;
  return 1;
}

#define LOC_CHECK(cond, msg)                                 \
  do {                                                       \
    if (!(cond)) return loc::fail(msg, __FILE__, __LINE__);  \
  } while (0)

#define LOC_CUDA(expr)                                                  \
  do {                                                                  \
    cudaError_t _e = (expr);                                            \
    if (_e != cudaSuccess) {                                            \
      char _b[384];                                                     \
      snprintf(_b, sizeof(_b), "CUDA error %s: %s", cudaGetErrorName(_e), cudaGetErrorString(_e)); \
      return loc::fail(_b, __FILE__, __LINE__);                         \
    }                                                                   \
  } while (0)

// After a kernel launch: count it and surface launch-configuration errors.
#define LOC_LAUNCHED()                 \
  do {                                 \
    loc::g_launches.fetch_add(1);      \
    LOC_CUDA(cudaGetLastError());      \
  } while (0)

inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// SMs of the device current at the first call (148 on a B200); launch geometry everywhere derives from this one value.
inline int sm_count() {
  static const int n = [] {
    int dev = 0, v = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    return v > 0 ? v : 148;
  }();
  return n;
}

// ---- Keras constants (SURVEY.md Appendix A) ----
constexpr float kBnEps = 1e-3f;
constexpr float kBnMom = 0.99f;
constexpr float kBnOneMinusMom = 0.01f;
constexpr float kAdamB1 = 0.9f;
constexpr float kAdamB2 = 0.999f;
constexpr float kAdam1mB1 = 0.1f;
constexpr float kAdam1mB2 = 0.001f;
constexpr float kAdamEps = 1e-7f;

// Device-resident optimizer / epoch / callback state. One per model.
struct DevState {
  int t;         // optimizer iterations completed
  int step_id;   // 0-based index of the step in flight (dropout stream)
  float lr;
  float alpha;   // lr * sqrt(1-b2^t) / (1-b1^t) for the step in flight
  float loss_total, loss_count;  // Keras Mean(loss) accumulators for the epoch
  float val_total, val_count;
  int epoch;
  int epoch0;     // epoch index at the start of the current loc_train_epochs call
  int stopped;
  int improved;
  int best_epoch;
  float ckpt_best, es_best, rlr_best;
  int es_wait, rlr_wait;
  int patience, rlr_patience;
  int max_epochs;
  int nonfinite;
  float last_loss, last_val;
  // Hand-over flags of the programmatic-dependent-launch chain (model.cu: train_step): kernels of one step are
  // launched before their producers have finished and wait here instead of at a kernel boundary.
  int chain_timeout;  // a kernel of a chained step gave up waiting for its producer (~2 s): reported by loc_model_state
  unsigned hid_seq;  // number of training hidden-stack launches completed (published at the kernel's very end)
  unsigned bwd_cnt;  // CTAs of first-layer backward launches completed, cumulative
  unsigned upd_cnt;  // blocks of small-layer update launches completed, cumulative
  unsigned dz_cnt[64];  // per Dense(width) layer i: CTAs of training hidden stacks that have written dz_i (and everything
                        // the layer's update needs), cumulative -- the update of layer i starts under the hidden stack
  float step_sum;  // batches of more than 32 rows: sum of the per-row losses over the chunks of the step in flight
};

// Spin until *flag has reached `expect` (wrap-safe); gives up after ~2 s and raises *err instead of hanging the GPU.
__device__ __forceinline__ void wait_counter(const unsigned* flag, unsigned expect, int* err, unsigned sleep_ns = 256u) {
  const long long t0 = clock64();
  while (true) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
    if ((int)(v - expect) >= 0) break;
    if (clock64() - t0 > 4000000000ll) {
      if (err != nullptr) *err = 1;
      break;
    }
    __nanosleep(sleep_ns);
  }
}

// Kernel timeline (LOC_TIMELINE=1, diagnostics): tl[0] = record count, then (globaltimer ns, tag << 32 | id) pairs.
constexpr unsigned kTlCap = 1u << 16;
__device__ __forceinline__ void tl_mark(unsigned long long* tl, unsigned tag, unsigned id) {
  if (tl == nullptr) return;
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  const unsigned idx = atomicAdd(reinterpret_cast<unsigned*>(tl), 1u);
  if (idx < kTlCap) {
    tl[1 + 2 * (size_t)idx] = t;
    tl[2 + 2 * (size_t)idx] = ((unsigned long long)tag << 32) | id;
  }
}

__device__ __forceinline__ float elu_f(float z) { return z > 0.f ? z : expm1f(z); }
// Branch-free elu for the latency-critical tensor-core hidden stack: libdevice's expm1f is a ~40-instruction
// dependent chain with data-dependent branches (the lanes of a warp diverge).  Here exp(z) - 1 comes from
// ex2.approx (2 ulp of a value near 1, i.e. ~1.2e-7 absolute) for z <= -1/32 and from the series
// z + z^2/2 + z^3/6 + z^4/24 above that (truncation < 3e-9 relative at |z| = 1/32): relative error <= ~4e-6
// over the whole negative axis -- 250 times below the tf32 rounding the next layer applies to this value.
__device__ __forceinline__ float elu_fast(float z) {
  const float e = exp2f(z * 1.4426950408889634f) - 1.0f;
  const float p = z * (1.0f + z * (0.5f + z * (0.16666667f + z * 0.041666668f)));
  const float neg = z > -0.03125f ? p : e;
  return z > 0.f ? z : neg;
}
// d elu / dz expressed through the activation value (EluGrad: out < 0 ? out + 1 : 1).
__device__ __forceinline__ float elu_grad_from_out(float a) { return a > 0.f ? 1.f : a + 1.f; }

// Keras Adam: m += (g-m)(1-b1); v += (g^2-v)(1-b2); w -= alpha*m/(sqrt(v)+eps).
__device__ __forceinline__ void adam_update(float& w, float& m, float& v, float g, float alpha) {
  m = m + (g - m) * kAdam1mB1;
  v = v + (g * g - v) * kAdam1mB2;
  w = w - (m * alpha) / (sqrtf(v) + kAdamEps);
}

}  // namespace loc
