// Shared device/host helpers for libaae_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/aae_b200.h"

namespace aae {

void set_error(const char* fmt, ...);
int check_launch(const char* what);

#define AAE_REQUIRE(cond, msg)                                   \
  do {                                                           \
    if (!(cond)) {                                               \
      aae::set_error("%s: %s", __func__, msg);                   \
      return AAE_E_ARG;                                          \
    }                                                            \
  } while (0)

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
int sm_count();

// ---------------------------------------------------------------------------------------------
// Adam, one element.  torch/optim/adam.py::_single_tensor_adam:
//   m.lerp_(g, 1-b1); v.mul_(b2).addcmul_(g, g, 1-b2); denom = sqrt(v)/sqrt(1-b2^t) + eps;
//   p.addcdiv_(m, denom, -lr/(1-b1^t))
// ---------------------------------------------------------------------------------------------
struct AdamK {
  float w1, beta2, w2, eps, step_size, inv_bc2_sqrt;
};
__device__ __forceinline__ AdamK adam_load(const aae_step_state* st, int which) {
  AdamK k;
  k.w1 = (float)(1.0 - 0.9);      // torch passes the python double 1-beta1
  k.beta2 = st->beta2;
  k.w2 = (float)(1.0 - 0.999);
  k.eps = st->eps;
  k.step_size = which ? st->step_size_reg : st->step_size_gen;
  k.inv_bc2_sqrt = 1.0f / st->bc2_sqrt;
  return k;
}
__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  // .ftz: one MUFU.SQRT instead of the denormal-range fix-up sequence; a second moment below 1.2e-38 (|g| < 1e-17)
  // flushes to 0 and leaves denom = eps, an update of < 1e-10 * lr either way.  Max relative error 2^-23.
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// m/denom uses the 2-ulp fast division, sqrt the approximate instruction: both far inside the 1e-4
// parity tolerance (the update is lr * O(1)), and they keep the fused epilogues off the slow paths.
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));   // max relative error 2^-23; denom >= eps = 1e-8 here
  return r;
}
__device__ __forceinline__ void adam_update(const AdamK& k, float g, float& p, float& m, float& v) {
  m = fmaf(k.w1, g - m, m);
  v = fmaf(k.w2 * g, g, v * k.beta2);
  float denom = fmaf(sqrt_approx(v), k.inv_bc2_sqrt, k.eps);
  p = fmaf(-k.step_size, m * rcp_approx(denom), p);
}
// zero-gradient update (rows that are not in the batch)
__device__ __forceinline__ void adam_update_zero(const AdamK& k, float& p, float& m, float& v) {
  m = fmaf(k.w1, -m, m);
  v = v * k.beta2;
  float denom = fmaf(sqrt_approx(v), k.inv_bc2_sqrt, k.eps);
  p = fmaf(-k.step_size, m * rcp_approx(denom), p);
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (counter-based RNG) for the native dropout / prior-sampling mode.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}
__device__ __forceinline__ float u01(uint32_t x) { return (x >> 8) * (1.0f / 16777216.0f) + (0.5f / 16777216.0f); }

// multiplicative dropout factor for element `idx` of a [B,width] layer
__device__ __forceinline__ float drop_factor(const aae_drop& d, const aae_step_state* st, uint32_t idx) {
  if (d.mask) return d.mask[idx];
  if (d.p <= 0.f) return 1.0f;
  uint4 r = philox4x32(make_uint4(idx, st->rng_step, d.stream_id, 0x5eedu),
                       make_uint2((uint32_t)st->seed, (uint32_t)(st->seed >> 32)));
  return u01(r.x) < d.p ? 0.0f : 1.0f / (1.0f - d.p);
}
__device__ __forceinline__ float randn_elem(const aae_step_state* st, uint32_t idx, uint32_t stream_id) {
  uint4 r = philox4x32(make_uint4(idx, st->rng_step, stream_id, 0xbeefu),
                       make_uint2((uint32_t)st->seed, (uint32_t)(st->seed >> 32)));
  float u1 = u01(r.x), u2 = u01(r.y);
  return sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
}

// ---------------------------------------------------------------------------------------------
// Step timeline (debug/profiling): when a trace buffer is installed (aae_trace_set), block 0 of every kernel
// of the step writes %globaltimer at its start (slot 2*id) and end (slot 2*id+1).  One pointer copy per
// translation unit (no relocatable device code); NULL = off (one uniform load per kernel).
// ---------------------------------------------------------------------------------------------
enum TraceId { TR_PREP = 0, TR_SWEEP, TR_AE_FWD, TR_K3, TR_AE_BWD, TR_AE_WGRAD, TR_ROWS1, TR_DISC, TR_DISC_WGRAD,
               TR_GEN, TR_GEN_WGRAD, TR_ROWS2, TR_FINISH, TR_BAG_FWD, TR_CATCHUP, TR_N };
static __device__ unsigned long long* g_trace_buf = nullptr;
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void trace_mark(int id, int end) {
  // start = earliest block start, end = latest block end (the host presets the slots to ~0 / 0)
  if (g_trace_buf && threadIdx.x == 0) {
    if (end) atomicMax(g_trace_buf + 2 * id + 1, globaltimer_ns());
    else atomicMin(g_trace_buf + 2 * id, globaltimer_ns());
  }
}
#define AAE_DEFINE_TRACE_SETTER(name)                                                    \
  void name(unsigned long long* p) { cudaMemcpyToSymbol(g_trace_buf, &p, sizeof(p)); }
void trace_set_bag(unsigned long long* p);   // bag.cu
void trace_set_mlp(unsigned long long* p);   // mlp.cu
void trace_set_tc(unsigned long long* p);    // dec_out_tc.cu
void trace_set_w1b(unsigned long long* p);   // w1_blocked.cu

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------------------------------------
// BCE term and logit gradient, following ATen exactly at the edges (SURVEY 8(a) A6):
//   x' = fl(x + 1e-12), t' in {1e-12, 1};  l = (t'-1)*max(log1p(-x'),-100) - t'*max(log x',-100)
//   dL/dz = (x'-t') / max((1-x')x', 1e-12) * x(1-x) / N
// `inv_n` = 1/N.  Returns the loss term, writes dz.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float bce_term(float z, bool positive, float inv_n, float& dz) {
  // stable sigmoid: u = exp(-|z|), x = 1/(1+u) or u/(1+u)  (ATen: 1/(1+exp(-z)); same to ~1 ulp)
  float u = __expf(-fabsf(z));
  float r = __fdividef(1.0f, 1.0f + u);
  float x = (z >= 0.f) ? r : u * r;
  float xp = x + 1e-12f;
  float om = 1.0f - xp;
  // -log1p(-x) = softplus(z) = max(z,0) + log1p(u); x' rounded to 1 -> log1p(-1) = -inf, clamped at
  // -100 by ATen.  (The reference's extra 1e-12*log(x') term, <= 1e-10, is dropped.)
  float poly = u * (1.0f - u * (0.5f - u * (0.33333334f - u * (0.25f - 0.2f * u))));
  float l1p = (u < 0.0625f) ? poly : __logf(1.0f + u);
  float l = fminf(fmaxf(z, 0.f) + l1p, 100.0f);
  l = (om <= 0.f) ? 100.0f : l;
  float t = 1e-12f;
  if (positive) {           // rare: the few items of the set that fall into this tile
    l = fminf(-__logf(xp), 100.0f);
    t = 1.0f;
  }
  float den = fmaxf(om * xp, 1e-12f);
  dz = __fdividef((xp - t) * (x * (1.0f - x)), den) * inv_n;
  return l;
}

}  // namespace aae
