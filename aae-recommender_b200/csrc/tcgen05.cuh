// sm_100a PTX wrappers of the tensor-core kernels (K3 in dec_out_tc.cu, K5 v1 in dec_out_select.cu, K5 v2 in
// dec_out_select2.cu): mbarriers, tcgen05 MMA / TMEM / fences, shared-memory and instruction descriptors, bulk and
// tensor copies; and the no-swizzle K-major hi/lo operand layer that K3 and K5 v1 share (namespace tc).
#pragma once
#include <cuda.h>
#include "common.cuh"

#ifndef TC_WAIT_HINT
#define TC_WAIT_HINT 0x989680u
#endif
#ifndef TC_WAIT_SLEEP_NS
#define TC_WAIT_SLEEP_NS 40
#endif

namespace aae {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarriers ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// Wait with a software back-off between polls (K3, K5 v1, the self-test): spinning warps steal issue slots from the
// MMA issuer.  TC_WAIT_HINT / TC_WAIT_SLEEP_NS are tunables (-D).
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  uint32_t spins = 0;
  while (!done) {
    if (spins) __nanosleep(TC_WAIT_SLEEP_NS);
    if (++spins > (1u << 22)) __trap();          // a lost MMA completion must not hang the device
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity), "r"(TC_WAIT_HINT)   // suspend-time hint: sleep in hardware, do not spin
        : "memory");
  }
}
// Wait that polls without a software sleep (K5 v2).
__device__ __forceinline__ void mbar_wait_spin(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, 0x989680;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (!done && ++spins > (1u << 24)) __trap();      // a lost completion must not hang the device
  }
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---- fences -------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- TMEM ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// store 16 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
      "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
      "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
      "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float* v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr),
               "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
               "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
               "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// 8 consecutive fp32 columns of this thread's TMEM lane, issue and wait
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
// N-column loads and stores (N = 8 or 16); the loaded registers are valid after ld_wait, which ties them to the wait
template <int N> struct TmemIO;
template <> struct TmemIO<8> {
  static __device__ __forceinline__ void ld_issue(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
  }
  static __device__ __forceinline__ void ld_wait(uint32_t* r) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7])::"memory");
  }
  static __device__ __forceinline__ void st(uint32_t taddr, const float* v) { tmem_st8(taddr, v); }
};
template <> struct TmemIO<16> {
  static __device__ __forceinline__ void ld_issue(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
  }
  static __device__ __forceinline__ void ld_wait(uint32_t* r) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])::"memory");
  }
  static __device__ __forceinline__ void st(uint32_t taddr, const float* v) { tmem_st16(taddr, v); }
};
// one wait for two TmemIO<16> loads (32 registers)
__device__ __forceinline__ void tmem_ld_wait32(uint32_t* r) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                 "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                 "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])::"memory");
}

// ---- descriptors --------------------------------------------------------------------------------------------------
// shared-memory matrix descriptor, SWIZZLE_NONE, Blackwell version bit
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
// the same with a swizzle mode in bits [61,64) (1 = SWIZZLE_128B_BASE32B: the layout of MN-major 32-bit operands,
// 2 = SWIZZLE_128B, 6 = SWIZZLE_32B)
__device__ __forceinline__ uint64_t make_desc_sw(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
  return make_desc(saddr, lbo_bytes, sbo_bytes) | ((uint64_t)layout_type << 61);
}
// K-major operand, SWIZZLE_32B: rows of 32 bytes, SBO = 256 bytes between 8-row groups (LBO unused)
__device__ __forceinline__ uint64_t make_desc_sw32(uint32_t saddr) { return make_desc_sw(saddr, 16u, 256u, 6u); }
// K-major operand, SWIZZLE_128B: rows of 128 bytes, SBO = 1024 bytes between 8-row groups (LBO unused)
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t saddr) { return make_desc_sw(saddr, 16u, 1024u, 2u); }
// instruction descriptor for kind::tf32, fp32 accumulate; a/b_mn_major = 1: that operand is MN-major
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn_major = 0, int b_mn_major = 0) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- MMA (kind::tf32, cta_group::1) -------------------------------------------------------------------------------
// both operands in shared memory
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// A operand from TMEM (lanes = M, columns = K), B from shared memory
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on `bar` once every MMA issued so far by this thread has completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// the same arrival on the barrier at the same offset in every CTA of the cluster named in `mask`
__device__ __forceinline__ void mma_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}
// the tf32 part of x (upper 19 bits); x - tf32_hi(x) is exact
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }

// ---- bulk and tensor copies ---------------------------------------------------------------------------------------
// TMA bulk copy global -> shared (contiguous bytes, 16-byte aligned), completion counted on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {
  if (bytes >= 16u)
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes & ~15u) : "memory");
}
// one 2-D box of a tensor map into this CTA's shared memory
__device__ __forceinline__ void tma_load(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}
// the same box multicast to every CTA of the cluster named in `mask` (same smem offset, same barrier offset)
__device__ __forceinline__ void tma_load_mc(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%2, %3}], "
      "[%4], %5;" ::"r"(smem_u32(dst)),
      "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar)), "h"(mask)
      : "memory");
}

// ---------------------------------------------------------------------------------------------------------------------
// K-major hi/lo operands without swizzle (K3, K5 v1).  tf32 operands are only usable K-major without the special
// 32-byte-base swizzle, so every shared-memory operand is stored K-major in the no-swizzle core-matrix layout (8 rows x
// 16 bytes per core matrix), each as a tf32 "hi" part and an fp32 remainder "lo" (x = hi + lo exactly).
// ---------------------------------------------------------------------------------------------------------------------
namespace tc {

constexpr int TN = 32;          // items per K3 tile
constexpr int BM = 128;         // batch rows per chunk (MMA M)
constexpr int CORE = 128;       // bytes of one core matrix (8 rows x 16 B)

// store 4 consecutive columns (one 16-byte chunk) of row r as hi / lo
__device__ __forceinline__ void store_split4(unsigned char* hi, unsigned char* lo, int r, int cg, uint32_t s_r,
                                             float4 x, bool with_lo) {
  uint32_t off = (uint32_t)(r >> 3) * s_r + (uint32_t)cg * CORE + (uint32_t)(r & 7) * 16u;
  float4 h = make_float4(tf32_hi(x.x), tf32_hi(x.y), tf32_hi(x.z), tf32_hi(x.w));
  *reinterpret_cast<float4*>(hi + off) = h;
  if (with_lo) *reinterpret_cast<float4*>(lo + off) = make_float4(x.x - h.x, x.y - h.y, x.z - h.z, x.w - h.w);
}

// Descriptors of one operand (hi and lo parts) with the per-k-step increment of the start-address
// field (units of 16 bytes); built once per kernel.
struct SmemOp {
  uint64_t hi, lo;
  uint32_t step16;
};
__device__ __forceinline__ SmemOp make_op(const void* hi, const void* lo, uint32_t lbo, uint32_t sbo, uint32_t step) {
  SmemOp o;
  o.hi = make_desc(smem_u32(hi), lbo, sbo);
  o.lo = make_desc(smem_u32(lo), lbo, sbo);
  o.step16 = step >> 4;
  return o;
}
// One GEMM, both operands in shared memory: up to 16 k-steps x (1 or 3) tcgen05.mma.  Fully unrolled with a
// warp-uniform bound so that the descriptor arithmetic stays on constants (the issuing lane executes a few
// instructions per MMA instead of rebuilding descriptors).  SPLIT 3 issues hi*hi + lo*hi + hi*lo (3xTF32, the dropped
// lo*lo term is 2^-22 relative), SPLIT 1 hi*hi only.
template <int SPLIT>
__device__ __forceinline__ void issue_gemm(uint32_t d_tmem, const SmemOp& a, const SmemOp& b, int ksteps,
                                           uint32_t idesc, uint32_t first_acc) {
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    if (k < ksteps) {
      const uint32_t acc = (k == 0) ? first_acc : 1u;
      const uint64_t ah = a.hi + (uint64_t)(k * a.step16), bh = b.hi + (uint64_t)(k * b.step16);
      if (SPLIT == 3) {
        mma_tf32(d_tmem, a.lo + (uint64_t)(k * a.step16), bh, idesc, acc);
        mma_tf32(d_tmem, ah, b.lo + (uint64_t)(k * b.step16), idesc, 1u);
        mma_tf32(d_tmem, ah, bh, idesc, 1u);
      } else {
        mma_tf32(d_tmem, ah, bh, idesc, acc);
      }
    }
  }
}
// One GEMM with the A operand in TMEM: k-step s reads A columns [8s, 8s+8).
template <int SPLIT>
__device__ __forceinline__ void issue_gemm_ts(uint32_t d_tmem, uint32_t a_hi_t, uint32_t a_lo_t, const SmemOp& b,
                                              int ksteps, uint32_t idesc, uint32_t first_acc) {
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    if (k < ksteps) {
      const uint32_t acc = (k == 0) ? first_acc : 1u;
      const uint64_t bh = b.hi + (uint64_t)(k * b.step16);
      if (SPLIT == 3) {
        mma_tf32_ts(d_tmem, a_lo_t + 8 * k, bh, idesc, acc);
        mma_tf32_ts(d_tmem, a_hi_t + 8 * k, b.lo + (uint64_t)(k * b.step16), idesc, 1u);
        mma_tf32_ts(d_tmem, a_hi_t + 8 * k, bh, idesc, 1u);
      } else {
        mma_tf32_ts(d_tmem, a_hi_t + 8 * k, bh, idesc, acc);
      }
    }
  }
}

// Shared-memory operand geometry (all K-major, no swizzle; LBO = stride between 16-byte column
// groups along K, SBO = stride between 8-row groups along M/N).
struct Geom {
  int H, Kp, Np;             // hidden, K of G1 padded to 8 (H+1 -> Kp), N of G2 padded to 16
  uint32_t hb_sbo, wb_sbo;   // Hb [128][Kp], Wb [32][Kp]: LBO = CORE
  uint32_t wt_lbo, wt_sbo;   // Wtb [Np][32]  (rows = hidden unit, cols = item)
  uint32_t dt_lbo, dt_sbo;   // Dtb [32][128] (rows = item, cols = batch row)
  uint32_t hb_bytes, wb_bytes, wt_bytes, dt_bytes;
};
__host__ __device__ inline Geom make_geom(int H) {
  Geom g;
  g.H = H;
  g.Kp = (H + 1 + 7) & ~7;
  g.Np = (g.Kp + 15) & ~15;
  g.hb_sbo = (uint32_t)(g.Kp / 4) * CORE;
  g.wb_sbo = (uint32_t)(g.Kp / 4) * CORE;
  g.wt_lbo = CORE + 16;                     // +16: the transposing stores of the W' tile are conflict-free
  g.wt_sbo = (TN / 4) * g.wt_lbo;
  g.dt_lbo = CORE + 16;                     // +16: the E1 transposing stores become conflict-free
  g.dt_sbo = (BM / 4) * g.dt_lbo;
  g.hb_bytes = (BM / 8) * g.hb_sbo;
  g.wb_bytes = (TN / 8) * g.wb_sbo;
  g.wt_bytes = (uint32_t)(g.Np / 8) * g.wt_sbo;
  g.dt_bytes = (TN / 8) * g.dt_sbo;
  return g;
}

}  // namespace tc

// Envelope of the K-major operand layout: 16-byte column groups of W' rows, at most 16 k-steps of 8 (K = H+1 <= 128).
static inline bool tc_supported(int B, int H, const char* what) {
  if ((H & 3) != 0 || H + 1 > 128) {
    set_error("%s: tensor-core kernel needs n_hidden %% 4 == 0 and n_hidden <= 124 (got %d); use impl=simt", what, H);
    return false;
  }
  return true;
}

}  // namespace aae
