// K5 v1: predict's dense scores and its first threshold filter on tcgen05, fp32-accurate through the 3xTF32 split
// (single-pass TF32 for impl 2).  aae_dec_out_scores runs this kernel over all tiles; aae_predict_topk (topk.cu) runs
// it over the threshold sample and then as the filter.  Shares the K-major hi/lo operand layer of tcgen05.cuh with K3
// (dec_out_tc.cu).
#include <algorithm>
#include "tcgen05.cuh"
#include "dec_out.cuh"

namespace aae {
namespace tc {

// ---------------------------------------------------------------------------------------------
// K5: pipelined scores kernel with a selection epilogue (predict + ranking without the [B,V] round trip).
//
// One CTA = one chunk of 128 query rows x a strided subset of 128-item tiles.  The A operand (the H2' chunk, hi and lo
// parts) lives in TMEM for the whole chunk (ts-form MMAs: lane = query row, column = k): an SS-mode M128 MMA would
// re-read 4 KB of A from shared memory per instruction, more than the 128 B/cycle shared memory delivers.
// Warp 16 issues the MMAs (39 x M128.N128.K8 per tile with the 3xTF32 split); warps 0-15 are loaders (W' tile -> tf32
// hi/lo K-major operand, two 106 KB shared-memory stages) and epilogue (two 128-column TMEM accumulator buffers):
// while tile i is drained and tile i+2 is staged, the tensor pipe runs tile i+1.  Per stage s one mbarrier pair:
// ready[s] (one arrival per loader warp: stage filled AND accumulator s drained) and mma[s] (tcgen05.commit: logits
// of the tile in TMEM, stage s free again).
// Epilogues: DENSE (scores, optionally sigmoid, to out[b, col]; col = item, or the visit order for the threshold
// sample) and FILTER (z > tau[b]: append (z, item) to a private sub-list of the row; ~0.07 % of the elements).
// Replaces the dense lin3 + sigmoid of predict (aae.py:866-868) and the front half of remove_non_missing + argtopk
// (evaluation.py:183-199, 20-58).
// ---------------------------------------------------------------------------------------------
// (Staging the W' tiles with cp.async straight into the hi operand half was measured slower with the 3xTF32 split --
// 2.59 vs 2.18 ms at V=2M / B=1000: the lo pass then sits between the epilogue and the stage hand-over -- and removed.)
constexpr int PN = 128;                // items per tile
constexpr int P_NWE = 16;              // loader / epilogue warps
constexpr int P_NT = 32 * P_NWE + 32;  // + the MMA warp
constexpr int P_CW = PN / 4;           // accumulator columns per epilogue thread (4 warps per TMEM lane quarter)
constexpr int P_WCH = 7;               // 16-byte W' chunks per loader thread (8 rows x <= 28 column groups per warp)
constexpr uint32_t P_T_AHI = 256, P_T_ALO = 384, P_TMEM_COLS = 512;   // TMEM: accumulators 2 x PN | A hi (Kp <= 128) | A lo

struct SelArgs {
  const float* h2; int B, H;
  const float* Wd3; const float* bd3; int Vloc, v_begin;
  int tile_stride, n_sel;              // tiles visited: j * tile_stride, j < n_sel
  int filter;                          // 0: dense scores, 1: threshold filter
  float* out; long long ldo; int out_by_visit, apply_sigmoid;
  // filter: row b owns gridDim.x * 4 private sub-lists (one per CTA column x and 32-column part of the tile) of cap_sub
  // slots; sub-list counters live in registers (one writer each: no atomics, deterministic order) and are stored to
  // cnt[b * nsub + sub] at the end of the chunk (a count above cap_sub = overflow)
  const float* tau; int tau_stride; int32_t* cnt; float* cand_val; int32_t* cand_idx; int cap_sub;
};

// Loader mapping (16 warps, 128 rows x Kp/4 <= 28 column groups of 16 bytes): warp w owns the 8 rows 8w .. 8w+7 and
// all column groups; lane & 7 = row inside the group, column groups (lane >> 3) + 4 j.  One warp-wide load touches
// 8 rows x 64 contiguous bytes (8-16 cache lines) instead of 32 rows x 16 bytes (32 lines): with a row-per-lane
// mapping the kernel was bound by the L1TEX tag stage (ncu: l1tex throughput 85 %, 31 sectors per request).  A
// quarter warp writes 8 consecutive rows of one column group = one 128-byte core matrix: conflict-free.
// All per-thread offsets are tile-invariant and computed once (goff: float offset inside the tile's rows, -1 = bias
// column, -2 = unused; soff: byte offset inside a stage half).
struct PChunks {
  int goff[P_WCH];
  uint32_t soff[P_WCH];
};
__device__ __forceinline__ void p_load_w(float4* wr, const PChunks& pc, const float* __restrict__ wtile,
                                         const float* __restrict__ btile, bool rv) {
#pragma unroll
  for (int j = 0; j < P_WCH; ++j) {
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (rv) {
      if (pc.goff[j] >= 0) x = __ldg(reinterpret_cast<const float4*>(wtile + pc.goff[j]));
      else if (pc.goff[j] == -1) x.x = __ldg(btile);
    }
    wr[j] = x;
  }
}
__device__ __forceinline__ void p_store_w(const float4* wr, const PChunks& pc, unsigned char* hi, unsigned char* lo,
                                          bool with_lo) {
#pragma unroll
  for (int j = 0; j < P_WCH; ++j) {
    if (pc.goff[j] == -2) continue;
    const float4 x = wr[j];
    const float4 h = make_float4(tf32_hi(x.x), tf32_hi(x.y), tf32_hi(x.z), tf32_hi(x.w));
    *reinterpret_cast<float4*>(hi + pc.soff[j]) = h;
    if (with_lo) *reinterpret_cast<float4*>(lo + pc.soff[j]) = make_float4(x.x - h.x, x.y - h.y, x.z - h.z, x.w - h.w);
  }
}

template <int SPLIT>
__global__ void __launch_bounds__(P_NT, 1) dec_out_select_kernel(SelArgs a) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ uint64_t bar_mma[2], bar_ready[2];
  __shared__ uint32_t tmem_base_s;
  constexpr bool with_lo = (SPLIT == 3);
  const Geom g = make_geom(a.H);
  const uint32_t wb_bytes = (PN / 8) * g.wb_sbo;
  unsigned char* wst = smem;                       // stage s: hi at wst + 2*s*wb_bytes, lo right after
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ncg = g.Kp / 4;
  const int n_chunks = (a.B + BM - 1) / BM;
  const int n_my = ((int)blockIdx.x < a.n_sel) ? (a.n_sel - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  for (uint32_t q = tid; q < 4u * wb_bytes / 16u; q += P_NT) reinterpret_cast<float4*>(wst)[q] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (warp == P_NWE) tmem_alloc(&tmem_base_s, P_TMEM_COLS);
  if (tid == 0) {
    mbar_init(&bar_mma[0], 1);
    mbar_init(&bar_mma[1], 1);
    mbar_init(&bar_ready[0], P_NWE);
    mbar_init(&bar_ready[1], P_NWE);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const uint32_t idesc = make_idesc(BM, PN, 0, 0);
  uint32_t ph0 = 0, ph1 = 0;                       // parity of the barrier this role waits on, per stage
  for (int chunk = blockIdx.y; chunk < n_chunks; chunk += gridDim.y) {
    const int b0 = chunk * BM, nb = min(BM, a.B - b0);
    __syncthreads();                               // the previous chunk is drained: the A operand may be rebuilt
    if (warp < P_NWE) {
      // H2' chunk -> TMEM (A operand of every MMA of this chunk: lane = query row, column = k; hi and lo parts).
      // A from TMEM instead of shared memory: an SS-mode M128 x K8 tf32 MMA reads 4 KB of A per slot on top of B,
      // more than the 128 B/cycle the shared memory delivers -- with A in shared memory the kernel was feed-bound.
      const int q4 = warp & 3, cpart = warp >> 2;
      const uint32_t lane_addr = tmem + ((uint32_t)(q4 * 32) << 16);
      const int brow = q4 * 32 + lane;
      for (int c = cpart; c < g.Kp / 8; c += 4) {
        float hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int kk = c * 8 + j;
          float x = 0.f;
          if (brow < nb) x = (kk < a.H) ? __ldg(a.h2 + (size_t)(b0 + brow) * a.H + kk) : (kk == a.H ? 1.0f : 0.f);
          hi[j] = tf32_hi(x);
          lo[j] = x - hi[j];
        }
        tmem_st8(lane_addr + P_T_AHI + c * 8, hi);
        if (with_lo) tmem_st8(lane_addr + P_T_ALO + c * 8, lo);
      }
      tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == P_NWE) {
      // ================= MMA issuer =================
      const SmemOp op_w0 = make_op(wst, wst + wb_bytes, CORE, g.wb_sbo, 2 * CORE);
      const SmemOp op_w1 = make_op(wst + 2 * wb_bytes, wst + 3 * wb_bytes, CORE, g.wb_sbo, 2 * CORE);
      for (int it = 0; it < n_my; ++it) {
        const int s = it & 1;
        mbar_wait_backoff(&bar_ready[s], s ? ph1 : ph0);
        if (s) ph1 ^= 1; else ph0 ^= 1;
        tc_fence_after();
        if (elect_one()) {
          issue_gemm_ts<SPLIT>(tmem + (uint32_t)(s * PN), tmem + P_T_AHI, tmem + P_T_ALO, s ? op_w1 : op_w0, g.Kp / 8,
                               idesc, 0u);
          mma_commit(&bar_mma[s]);
        }
        __syncwarp();
      }
    } else {
      // ================= loaders + epilogue =================
      const int q4 = warp & 3, cpart = warp >> 2;
      const uint32_t lane_addr = tmem + ((uint32_t)(q4 * 32) << 16);
      const int brow = q4 * 32 + lane;
      const bool rowv = brow < nb;
      float tau = __int_as_float(0x7f800000);
      if (a.filter && rowv) tau = a.tau[(size_t)(b0 + brow) * a.tau_stride];
      const int nsub = (int)gridDim.x * 4, sub = (int)blockIdx.x * 4 + cpart;
      const size_t sub_base = ((size_t)(b0 + brow) * nsub + sub) * (size_t)a.cap_sub;
      int my_cnt = 0;
      // loader role of this thread
      const int lrow = warp * 8 + (lane & 7);
      PChunks pc;
#pragma unroll
      for (int j = 0; j < P_WCH; ++j) {
        const int cg = (lane >> 3) + 4 * j, c = cg * 4;
        pc.goff[j] = (cg < ncg) ? ((c + 3 < a.H) ? lrow * a.H + c : (c == a.H ? -1 : -3)) : -2;
        pc.soff[j] = (uint32_t)(lrow >> 3) * g.wb_sbo + (uint32_t)cg * CORE + (uint32_t)(lrow & 7) * 16u;
      }
      const int tile_step = (int)gridDim.x * a.tile_stride * PN;           // items between two tiles of this CTA
      const int v_first = (int)blockIdx.x * a.tile_stride * PN;
      auto load_tile = [&](float4* wr, int v0) {
        p_load_w(wr, pc, a.Wd3 + (size_t)v0 * a.H, a.bd3 + v0 + lrow, v0 + lrow < a.Vloc);
      };
      float4 wr[P_WCH];
      for (int p = 0; p < 2 && p < n_my; ++p) {
        load_tile(wr, v_first + p * tile_step);
        p_store_w(wr, pc, wst + 2 * p * wb_bytes, wst + (2 * p + 1) * wb_bytes, with_lo);
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_ready[p]);
      }
      if (n_my > 2) load_tile(wr, v_first + 2 * tile_step);
      for (int i = 0; i < n_my; ++i) {
        const int s = i & 1;
        const int v0 = v_first + i * tile_step;
        mbar_wait_backoff(&bar_mma[s], s ? ph1 : ph0);       // logits of tile i in TMEM buffer s, stage s free again
        if (s) ph1 ^= 1; else ph0 ^= 1;
        tc_fence_after();
        uint32_t zr[P_CW];
        TmemIO<16>::ld_issue(lane_addr + (uint32_t)(s * PN + cpart * P_CW), zr);
        TmemIO<16>::ld_issue(lane_addr + (uint32_t)(s * PN + cpart * P_CW + 16), zr + 16);
        TmemIO<16>::ld_wait(zr);
        TmemIO<16>::ld_wait(zr + 16);
        tc_fence_before();
        if (i + 2 < n_my) {
          p_store_w(wr, pc, wst + 2 * s * wb_bytes, wst + (2 * s + 1) * wb_bytes, with_lo);
          fence_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(&bar_ready[s]);
          if (i + 3 < n_my) load_tile(wr, v0 + 3 * tile_step);
        }
        // ---- epilogue of tile i
        const int c0 = cpart * P_CW;
        const int vm = a.Vloc - v0 - c0;                         // valid columns among this thread's 32
        if (a.filter) {
          float zmax = __uint_as_float(zr[0]);
#pragma unroll
          for (int j = 1; j < P_CW; ++j) zmax = fmaxf(zmax, __uint_as_float(zr[j]));
          if (zmax > tau) {
#pragma unroll
            for (int j = 0; j < P_CW; ++j) {
              const float z = __uint_as_float(zr[j]);
              if (z > tau && j < vm) {
                if (my_cnt < a.cap_sub) {
                  a.cand_val[sub_base + my_cnt] = z;
                  a.cand_idx[sub_base + my_cnt] = a.v_begin + v0 + c0 + j;
                }
                ++my_cnt;
              }
            }
          }
        } else if (rowv) {
          const int colbase = a.out_by_visit ? ((int)blockIdx.x + i * (int)gridDim.x) * PN : v0;
          float* orow = a.out + (size_t)(b0 + brow) * a.ldo + colbase + c0;
          if (vm >= P_CW && ((reinterpret_cast<uintptr_t>(orow) & 15) == 0)) {
#pragma unroll
            for (int j = 0; j < P_CW; j += 4) {
              float4 o;
              o.x = __uint_as_float(zr[j]); o.y = __uint_as_float(zr[j + 1]);
              o.z = __uint_as_float(zr[j + 2]); o.w = __uint_as_float(zr[j + 3]);
              if (a.apply_sigmoid) {
                o.x = 1.0f / (1.0f + expf(-o.x)); o.y = 1.0f / (1.0f + expf(-o.y));
                o.z = 1.0f / (1.0f + expf(-o.z)); o.w = 1.0f / (1.0f + expf(-o.w));
              }
              __stcs(reinterpret_cast<float4*>(orow + j), o);
            }
          } else {
#pragma unroll
            for (int j = 0; j < P_CW; ++j) {
              if (j < vm) {
                float sc = __uint_as_float(zr[j]);
                if (a.apply_sigmoid) sc = 1.0f / (1.0f + expf(-sc));
                orow[j] = sc;
              }
            }
          }
        }
      }
      if (a.filter && rowv) a.cnt[(size_t)(b0 + brow) * nsub + sub] = my_cnt;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == P_NWE) tmem_dealloc(tmem, P_TMEM_COLS);
}

}  // namespace tc

// grid of the K5 kernel for B query rows and n_sel tiles: y = chunks of 128 rows, x = CTAs sharing a chunk
void dec_out_select_grid(int B, int n_sel, int* gx, int* gy) {
  const int n_chunks = (B + tc::BM - 1) / tc::BM;
  *gy = std::min(n_chunks, sm_count());
  *gx = std::max(1, std::min(n_sel, sm_count() / *gy));
}

// K5 launcher: dense scores (filter == 0) or threshold filter (filter == 1) over the tiles j * tile_stride, j < n_sel.
int dec_out_select_tc(const float* h2, int B, int H, const float* Wd3, const float* bd3, int Vloc, int v_begin,
                      int tile_stride, int n_sel, int filter, float* out, int64_t ldo, int out_by_visit,
                      int apply_sigmoid, const float* tau, int tau_stride, int32_t* cnt, float* cand_val,
                      int32_t* cand_idx, int cap, int split, cudaStream_t s) {
  if (!tc_supported(B, H, "dec_out_select")) return AAE_E_UNSUPPORTED;
  tc::Geom g = tc::make_geom(H);
  const size_t smem = 4 * (size_t)(tc::PN / 8) * g.wb_sbo + 256;
  auto kern = (split == 3) ? tc::dec_out_select_kernel<3> : tc::dec_out_select_kernel<1>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) {
    set_error("dec_out_select: smem %zu: %s", smem, cudaGetErrorString(e));
    return AAE_E_CUDA;
  }
  tc::SelArgs a;
  a.h2 = h2; a.B = B; a.H = H; a.Wd3 = Wd3; a.bd3 = bd3; a.Vloc = Vloc; a.v_begin = v_begin;
  a.tile_stride = tile_stride; a.n_sel = n_sel; a.filter = filter;
  a.out = out; a.ldo = ldo; a.out_by_visit = out_by_visit; a.apply_sigmoid = apply_sigmoid;
  a.tau = tau; a.tau_stride = tau_stride; a.cnt = cnt; a.cand_val = cand_val; a.cand_idx = cand_idx; a.cap_sub = cap;
  int gx, gy;
  dec_out_select_grid(B, n_sel, &gx, &gy);
  kern<<<dim3(gx, gy), tc::P_NT, smem, s>>>(a);
  return check_launch("dec_out_select");
}

// Dense scores of all Vloc items (aae_dec_out_scores, impl 1-4): the K5 kernel over every tile.
int dec_out_scores_tc(const float* h2, int B, int H, const float* Wd3, const float* bd3, int Vloc, int apply_sigmoid,
                      float* out, int64_t ldo, int split, cudaStream_t s) {
  if (!tc_supported(B, H, "dec_out_scores")) return AAE_E_UNSUPPORTED;
  return dec_out_select_tc(h2, B, H, Wd3, bd3, Vloc, 0, 1, (Vloc + tc::PN - 1) / tc::PN, 0, out, ldo, 0, apply_sigmoid,
                           nullptr, 0, nullptr, nullptr, nullptr, 0, split, s);
}

}  // namespace aae
