// K3: the n_items-wide decoder output layer, training, on tcgen05 (5th-gen tensor cores, accumulators in
// TMEM), fp32-accurate through a 3xTF32 split.  Two kernels (one tile at a time; the role-split pipeline
// that is the default for the reference's shapes), their launchers and the operand self-test.  The PTX
// wrappers and the K-major hi/lo operand layer are in tcgen05.cuh.
//
// Per tile of TN=32 items and a batch of up to 128 rows, three GEMMs (each operand kept as a tf32
// "hi" part and an fp32 remainder "lo"; x = hi + lo exactly; products issued as hi*hi + lo*hi + hi*lo,
// the dropped lo*lo term is 2^-22 relative):
//   G1  Z   [b,v]  = H2'[b,:] . W'[v,:]     M=128(b) N=32(v) K=H+1   A = Hb  smem [b][k]    B = Wb  smem [v][k]
//   G2  dh2 [b,k] += dZ[b,:]  . W'[:,k]     M=128(b) N=Np(k) K=32(v) A = dZ  TMEM (b,v)     B = Wtb smem [k][v]
//   G3  dW'^T[k,v] = H2'[:,k] . dZ[:,v]     M=128(k) N=32(v) K=B(b)  A = H2'^T TMEM (k,b)   B = Dtb smem [v][b]
// with H2' = [h2 | 1] and W' = [Wd3 | bd3], so the bias rides inside the MMA (logit = G1, bias
// gradient = row H of G3).  tf32 operands are only usable K-major without the special 32-byte-base
// swizzle, so every shared-memory operand is stored K-major in the no-swizzle core-matrix layout
// (8 rows x 16 bytes per core matrix) and the two operands that would need a transposed view are
// instead fed from TMEM (A operand of G2 and G3): dZ is written back to TMEM by the epilogue that
// computes it, H2'^T is loaded into TMEM once per CTA.  TMEM budget (512 columns): Z 32, dW'^T 32,
// dh2 128, dZ hi/lo 64, H2'^T hi/lo 256.
// Epilogues: (E1) TMEM -> registers, sigmoid + BCE + dZ exactly as the fp32 kernel (common.cuh), dZ
// split into hi/lo and stored to TMEM (A of G2) and transposed to shared memory (B of G3);
// (E2) TMEM lane = hidden unit k, so each warp reads/writes 128-byte coalesced segments of W/m/v rows
// and applies Adam in registers.  Logits never reach HBM.
//
// Reference: aaerec/aae.py:176-177 (lin3 + sigmoid), :693-695 (BCE), :703 (backward), :707 (dec_optim).
#include "tcgen05.cuh"
#include "dec_out.cuh"

#ifndef TC2_CW
#define TC2_CW 16   // accumulator columns per epilogue thread of the pipelined kernel (two roles of 8 warps each)
#endif
#ifndef TC2_G1_FIRST
#define TC2_G1_FIRST 1
#endif

namespace aae {
AAE_DEFINE_TRACE_SETTER(trace_set_tc)
namespace tc {

constexpr int NT = 512;         // threads: 16 warps = 4 TMEM lane quarters x 4 column parts
constexpr int CW = 8;           // accumulator columns per thread in the epilogues

// Pins a prefetched register tile to its point of use: without it the compiler hoists the hi/lo split (pure ALU work
// on the loaded values) up to right behind the global loads, and the warp then waits for the load latency one
// iteration early, in the middle of the pipeline, instead of letting it overlap the MMAs of that iteration.
#ifndef TC_PIN_PREFETCH
#define TC_PIN_PREFETCH 1
#endif
__device__ __forceinline__ void pin4(float4& x) {
#if TC_PIN_PREFETCH
  asm volatile("" : "+f"(x.x), "+f"(x.y), "+f"(x.z), "+f"(x.w));
#endif
}
__host__ __device__ inline size_t smem_bytes(const Geom& g) {
  return 2 * ((size_t)g.hb_bytes + g.wb_bytes + g.wt_bytes + g.dt_bytes) + 256;
}

constexpr uint32_t TMEM_COLS = 512;
// TMEM column map: Z, dW'^T, dZ hi, dZ lo, dh2, H2'^T hi, H2'^T lo
constexpr uint32_t TM_Z = 0, TM_DW = 32, TM_DZH = 64, TM_DZL = 96, TM_DH = 128, TM_HTH = 256, TM_HTL = 384;

// H2' chunk -> Hb hi/lo (rows >= nb and columns > H are zero, column H is the ones column)
__device__ __forceinline__ void fill_hb(unsigned char* hb_hi, unsigned char* hb_lo, const Geom& g,
                                        const float* __restrict__ h2, int b0, int nb, bool with_lo, int nthreads = NT) {
  const int ncg = g.Kp / 4;
  for (int q = threadIdx.x; q < BM * ncg; q += nthreads) {
    int r = q / ncg, cg = q - r * ncg;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < nb) {
      int c = cg * 4;
      if (c + 3 < g.H) x = *reinterpret_cast<const float4*>(h2 + (size_t)(b0 + r) * g.H + c);
      else if (c == g.H) x.x = 1.0f;
    }
    store_split4(hb_hi, hb_lo, r, cg, g.hb_sbo, x, with_lo);
  }
}
// H2'^T -> TMEM (lane = hidden unit k, column = batch row), hi and lo halves
__device__ __forceinline__ void fill_ht_tmem(uint32_t lane_addr, int k, int cpart, const Geom& g,
                                             const float* __restrict__ h2, int B, bool with_lo) {
  for (int c = cpart; c < BM / CW; c += NT / 128) {
    float hi[CW], lo[CW];
#pragma unroll
    for (int j = 0; j < CW; ++j) {
      int b = c * CW + j;
      float x = 0.f;
      if (b < B) x = (k < g.H) ? h2[(size_t)b * g.H + k] : (k == g.H ? 1.0f : 0.f);
      hi[j] = tf32_hi(x);
      lo[j] = x - hi[j];
    }
    tmem_st8(lane_addr + TM_HTH + c * CW, hi);
    if (with_lo) tmem_st8(lane_addr + TM_HTL + c * CW, lo);
  }
  tmem_st_wait();
}

// This thread's share of the W' tile: lane = item row r, warp w owns the 16-byte column groups cg = w and
// w + 16 (Kp/4 <= 32): with this mapping both the K-major store into Wb and the transposing store into Wtb
// are bank-conflict free; all index arithmetic is tile-invariant and done once.
constexpr int WCH = 2;
struct WChunk {
  int goff;            // float offset inside the tile's rows of Wd3 (r*H + 4cg); -1 bias column, -2 unused, -3 zero pad
  uint32_t wb_off;     // byte offset in Wb (16-byte chunk)
  uint32_t wt_off;     // byte offset in Wtb of element 0 (elements e at +16e)
};
__device__ __forceinline__ void make_wchunks(WChunk* wc, const Geom& g) {
  const int ncg = g.Kp / 4;
  const int r = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < WCH; ++j) {
    int cg = w + 16 * j;
    wc[j].goff = -2;
    if (cg < ncg) {
      int c = cg * 4;
      wc[j].goff = (c + 3 < g.H) ? r * g.H + c : (c == g.H ? -1 : -3);
    }
    wc[j].wb_off = (uint32_t)(r >> 3) * g.wb_sbo + (uint32_t)cg * CORE + (uint32_t)(r & 7) * 16u;
    wc[j].wt_off = (uint32_t)(cg >> 1) * g.wt_sbo + (uint32_t)(r >> 2) * g.wt_lbo + (uint32_t)(cg & 1) * 64u +
                   (uint32_t)(r & 3) * 4u;
  }
}
__device__ __forceinline__ void load_w_regs(float4* wr, const WChunk* wc, const float* __restrict__ Wd3,
                                            const float* __restrict__ bd3, int H, int v0, int nv) {
  const int r = threadIdx.x & 31;
#pragma unroll
  for (int j = 0; j < WCH; ++j) {
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < nv) {
      if (wc[j].goff >= 0) x = __ldcs(reinterpret_cast<const float4*>(Wd3 + (size_t)v0 * H + wc[j].goff));
      else if (wc[j].goff == -1) x.x = __ldg(bd3 + v0 + r);
    }
    wr[j] = x;
  }
}
// W' tile -> Wb ([v][k], G1) and, transposed, Wtb ([k][v], G2)
__device__ __forceinline__ void store_w_regs(const float4* wr, const WChunk* wc, unsigned char* wb_hi,
                                             unsigned char* wb_lo, unsigned char* wt_hi, unsigned char* wt_lo,
                                             bool with_lo) {
#pragma unroll
  for (int j = 0; j < WCH; ++j) {
    if (wc[j].goff == -2) continue;
    float4 x = wr[j];
    float4 h = make_float4(tf32_hi(x.x), tf32_hi(x.y), tf32_hi(x.z), tf32_hi(x.w));
    float4 l = make_float4(x.x - h.x, x.y - h.y, x.z - h.z, x.w - h.w);
    *reinterpret_cast<float4*>(wb_hi + wc[j].wb_off) = h;
    if (with_lo) *reinterpret_cast<float4*>(wb_lo + wc[j].wb_off) = l;
    if (wt_hi) {
      float* th = reinterpret_cast<float*>(wt_hi + wc[j].wt_off);
      th[0] = h.x; th[4] = h.y; th[8] = h.z; th[12] = h.w;
      if (with_lo) {
        float* tl = reinterpret_cast<float*>(wt_lo + wc[j].wt_off);
        tl[0] = l.x; tl[4] = l.y; tl[8] = l.z; tl[12] = l.w;
      }
    }
  }
}

// Positives of a tile for one batch row, from a cursor into the row's sorted CSR columns (tiles are
// visited in increasing item order, so the cursor only moves forward; `nxt` caches indices[pos]).
struct RowCursor {
  int pos, end, nxt;
};
__device__ __forceinline__ uint32_t tile_targets(RowCursor& c, const int32_t* __restrict__ indices, int v0g) {
  uint32_t m = 0;
  while (c.nxt < v0g + TN) {
    if (c.nxt >= v0g) m |= 1u << (c.nxt - v0g);
    ++c.pos;
    c.nxt = (c.pos < c.end) ? indices[c.pos] : 0x7fffffff;
  }
  return m;
}

// ---------------------------------------------------------------------------------------------
// training kernel (B <= 128: the whole batch is one chunk, dh2 accumulates in TMEM over all tiles)
// ---------------------------------------------------------------------------------------------
template <int SPLIT>
__global__ void __launch_bounds__(NT, 1) dec_out_train_tc_kernel(
    const float* __restrict__ h2, int B, int H, float* __restrict__ Wd3, float* __restrict__ bd3,
    float* __restrict__ mW, float* __restrict__ vW, float* __restrict__ mb, float* __restrict__ vb, int v_begin,
    int Vloc, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices, float inv_n,
    const aae_step_state* __restrict__ st, float* __restrict__ dh2, double* __restrict__ loss_sum) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ uint64_t bar_mma;
  __shared__ uint32_t tmem_base_s;
  __shared__ float red[NT / 32];
  constexpr int split = SPLIT;
  const Geom g = make_geom(H);
  unsigned char* hb_hi = smem;
  unsigned char* hb_lo = hb_hi + g.hb_bytes;
  unsigned char* wb_hi = hb_lo + g.hb_bytes;
  unsigned char* wb_lo = wb_hi + g.wb_bytes;
  unsigned char* wt_hi = wb_lo + g.wb_bytes;
  unsigned char* wt_lo = wt_hi + g.wt_bytes;
  unsigned char* dt_hi = wt_lo + g.wt_bytes;
  unsigned char* dt_lo = dt_hi + g.dt_bytes;
  const bool with_lo = (split == 3);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q4 = warp & 3, cpart = warp >> 2;      // TMEM lane quarter, 8-column part of the 32-wide tile
  const int n_tiles = (Vloc + TN - 1) / TN;
  const AdamK ak = adam_load(st, 0);

  if (warp == 0) tmem_alloc(&tmem_base_s, TMEM_COLS);
  if (tid == 0) {
    mbar_init(&bar_mma, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // zero the transposed W' buffers once (rows Kp..Np stay zero), build Hb
  for (int q = tid; q < (int)(2 * g.wt_bytes) / 16; q += NT) reinterpret_cast<float4*>(wt_hi)[q] = make_float4(0, 0, 0, 0);
  fill_hb(hb_hi, hb_lo, g, h2, 0, B, with_lo);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const uint32_t lane_addr = tmem + ((uint32_t)(q4 * 32) << 16);
  const int brow = q4 * 32 + lane;                 // E1: batch row of this thread; E2: hidden unit
  fill_ht_tmem(lane_addr, brow, cpart, g, h2, B, with_lo);
  uint32_t phase = 0;

  const uint32_t idesc_g1 = make_idesc(BM, TN, 0, 0);
  const uint32_t idesc_g2 = make_idesc(BM, g.Np, 0, 0);
  const SmemOp op_hb = make_op(hb_hi, hb_lo, CORE, g.hb_sbo, 2 * CORE);
  const SmemOp op_wb = make_op(wb_hi, wb_lo, CORE, g.wb_sbo, 2 * CORE);
  const SmemOp op_wt = make_op(wt_hi, wt_lo, g.wt_lbo, g.wt_sbo, 2 * g.wt_lbo);
  const SmemOp op_dt = make_op(dt_hi, dt_lo, g.dt_lbo, g.dt_sbo, 2 * g.dt_lbo);
  const int ksteps_b = (B + 7) / 8;
  // E1 transposing-store base of this thread: element (v = 8*cpart + j, b = brow) at +16j
  const uint32_t dt_off = (uint32_t)cpart * g.dt_sbo + (uint32_t)(brow >> 2) * g.dt_lbo + (uint32_t)(brow & 3) * 4u;

  RowCursor cur;
  cur.pos = cur.end = 0;
  cur.nxt = 0x7fffffff;
  if (brow < B) {
    cur.pos = indptr[brow];
    cur.end = indptr[brow + 1];
    // first tile of this CTA: skip the row's items below it
    int first = v_begin + (int)blockIdx.x * TN;
    while (cur.pos < cur.end && indices[cur.pos] < first) ++cur.pos;
    if (cur.pos < cur.end) cur.nxt = indices[cur.pos];
  }

  WChunk wc[WCH];
  make_wchunks(wc, g);
  float loss_local = 0.f;
  float4 wr[WCH];
  int tile = blockIdx.x;
  if (tile < n_tiles) load_w_regs(wr, wc, Wd3, bd3, H, tile * TN, min(TN, Vloc - tile * TN));
  bool dh_started = false;

  for (; tile < n_tiles; tile += gridDim.x) {
    const int v0 = tile * TN;
    const int nv = min(TN, Vloc - v0);
    // ---- W' tile (prefetched registers) -> operand buffers; prefetch the next tile
    store_w_regs(wr, wc, wb_hi, wb_lo, wt_hi, wt_lo, with_lo);
    {
      int nt = tile + gridDim.x;
      if (nt < n_tiles) load_w_regs(wr, wc, Wd3, bd3, H, nt * TN, min(TN, Vloc - nt * TN));
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    // ---- G1: logits
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
        issue_gemm<SPLIT>(tmem + TM_Z, op_hb, op_wb, g.Kp / 8, idesc_g1, 0u);
        mma_commit(&bar_mma);
      }
      __syncwarp();
    }
    // targets of this tile for this thread's row, and the E2 operands, while the MMAs run
    // skip items of the tiles other CTAs own, then collect this tile's positives
    while (cur.nxt < v_begin + v0) {
      ++cur.pos;
      cur.nxt = (cur.pos < cur.end) ? indices[cur.pos] : 0x7fffffff;
    }
    uint32_t tmask = tile_targets(cur, indices, v_begin + v0);
    const int k = brow;
    float pw[CW], pm[CW], pv[CW];
#pragma unroll
    for (int j = 0; j < CW; ++j) {
      int v = cpart * CW + j;
      pw[j] = pm[j] = pv[j] = 0.f;
      if (v < nv) {
        if (k < H) {
          size_t off = (size_t)(v0 + v) * H + k;
          pw[j] = Wd3[off]; pm[j] = __ldcs(mW + off); pv[j] = __ldcs(vW + off);
        } else if (k == H) {
          pw[j] = bd3[v0 + v]; pm[j] = mb[v0 + v]; pv[j] = vb[v0 + v];
        }
      }
    }
    mbar_wait_backoff(&bar_mma, phase);
    phase ^= 1;
    tc_fence_after();
    // ---- E1: sigmoid + BCE + dZ for (row brow, columns 8*cpart .. +7)
    {
      float z[CW], dzh[CW], dzl[CW];
      tmem_ld8(lane_addr + TM_Z + cpart * CW, z);
#pragma unroll
      for (int j = 0; j < CW; ++j) {
        int v = cpart * CW + j;
        float d = 0.f;
        if (brow < B && v < nv) loss_local += bce_term(z[j], (tmask >> v) & 1u, inv_n, d);
        float h = tf32_hi(d);
        dzh[j] = h;
        dzl[j] = d - h;
        *reinterpret_cast<float*>(dt_hi + dt_off + 16 * j) = h;
        if (with_lo) *reinterpret_cast<float*>(dt_lo + dt_off + 16 * j) = d - h;
      }
      tmem_st8(lane_addr + TM_DZH + cpart * CW, dzh);
      if (with_lo) tmem_st8(lane_addr + TM_DZL + cpart * CW, dzl);
      tmem_st_wait();
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    // ---- G2 (dh2 accumulates over tiles) and G3 (dW'^T)
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
        issue_gemm_ts<SPLIT>(tmem + TM_DW, tmem + TM_HTH, tmem + TM_HTL, op_dt, ksteps_b, idesc_g1, 0u);
        issue_gemm_ts<SPLIT>(tmem + TM_DH, tmem + TM_DZH, tmem + TM_DZL, op_wt, TN / 8, idesc_g2, dh_started ? 1u : 0u);
        mma_commit(&bar_mma);
      }
      __syncwarp();
    }
    dh_started = true;
    mbar_wait_backoff(&bar_mma, phase);
    phase ^= 1;
    tc_fence_after();
    // ---- E2: Adam on (hidden unit k, items 8*cpart .. +7): coalesced over k
    {
      float gw[CW];
      tmem_ld8(lane_addr + TM_DW + cpart * CW, gw);
#pragma unroll
      for (int j = 0; j < CW; ++j) {
        int v = cpart * CW + j;
        if (v < nv && k <= H) {
          float p = pw[j], m = pm[j], vv = pv[j];
          adam_update(ak, gw[j], p, m, vv);
          if (k < H) {
            size_t off = (size_t)(v0 + v) * H + k;
            Wd3[off] = p; __stcs(mW + off, m); __stcs(vW + off, vv);
          } else {
            bd3[v0 + v] = p; mb[v0 + v] = m; vb[v0 + v] = vv;
          }
        }
      }
    }
    tc_fence_before();
    __syncthreads();   // TMEM Z / dW / dZ and the operand buffers are free again
  }
  // ---- flush dh2 (lane = batch row, columns = hidden unit)
  tc_fence_after();
  if (dh_started) {
    for (int c = cpart; c < g.Np / CW; c += NT / 128) {
      float d[CW];
      tmem_ld8(lane_addr + TM_DH + c * CW, d);
      if (brow < B) {
#pragma unroll
        for (int j = 0; j < CW; ++j) {
          int kk = c * CW + j;
          if (kk < H) atomicAdd(dh2 + (size_t)brow * H + kk, d[j]);
        }
      }
    }
  }
  float s = warp_sum(loss_local);
  if (lane == 0) red[warp] = s;
  tc_fence_before();
  __syncthreads();
  if (tid == 0) {
    double tot = 0.0;
    for (int w = 0; w < NT / 32; ++w) tot += (double)red[w];
    atomicAdd(loss_sum, tot);
  }
  if (warp == 0) tmem_dealloc(tmem, TMEM_COLS);
}

// ---------------------------------------------------------------------------------------------
// Pipelined training kernel (the default for the reference's shapes).  Same three GEMMs and epilogues as
// above, as a role-split pipeline of 18 warps (CWT = 16 accumulator columns per epilogue thread):
//
//   warps 0-7   E1 / loader : wait G1(i) -> Z[i&1] -> sigmoid / BCE -> dZ(i) (TMEM hi/lo for G2, transposed smem for G3);
//                             W'(i+2) global -> registers, W'(i+1) -> Wb (hand-over barrier 3), W'(i) transposed -> Wtb
//                             (hand-over barrier 1, once G2/G3(i-1) are done with dZ / Dtb / Wtb)
//   warps 8-15  E2          : old W/m/v rows of tile j from the TMA-filled stage (hand-back barrier 2), wait G3(j) ->
//                             dW'^T[j&1] -> Adam -> global; runs up to two tiles behind the MMA warp
//   warp 16     MMA issuer  : G1(i+1) as soon as W'(i+1) is stored, then G3(i), G2(i); tcgen05.commit onto bar_g1 /
//                             bar_dw[i&1] / bar_g23
//   warp 17     copy        : cp.async.bulk refill of the E2 stage, cp.async.bulk.prefetch.L2 of W/m/v K3_PF_AHEAD tiles ahead
//
// Z and dW'^T are double-buffered in TMEM, so the tensor core works on tile i's backward GEMMs and tile i+1's logits
// while the CUDA cores finish tile i-1; no block-wide barrier inside the tile loop (mbarriers and named barriers only).
// TMEM (512 columns): Z 2x32 | dW'^T 2x32 | dZ hi,lo 2x32 | dh2 Np | H2'^T hi,lo 2x round8(B)
//   -> needs Np + 2*round8(B) <= 320 (n_hidden 100: batch <= 104).
// Bias: lane k == H of dW'^T holds the bias gradients; they are handed to lanes H+1..H+8 of the same warp,
// which run the same Adam code on bd3/mb/vb (one element each) -- no divergent bias path.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t T2_Z = 0, T2_DW = 64, T2_DZH = 128, T2_DZL = 160, T2_DH = 192;

__device__ __forceinline__ void named_bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// MUFU approximations of the BCE fast paths (target 0 and |z| < 16, where ATen's clamped formula, common.cuh bce_term,
// equals softplus(z) / sigmoid(z)/N to far below 1e-6 relative; everything else goes through bce_term).  log(1+u)
// through lg2 has an absolute error of one rounding of 1+u (6e-8, unbiased) per element: invisible in the mean over
// B*V terms; the gradient sigmoid(z)/N is accurate to ~2 ulp.
__device__ __forceinline__ float ex2_approx(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float lg2_approx(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// this thread's share of the W' tile when NW warps split the Kp/4 (<= 32) 16-byte column groups
template <int NCH, int NW>
__device__ __forceinline__ void make_wchunks_t(WChunk* wc, const Geom& g) {
  const int ncg = g.Kp / 4;
  const int r = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < NCH; ++j) {
    int cg = w + NW * j;
    wc[j].goff = -2;
    if (cg < ncg) {
      int c = cg * 4;
      wc[j].goff = (c + 3 < g.H) ? r * g.H + c : (c == g.H ? -1 : -3);
    }
    wc[j].wb_off = (uint32_t)(r >> 3) * g.wb_sbo + (uint32_t)cg * CORE + (uint32_t)(r & 7) * 16u;
    wc[j].wt_off = (uint32_t)(cg >> 1) * g.wt_sbo + (uint32_t)(r >> 2) * g.wt_lbo + (uint32_t)(cg & 1) * 64u +
                   (uint32_t)(r & 3) * 4u;
  }
}
template <int NCH>
__device__ __forceinline__ void load_w_regs_t(float4* wr, const WChunk* wc, const float* __restrict__ Wd3,
                                              const float* __restrict__ bd3, int H, int v0, int nv) {
  const int r = threadIdx.x & 31;
#pragma unroll
  for (int j = 0; j < NCH; ++j) {
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < nv) {
      if (wc[j].goff >= 0) x = __ldcs(reinterpret_cast<const float4*>(Wd3 + (size_t)v0 * H + wc[j].goff));
      else if (wc[j].goff == -1) x.x = __ldg(bd3 + v0 + r);
    }
    wr[j] = x;
  }
}
template <int NCH>
__device__ __forceinline__ void store_wb_regs(const float4* wr, const WChunk* wc, unsigned char* wb_hi,
                                              unsigned char* wb_lo, bool with_lo) {
#pragma unroll
  for (int j = 0; j < NCH; ++j) {
    if (wc[j].goff == -2) continue;
    float4 x = wr[j];
    pin4(x);
    float4 h = make_float4(tf32_hi(x.x), tf32_hi(x.y), tf32_hi(x.z), tf32_hi(x.w));
    *reinterpret_cast<float4*>(wb_hi + wc[j].wb_off) = h;
    if (with_lo) *reinterpret_cast<float4*>(wb_lo + wc[j].wb_off) = make_float4(x.x - h.x, x.y - h.y, x.z - h.z, x.w - h.w);
  }
}
template <int NCH>
__device__ __forceinline__ void store_wt_regs(const float4* wr, const WChunk* wc, unsigned char* wt_hi,
                                              unsigned char* wt_lo, bool with_lo) {
#pragma unroll
  for (int j = 0; j < NCH; ++j) {
    if (wc[j].goff == -2) continue;
    float4 x = wr[j];
    float4 h = make_float4(tf32_hi(x.x), tf32_hi(x.y), tf32_hi(x.z), tf32_hi(x.w));
    float* th = reinterpret_cast<float*>(wt_hi + wc[j].wt_off);
    th[0] = h.x; th[4] = h.y; th[8] = h.z; th[12] = h.w;
    if (with_lo) {
      float* tl = reinterpret_cast<float*>(wt_lo + wc[j].wt_off);
      tl[0] = x.x - h.x; tl[4] = x.y - h.y; tl[8] = x.z - h.z; tl[12] = x.w - h.w;
    }
  }
}

#ifndef K3_PF_MV
#define K3_PF_MV 1
#endif
#ifndef K3_PF_AHEAD
#define K3_PF_AHEAD 4
#endif
#ifdef K3X_TRACE
// timing experiment only: clock64() of CTA 0 at the synchronisation points of tile iterations 8..39
static __device__ long long k3x_tr[32 * 16];
#define K3X_MARK(it, slot) do { if (blockIdx.x == 0 && (it) >= 8 && (it) < 40 && (threadIdx.x & 31) == 0) k3x_tr[((it) - 8) * 16 + (slot)] = clock64(); } while (0)
#else
#define K3X_MARK(it, slot) do { } while (0)
#endif
// CWT = accumulator columns per epilogue thread (8: 16 epilogue warps, 16: 8 fatter warps with twice the
// instruction-level parallelism and half the per-warp fixed work)
template <int CWT> struct Tc2Cfg {
  static constexpr int NPART = TN / CWT;          // column parts per TMEM lane quarter
  static constexpr int NWE = 4 * NPART;           // warps per epilogue role (E1 / loader warps, E2 warps)
  static constexpr int NTT = 32 * NWE + 32;       // one role + the MMA warp (barriers 1, 3) or the copy warp (barrier 2)
  static constexpr int NTHR = 64 * NWE + 64;      // E1 warps | E2 warps | MMA warp | copy warp
  static constexpr int WCHT = 32 / NWE;           // W' chunks per loader thread
  static_assert(NTHR <= 1024, "two epilogue roles of 4*TN/CWT warps each: CWT = 16");
};
// MODE (batches larger than one row chunk are walked chunk by chunk, one launch each; the weight gradient of the
// chunks is summed in a global scratch [Vloc,H] + [Vloc] before the one Adam update):
//   0  single chunk: gradient -> Adam                     1  first chunk:  gW  = dW'   (no Adam, no W/m/v stage)
//   2  middle chunk: gW += dW'                            3  last chunk:   Adam with gW + dW'
template <int SPLIT, int HC, int CWT, int MODE>
__global__ void __launch_bounds__(Tc2Cfg<CWT>::NTHR, 1) dec_out_train_tc2_kernel(
    const float* __restrict__ h2, int B, int Hrt, float* __restrict__ Wd3, float* __restrict__ bd3,
    float* __restrict__ mW, float* __restrict__ vW, float* __restrict__ mb, float* __restrict__ vb, int v_begin,
    int Vloc, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices, float inv_n,
    const aae_step_state* __restrict__ st, float* __restrict__ dh2, double* __restrict__ loss_sum, int smem_total,
    float* __restrict__ gW, float* __restrict__ gB) {
  constexpr bool kAdam = (MODE == 0 || MODE == 3);     // this launch applies dec_optim
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ uint64_t bar_g1, bar_g23;   // completion of G1(i) / of G3(i-1)+G2(i-1)
  __shared__ uint64_t bar_stage;         // E2 stage (W/m/v rows of one tile) filled by TMA
  __shared__ uint64_t bar_dw[2];         // G3(i) complete: dW'^T buffer i&1 may be read by the E2 warps
  __shared__ uint64_t bar_dwfree[2];     // the E2 warps have read dW'^T buffer i&1 (one arrival per warp)
  __shared__ uint32_t tmem_base_s;
  constexpr int NPART = Tc2Cfg<CWT>::NPART, NWE = Tc2Cfg<CWT>::NWE, NTT = Tc2Cfg<CWT>::NTT, WCHT = Tc2Cfg<CWT>::WCHT;
  constexpr int NTHR = Tc2Cfg<CWT>::NTHR;
  __shared__ float red[NWE];
  const int H = HC ? HC : Hrt;
  const Geom g = make_geom(H);
  constexpr bool with_lo = (SPLIT == 3);
  const int BK = (B + 7) & ~7;
  // Hb keeps only round8(B) rows: the M = 128 MMA reads the rows beyond from whatever follows in shared
  // memory (finite numbers: everything is zero-filled first), and those logit rows are never used.
  const uint32_t hb_eff = (uint32_t)(BK / 8) * g.hb_sbo;
  unsigned char* hb_hi = smem;
  unsigned char* hb_lo = hb_hi + hb_eff;
  unsigned char* wb_hi = hb_lo + hb_eff;
  unsigned char* wb_lo = wb_hi + g.wb_bytes;
  unsigned char* wt_hi = wb_lo + g.wb_bytes;
  unsigned char* wt_lo = wt_hi + g.wt_bytes;
  unsigned char* dt_hi = wt_lo + g.wt_bytes;
  unsigned char* dt_lo = dt_hi + g.dt_bytes;
  float* sW = reinterpret_cast<float*>(dt_lo + g.dt_bytes);
  float* sM = sW + TN * H;
  float* sV = sM + TN * H;
  float* sB = sV + TN * H;               // [3][TN]: bd3, mb, vb of the tile
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_tiles = (Vloc + TN - 1) / TN;
  const int G = gridDim.x;
  const int n_my = (n_tiles - (int)blockIdx.x + G - 1) / G;     // tiles blockIdx.x, +G, ... (grid <= n_tiles)
  const uint32_t T2_HTH = T2_DH + (uint32_t)g.Np, T2_HTL = T2_HTH + (uint32_t)BK;

  trace_mark(TR_K3, 0);
  if (warp == 0) K3X_MARK(39, 0);
  if (warp == 2 * NWE) tmem_alloc(&tmem_base_s, TMEM_COLS);
  if (tid == 0) {
    mbar_init(&bar_g1, 1);
    mbar_init(&bar_g23, 1);
    mbar_init(&bar_stage, 1);
    mbar_init(&bar_dw[0], 1);
    mbar_init(&bar_dw[1], 1);
    mbar_init(&bar_dwfree[0], NWE);
    mbar_init(&bar_dwfree[1], NWE);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // The loads of the prologue are issued in batches (all loads of a batch before their first use): issued one by one
  // they cost a global-memory round trip each, 12 us of every launch before the first tile.
  constexpr int HB_BATCH = 5;
  const int ncg0 = g.Kp / 4;
  float4 hbx[HB_BATCH];
#pragma unroll
  for (int u = 0; u < HB_BATCH; ++u) {                       // first batch of the Hb fill: in flight during the zero fill
    const int q = tid + u * NTHR;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q < BK * ncg0) {
      const int r = q / ncg0, c = (q - r * ncg0) * 4;
      if (r < B) {
        if (c + 3 < H) x = *reinterpret_cast<const float4*>(h2 + (size_t)r * H + c);
        else if (c == H) x.x = 1.0f;
      }
    }
    hbx[u] = x;
  }
  for (int q = tid; q < smem_total / 16; q += NTHR) reinterpret_cast<float4*>(smem)[q] = make_float4(0, 0, 0, 0);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  if (warp == 0) K3X_MARK(39, 1);
  if (warp < 2 * NWE) {
    // H2'^T -> TMEM (lane = hidden unit, column = batch row), BK columns; all epilogue warps, two 8-column chunks at a time
    const int q4 = warp & 3, part = warp >> 2;               // TMEM lane quarter; chunk phase
    const uint32_t lane_addr = tmem + ((uint32_t)(q4 * 32) << 16);
    const int k = q4 * 32 + lane;
    constexpr int NP4 = 2 * NPART;
    for (int c0 = part; c0 < BK / 8; c0 += 2 * NP4) {
      float x[16];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int c = c0 + u * NP4;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int b = c * 8 + j;
          float v = 0.f;
          if (c < BK / 8 && b < B) v = (k < H) ? h2[(size_t)b * H + k] : (k == H ? 1.0f : 0.f);
          x[u * 8 + j] = v;
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int c = c0 + u * NP4;
        if (c < BK / 8) {
          float hi[8], lo[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            hi[j] = tf32_hi(x[u * 8 + j]);
            lo[j] = x[u * 8 + j] - hi[j];
          }
          tmem_st8(lane_addr + T2_HTH + c * 8, hi);
          if (with_lo) tmem_st8(lane_addr + T2_HTL + c * 8, lo);
        }
      }
    }
    tmem_st_wait();
  }
#pragma unroll
  for (int u = 0; u < HB_BATCH; ++u) {
    const int q = tid + u * NTHR;
    if (q < BK * ncg0) {
      const int r = q / ncg0, cg = q - r * ncg0;
      store_split4(hb_hi, hb_lo, r, cg, g.hb_sbo, hbx[u], with_lo);
    }
  }
  for (int q = tid + HB_BATCH * NTHR; q < BK * ncg0; q += NTHR) {      // shapes beyond HB_BATCH chunks per thread
    int r = q / ncg0, cg = q - r * ncg0;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < B) {
      int c = cg * 4;
      if (c + 3 < H) x = *reinterpret_cast<const float4*>(h2 + (size_t)r * H + c);
      else if (c == H) x.x = 1.0f;
    }
    store_split4(hb_hi, hb_lo, r, cg, g.hb_sbo, x, with_lo);
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t idesc_g1 = make_idesc(BM, TN, 0, 0);
  const uint32_t idesc_g2 = make_idesc(BM, g.Np, 0, 0);
  if (warp == 0) K3X_MARK(39, 2);

  if (warp == 2 * NWE) {
    // ================= MMA issuer =================
    // Two hand-overs per tile: barrier 3 = W'(it) is in Wb -> G1(it) is issued at once, one tile ahead of the backward
    // GEMMs, so the tensor pipe has work while the epilogue warps are busy with the operand stores of tile it-1;
    // barrier 1 = dZ(it-1), Dtb and Wtb are stored -> G3(it-1), G2(it-1).
    const SmemOp op_hb = make_op(hb_hi, hb_lo, CORE, g.hb_sbo, 2 * CORE);
    const SmemOp op_wb = make_op(wb_hi, wb_lo, CORE, g.wb_sbo, 2 * CORE);
    // (MN-major B operands -- SWIZZLE_128B_BASE32B, probed in aae_tc_selftest modes 6/7 -- would let Wtb / Dtb be written
    // as 16-byte vectors instead of transposing scalars, but the tensor pipe reads them ~50 % slower: measured, dropped)
    const SmemOp op_wt = make_op(wt_hi, wt_lo, g.wt_lbo, g.wt_sbo, 2 * g.wt_lbo);
    const SmemOp op_dt = make_op(dt_hi, dt_lo, g.dt_lbo, g.dt_sbo, 2 * g.dt_lbo);
    const uint32_t idesc_g3 = idesc_g1, idesc_g2n = idesc_g2;
    const int ksteps_b = BK / 8;
    uint32_t ph_f0 = 0, ph_f1 = 0;
    for (int it = 0; it <= n_my; ++it) {
      // K3X_* (here and below): timing experiments only (scripts/k3_experiments.sh); never defined in the product build
      if (it < n_my) {
        named_bar_sync(3, NTT);
        tc_fence_after();
        K3X_MARK(it, 0);
        if (elect_one()) {
#ifndef K3X_NO_G1
          issue_gemm<SPLIT>(tmem + T2_Z + (uint32_t)(it & 1) * 32u, op_hb, op_wb, g.Kp / 8, idesc_g1, 0u);
#endif
          mma_commit(&bar_g1);
        }
        __syncwarp();
        K3X_MARK(it, 1);
      }
      if (it > 0) {
        named_bar_sync(1, NTT);
        tc_fence_after();
        K3X_MARK(it, 14);
      }
      if (it > 2) {                 // G3(it-1) overwrites the dW'^T buffer that E2(it-3) reads
        if ((it - 1) & 1) { mbar_wait_backoff(&bar_dwfree[1], ph_f1); ph_f1 ^= 1; } else { mbar_wait_backoff(&bar_dwfree[0], ph_f0); ph_f0 ^= 1; }
        tc_fence_after();
      }
      if (elect_one()) {
        if (it > 0) {
          const uint32_t bo = (uint32_t)((it - 1) & 1) * 32u;
#ifndef K3X_NO_G3
          issue_gemm_ts<SPLIT>(tmem + T2_DW + bo, tmem + T2_HTH, tmem + T2_HTL, op_dt, ksteps_b, idesc_g3, 0u);
#endif
          mma_commit(&bar_dw[(it - 1) & 1]);       // the E2 warps start on dW'^T without waiting for G2
#ifndef K3X_NO_G2
          issue_gemm_ts<SPLIT>(tmem + T2_DH, tmem + T2_DZH, tmem + T2_DZL, op_wt, TN / 8, idesc_g2n, it > 1 ? 1u : 0u);
#endif
          (void)bo;
        }
        mma_commit(&bar_g23);      // it == 0: nothing pending, completes at once (the epilogue's first wait)
      }
      __syncwarp();
      K3X_MARK(it, 15);
    }
  } else if (warp == 2 * NWE + 1) {
    // ================= copy warp: E2 stage refill, L2 prefetch =================
    // The stage holds the W/m/v rows (and bias triplets) of ONE tile; it is refilled as soon as the E2 warps have read
    // it into registers (barrier 2), while they are still computing and storing.
    auto stage_copy = [&](int j) {
      const int v0 = ((int)blockIdx.x + j * G) * TN;
      if (kAdam && Vloc - v0 >= TN) {
        const uint32_t wbytes = (uint32_t)(TN * H) * 4u, bbytes = TN * 4u;
        mbar_arrive_expect_tx(&bar_stage, 3u * wbytes + 3u * bbytes);
        bulk_g2s(sW, Wd3 + (size_t)v0 * H, wbytes, &bar_stage);
        bulk_g2s(sM, mW + (size_t)v0 * H, wbytes, &bar_stage);
        bulk_g2s(sV, vW + (size_t)v0 * H, wbytes, &bar_stage);
        bulk_g2s(sB, bd3 + v0, bbytes, &bar_stage);
        bulk_g2s(sB + TN, mb + v0, bbytes, &bar_stage);
        bulk_g2s(sB + 2 * TN, vb + v0, bbytes, &bar_stage);
      } else {
        mbar_arrive(&bar_stage);     // ragged last tile / no Adam in this launch: E2 works on global memory
      }
    };
    // L2 prefetch, K3_PF_AHEAD tiles ahead: the W rows that the loader warps read and (K3_PF_MV) the m/v rows and
    // bias triplets of the stage, so that the HBM streams of the next tiles stay open while this tile computes.
    auto prefetch_w = [&](int j) {
      if (j >= n_my) return;
      const int v0 = ((int)blockIdx.x + j * G) * TN;
      const int nv = min(TN, Vloc - v0);
      const uint32_t wbytes = (uint32_t)nv * (uint32_t)H * 4u;
      if (j >= 2) prefetch_l2_bulk(Wd3 + (size_t)v0 * H, wbytes);
      if (!kAdam) return;
#if K3_PF_MV
      prefetch_l2_bulk(mW + (size_t)v0 * H, wbytes);
      prefetch_l2_bulk(vW + (size_t)v0 * H, wbytes);
      if (nv == TN) {
        prefetch_l2_bulk(bd3 + v0, TN * 4u);
        prefetch_l2_bulk(mb + v0, TN * 4u);
        prefetch_l2_bulk(vb + v0, TN * 4u);
      }
#endif
    };
    if (lane == 0) {
      stage_copy(0);
      for (int j = 1; j < K3_PF_AHEAD; ++j) prefetch_w(j);
    }
    __syncwarp();
    for (int j = 1; j < n_my; ++j) {
      if (lane == 0) prefetch_w(j + K3_PF_AHEAD - 1);
      named_bar_sync(2, NTT);          // E2(j-1) has read the stage
      if (lane == 0) stage_copy(j);
      __syncwarp();
    }
  } else if (warp < NWE) {
    // ================= E1 / loader warps: logits -> dZ, the W' tile -> Wb / Wtb =================
    const int q4 = warp & 3, cpart = warp >> 2;      // TMEM lane quarter, CWT-column part of the 32-wide tile
    const uint32_t lane_addr = tmem + ((uint32_t)(q4 * 32) << 16);
    const int brow = q4 * 32 + lane;                 // batch row of this thread
    if (warp == 0) K3X_MARK(39, 3);
    const uint32_t dt_off = (uint32_t)(cpart * (CWT / 8)) * g.dt_sbo + (uint32_t)(brow >> 2) * g.dt_lbo + (uint32_t)(brow & 3) * 4u;
    const float inv_n_row = (brow < B) ? inv_n : 0.f;
    WChunk wc[WCHT];
    make_wchunks_t<WCHT, NWE>(wc, g);
    float4 wA[WCHT], wB[WCHT];
    {
      const int t0 = blockIdx.x;
      load_w_regs_t<WCHT>(wA, wc, Wd3, bd3, H, t0 * TN, min(TN, Vloc - t0 * TN));
      store_wb_regs<WCHT>(wA, wc, wb_hi, wb_lo, with_lo);
      if (n_my > 1) load_w_regs_t<WCHT>(wB, wc, Wd3, bd3, H, (t0 + G) * TN, min(TN, Vloc - (t0 + G) * TN));
    }
    fence_async_smem();
    tc_fence_before();
    named_bar_arrive(3, NTT);                        // W'(0) is in Wb
    if (warp == 0) K3X_MARK(39, 5);
    // Positives of this thread's row inside THIS CTA's tiles, found once (while G1 of the first tile runs): a row has
    // ~|set|/gridDim items per CTA, so up to four (tile iteration, CWT-bit column mask) events live in registers and
    // the tile loop only compares its counter with the next event.  More than four: per-tile bisection of the row (rare).
    constexpr uint32_t EV_NONE = 0xffffffffu;
    uint32_t ev0 = EV_NONE, ev1 = EV_NONE, ev2 = EV_NONE, ev3 = EV_NONE;   // (iteration << 16) | mask of my CWT columns
    bool ev_over = false;
    int row_p0 = 0, row_p1 = 0;
    if (brow < B) {
      row_p0 = indptr[brow];
      row_p1 = indptr[brow + 1];
      uint32_t last_it = EV_NONE >> 16;
      for (int p0 = row_p0; p0 < row_p1; p0 += 8) {
        int vv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) vv[u] = (p0 + u < row_p1) ? __ldg(indices + p0 + u) - v_begin : -1;   // 8 loads in flight
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int v = vv[u];
          if (v < 0 || v >= Vloc) continue;
          const int t = v / TN;
          if (t % G != (int)blockIdx.x) continue;
          const int col = v - t * TN;
          if (col / CWT != cpart) continue;             // another warp's columns
          const uint32_t it_ = (uint32_t)(t / G), bit = 1u << (col % CWT);
          if (it_ == last_it) {                          // same tile as the previous event: merge
            if (ev3 != EV_NONE) ev3 |= bit;
            else if (ev2 != EV_NONE) ev2 |= bit;
            else if (ev1 != EV_NONE) ev1 |= bit;
            else ev0 |= bit;
          } else {
            const uint32_t e = (it_ << 16) | bit;
            if (ev0 == EV_NONE) ev0 = e;
            else if (ev1 == EV_NONE) ev1 = e;
            else if (ev2 == EV_NONE) ev2 = e;
            else if (ev3 == EV_NONE) ev3 = e;
            else ev_over = true;
            last_it = it_;
          }
        }
      }
    }
    if (warp == 0) K3X_MARK(39, 4);
    uint32_t phase = 0;
    float loss_local = 0.f;

    for (int i = 0; i < n_my; ++i) {
      const int tile = blockIdx.x + i * G;
      const int v0 = tile * TN;
      const int nv = min(TN, Vloc - v0);
      // positives of this tile among this thread's CWT columns
      uint32_t tb = 0u;
      if ((ev0 >> 16) == (uint32_t)i) {
        tb = ev0 & 0xffffu;
        ev0 = ev1; ev1 = ev2; ev2 = ev3; ev3 = EV_NONE;
      }
      if (ev_over) {                                   // overflowed event list: bisect the row for this tile
        const int lo_item = v_begin + v0 + cpart * CWT;
        int lo = row_p0, hi = row_p1;
        while (lo < hi) {
          int mid = (lo + hi) >> 1;
          if (__ldg(indices + mid) < lo_item) lo = mid + 1; else hi = mid;
        }
        tb = 0u;
        for (int p = lo; p < row_p1; ++p) {
          int d = __ldg(indices + p) - lo_item;
          if (d >= CWT) break;
          tb |= 1u << d;
        }
      }
      const int vm = nv - cpart * CWT;                 // valid columns of this thread's CWT (>= CWT: all)

      // ---- E1(i), math part: needs only G1(i)
      if (warp == 0) K3X_MARK(i, 2);
      mbar_wait_backoff(&bar_g1, phase);
      tc_fence_after();
      if (warp == 0) K3X_MARK(i, 3);
      float dzh[CWT], dzl[CWT];
      {
        float z[CWT];
        uint32_t zr[CWT];
        TmemIO<CWT>::ld_issue(lane_addr + T2_Z + (uint32_t)(i & 1) * 32u + cpart * CWT, zr);
        // W'(i+1) for G1(i+1): G1(i) has finished reading the buffer; handed to the MMA warp at once
        if (i + 1 < n_my) {
          store_wb_regs<WCHT>(wB, wc, wb_hi, wb_lo, with_lo);
          fence_async_smem();
          named_bar_arrive(3, NTT);
        }
        TmemIO<CWT>::ld_wait(zr);
#pragma unroll
        for (int j = 0; j < CWT; ++j) z[j] = __uint_as_float(zr[j]);
        float zhi = -3.0e38f, zlo = 3.0e38f;
#pragma unroll
        for (int j = 0; j < CWT; ++j) {
          zhi = fmaxf(zhi, z[j]);
          zlo = fminf(zlo, z[j]);
        }
        // Four paths.  The target is 0 nearly everywhere, and for target 0 and z < 16 ATen's clamped formula
        // (common.cuh bce_term) equals softplus(z) / sigmoid(z)/N to far below 1e-6 relative -- for ANY negative depth:
        // below z = -16.6 ATen's own fp32 loss term log(1 - x) is exactly 0, as is log(1 + e^z) here.
        //   P0  whole warp clean and z <= 0 (the usual state of a model after a few dozen steps: mean logit -5 .. -10):
        //       sigmoid = 1/(1+e^-z), loss = -log(1 - sigmoid) as ATen writes it, ONE lg2 per four elements, any depth
        //   P1  whole warp clean and -16 < z < 16 (mixed signs, the first steps): loss = z + log(1+e^-z), which cancels
        //       for deep-negative z -- hence the -16
        //   P2  this thread clean (no positive, full tile, z < 16), mixed signs and deep: through e^-|z|
        //   P3  per element: positives, z >= 16 and ragged tiles through bce_term, the rest as in P2
        // Logits below -16 are everyday values; when they took the per-element path the whole warp waited for it and
        // the kernel ran 1.7x slower (2.0 instead of 1.2 ms at V = 2M).  Rows >= B (dead lanes) never veto a warp path.
        const bool live = brow < B;
        const bool clean = (tb == 0u) && (vm >= CWT) && (zhi < 16.0f);
        if (__all_sync(0xffffffffu, !live || (clean && zhi <= 0.0f))) {
          float pr[CWT / 4];
#pragma unroll
          for (int q = 0; q < CWT / 4; ++q) pr[q] = 1.0f;
#pragma unroll
          for (int j = 0; j < CWT; ++j) {
            const float u = ex2_approx(-1.4426950408889634f * z[j]);     // e^-z >= 1
            const float r = rcp_approx(1.0f + u);                         // sigmoid(z) in (0, 0.5]
            const float d = r * inv_n_row;
            pr[j >> 2] *= 1.0f - r;                                        // in [0.5, 1]: no cancellation
            const float h = tf32_hi(d);
            dzh[j] = h;
            dzl[j] = d - h;
          }
          float lg = 0.f;
#pragma unroll
          for (int q = 0; q < CWT / 4; ++q) lg += lg2_approx(pr[q]);
          if (live) loss_local = fmaf(lg, -0.6931471805599453f, loss_local);
        } else if (__all_sync(0xffffffffu, !live || (clean && zlo > -16.0f))) {
          // sigmoid(z) = 1/(1+e^-z) and -log(1-sigmoid(z)) = z + log(1+e^-z); the logarithms of four elements are taken
          // as ONE lg2 of the product of their (1+e^-z) <= 8.9e6 (product < 6.3e27): 7 FP32 + 2 MUFU per element
          float sz = 0.f;
          float pr[CWT / 4];
#pragma unroll
          for (int q = 0; q < CWT / 4; ++q) pr[q] = 1.0f;
#pragma unroll
          for (int j = 0; j < CWT; ++j) {
#ifdef K3X_NO_E1MATH
            const float u = z[j], t = 1.0f + u;
            const float d = t * inv_n_row;
#else
            const float u = ex2_approx(-1.4426950408889634f * z[j]);
            const float t = 1.0f + u;
            const float d = rcp_approx(t) * inv_n_row;
#endif
            sz += z[j];
            pr[j >> 2] *= t;
            const float h = tf32_hi(d);
            dzh[j] = h;
            dzl[j] = d - h;
          }
          float lg = 0.f;
#pragma unroll
          for (int q = 0; q < CWT / 4; ++q) lg += lg2_approx(pr[q]);
          if (live) loss_local += fmaf(lg, 0.6931471805599453f, sz);
        } else if (clean) {
          // u = e^-|z| in (0,1]: sigmoid(z) = 1/(1+u) or u/(1+u), softplus(z) = max(z,0) + log(1+u); products <= 16
          float sz = 0.f;
          float pr[CWT / 4];
#pragma unroll
          for (int q = 0; q < CWT / 4; ++q) pr[q] = 1.0f;
#pragma unroll
          for (int j = 0; j < CWT; ++j) {
            const float u = ex2_approx(-1.4426950408889634f * fabsf(z[j]));
            const float t = 1.0f + u;
            const float r = rcp_approx(t);
            const float d = ((z[j] >= 0.f) ? r : u * r) * inv_n_row;
            sz += fmaxf(z[j], 0.f);
            pr[j >> 2] *= t;
            const float h = tf32_hi(d);
            dzh[j] = h;
            dzl[j] = d - h;
          }
          float lg = 0.f;
#pragma unroll
          for (int q = 0; q < CWT / 4; ++q) lg += lg2_approx(pr[q]);
          if (live) loss_local += fmaf(lg, 0.6931471805599453f, sz);
        } else {
#pragma unroll
          for (int j = 0; j < CWT; ++j) {
            float d = 0.f;
            if (brow < B && j < vm) {
              const uint32_t tgt = (tb >> j) & 1u;
              if (tgt != 0u || z[j] >= 16.0f) {
                loss_local += bce_term(z[j], tgt, inv_n, d);
              } else {
                const float u = ex2_approx(-1.4426950408889634f * fabsf(z[j]));
                const float t = 1.0f + u;
                const float r = rcp_approx(t);
                d = ((z[j] >= 0.f) ? r : u * r) * inv_n;
                loss_local += fmaf(lg2_approx(t), 0.6931471805599453f, fmaxf(z[j], 0.f));
              }
            }
            float h = tf32_hi(d);
            dzh[j] = h;
            dzl[j] = d - h;
          }
        }
      }
      // ---- operand stores: need G2/G3(i-1) to be done with dZ, Dtb and Wtb
      if (warp == 0) K3X_MARK(i, 4);
      mbar_wait_backoff(&bar_g23, phase);
      phase ^= 1;
      tc_fence_after();
      if (warp == 0) K3X_MARK(i, 5);
#pragma unroll
      for (int j = 0; j < CWT; ++j) {
        const uint32_t o = dt_off + (uint32_t)(j >> 3) * g.dt_sbo + (uint32_t)(j & 7) * 16u;
        *reinterpret_cast<float*>(dt_hi + o) = dzh[j];
        if (with_lo) *reinterpret_cast<float*>(dt_lo + o) = dzl[j];
      }
      TmemIO<CWT>::st(lane_addr + T2_DZH + cpart * CWT, dzh);
      if (with_lo) TmemIO<CWT>::st(lane_addr + T2_DZL + cpart * CWT, dzl);
#ifndef K3X_NO_WT
      store_wt_regs<WCHT>(wA, wc, wt_hi, wt_lo, with_lo);              // W'(i) transposed for G2(i)
#endif
      tmem_st_wait();
      fence_async_smem();
      tc_fence_before();
      named_bar_arrive(1, NTT);
      if (warp == 0) K3X_MARK(i, 6);
#pragma unroll
      for (int j = 0; j < WCHT; ++j) wA[j] = wB[j];
      if (i + 2 < n_my) {
        const int t2 = tile + 2 * G;
        load_w_regs_t<WCHT>(wB, wc, Wd3, bd3, H, t2 * TN, min(TN, Vloc - t2 * TN));
      }
    }
    mbar_wait_backoff(&bar_g23, phase);                       // G2/G3 of the last tile
    tc_fence_after();
    if (warp == 0) K3X_MARK(39, 6);
    // ---- flush dh2 (lane = batch row, columns = hidden unit) while the E2 warps finish the last tile; the column
    // order is rotated per CTA so that the 148 CTAs, which finish together, do not all hit the same addresses at once
    {
      const int nch = g.Np / CWT;
      const int rot = (int)(blockIdx.x % (unsigned)nch);
      for (int c = cpart; c < nch; c += NPART) {
        int cc = c + rot;
        if (cc >= nch) cc -= nch;
        float d[CWT];
        {
          uint32_t dr[CWT];
          TmemIO<CWT>::ld_issue(lane_addr + T2_DH + cc * CWT, dr);
          TmemIO<CWT>::ld_wait(dr);
#pragma unroll
          for (int j = 0; j < CWT; ++j) d[j] = __uint_as_float(dr[j]);
        }
        if (brow < B) {
          float* dst = dh2 + (size_t)brow * H + cc * CWT;       // H % 4 == 0: 16-byte aligned groups of 4
#pragma unroll
          for (int j = 0; j < CWT; j += 4) {
            if (cc * CWT + j + 3 < H)
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + j), "f"(d[j]), "f"(d[j + 1]),
                           "f"(d[j + 2]), "f"(d[j + 3])
                           : "memory");
          }
        }
      }
    }
    float s = warp_sum(loss_local);
    if (lane == 0) red[warp] = s;
    if (warp == 0) K3X_MARK(39, 7);
  } else {
    // ================= E2 warps: dW'^T(j) -> dec_optim on the W/m/v rows of tile j =================
    // Lane = hidden unit k (the TMEM lane of dW'^T), CWT item rows at pitch H.  Lanes H+1..H+CWT of the warp that
    // holds lane H own one bias element each: the bias gradients (lane H) are handed to them by shuffles and they
    // run the same Adam code on bd3/mb/vb -- no divergent bias path.
    const int we = warp - NWE;
    const int q4 = we & 3, cpart = we >> 2;
    const uint32_t lane_addr = tmem + ((uint32_t)(q4 * 32) << 16);
    const int brow = q4 * 32 + lane;                 // hidden unit of this thread
    const AdamK ak = adam_load(st, 0);
    const int kb = H & 31;                           // lane of hidden unit H inside its warp
    const bool bias_warp = (q4 == (H >> 5));
    const int jb = brow - (H + 1);                   // bias lanes: 0..CWT-1
    const bool is_bias = (jb >= 0 && jb < CWT);
    float* const eW = is_bias ? bd3 : Wd3;
    float* const eM = is_bias ? mb : mW;
    float* const eV = is_bias ? vb : vW;
    const float* const sWp = is_bias ? sB + cpart * CWT + jb : sW + cpart * CWT * H + brow;
    const float* const sMp = is_bias ? sB + TN + cpart * CWT + jb : sM + cpart * CWT * H + brow;
    const float* const sVp = is_bias ? sB + 2 * TN + cpart * CWT + jb : sV + cpart * CWT * H + brow;
    const int ecnt_full = is_bias ? 1 : (brow < H ? CWT : 0);
    uint32_t phase_e = 0, ph_dw0 = 0, ph_dw1 = 0;
    const uint32_t rt_zero = (uint32_t)smem_total >> 31;
    for (int jt = 0; jt < n_my; ++jt) {
      const int tile = blockIdx.x + jt * G;
      const int v0 = tile * TN;
      const int nv = min(TN, Vloc - v0);
      size_t eoff;
      int ecnt;
      if (is_bias) {
        eoff = (size_t)v0 + cpart * CWT + jb;
        ecnt = (cpart * CWT + jb < nv) ? 1 : 0;
      } else {
        eoff = (size_t)(v0 + cpart * CWT) * H + brow;
        ecnt = (brow < H) ? max(0, min(CWT, nv - cpart * CWT)) : 0;
      }
      float* pW = eW + eoff;
      float* pM = eM + eoff;
      float* pV = eV + eoff;
      float* pG = (MODE != 0) ? ((is_bias ? gB : gW) + eoff) : nullptr;
      float pw[CWT], pm[CWT], pv[CWT], pg[CWT];
#pragma unroll
      for (int j = 0; j < CWT; ++j) pw[j] = pm[j] = pv[j] = 0.f;
      if (MODE == 2 || MODE == 3) {                      // gradient of the earlier chunks (coalesced over the lanes)
#pragma unroll
        for (int j = 0; j < CWT; ++j) pg[j] = (j < ecnt) ? pG[(size_t)j * H] : 0.f;
      }
      // old W/m/v from the TMA-filled stage; the stage is handed back for the refill as soon as it has been read
      if (warp == NWE) K3X_MARK(jt, 8);
      mbar_wait_backoff(&bar_stage, phase_e);
      phase_e ^= 1;
      if (warp == NWE) K3X_MARK(jt, 9);
#ifdef K3X_NO_E2LD
      if (false) {
#else
      if (kAdam) {
#endif
        if (nv == TN) {
#pragma unroll
          for (int j = 0; j < CWT; ++j) {
            if (j < ecnt_full) {
              pw[j] = sWp[j * H];
              pm[j] = sMp[j * H];
              pv[j] = sVp[j * H];
            }
          }
        } else {
#pragma unroll
          for (int j = 0; j < CWT; ++j) {
            if (j < ecnt) {
              pw[j] = pW[(size_t)j * H];
              pm[j] = pM[(size_t)j * H];
              pv[j] = pV[(size_t)j * H];
            }
          }
        }
      }
      if (jt + 1 < n_my) {
        // The stage may be refilled (tile jt + 1) -- but only once the loads above have RETURNED: bar.arrive does not
        // order earlier shared-memory reads, and the refill (an L2 hit) can overtake loads that are still queued behind
        // the other warps' traffic.  The barrier id is made to depend on every loaded register (rt_zero is 0 at run time).
        uint32_t dep = 0u;
#pragma unroll
        for (int j = 0; j < CWT; ++j) dep ^= __float_as_uint(pw[j]) ^ __float_as_uint(pm[j]) ^ __float_as_uint(pv[j]);
        named_bar_arrive(2 + (int)(dep & rt_zero), NTT);
      }
      // dW'^T(jt): its own mbarrier per TMEM buffer (these warps run behind the MMA warp by up to two tiles)
      if (jt & 1) { mbar_wait_backoff(&bar_dw[1], ph_dw1); ph_dw1 ^= 1; } else { mbar_wait_backoff(&bar_dw[0], ph_dw0); ph_dw0 ^= 1; }
      tc_fence_after();
      if (warp == NWE) K3X_MARK(jt, 10);
      float gw[CWT];
      {
        uint32_t gr[CWT];
        TmemIO<CWT>::ld_issue(lane_addr + T2_DW + (uint32_t)(jt & 1) * 32u + cpart * CWT, gr);
        TmemIO<CWT>::ld_wait(gr);
#pragma unroll
        for (int j = 0; j < CWT; ++j) gw[j] = __uint_as_float(gr[j]);
      }
      // this dW'^T buffer may be overwritten by G3(jt + 2)
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_dwfree[jt & 1]);
      if (bias_warp) {
        float gb = 0.f;
#pragma unroll
        for (int j = 0; j < CWT; ++j) {
          float t = __shfl_sync(0xffffffffu, gw[j], kb);
          if (jb == j) gb = t;
        }
        if (is_bias) gw[0] = gb;
      }
      if (MODE == 2 || MODE == 3) {
#pragma unroll
        for (int j = 0; j < CWT; ++j) gw[j] += pg[j];
      }
      if (kAdam) {
        // Adam (common.cuh adam_update, same operations in the same order per element), written stage by stage over the
        // CWT independent elements: the per-element chain is ~10 dependent instructions incl. two MUFU.
        float dn[CWT];
#ifndef K3X_NO_E2MATH
#pragma unroll
        for (int j = 0; j < CWT; ++j) pm[j] = fmaf(ak.w1, gw[j] - pm[j], pm[j]);
#pragma unroll
        for (int j = 0; j < CWT; ++j) pv[j] = fmaf(ak.w2 * gw[j], gw[j], pv[j] * ak.beta2);
#pragma unroll
        for (int j = 0; j < CWT; ++j) dn[j] = fmaf(sqrt_approx(pv[j]), ak.inv_bc2_sqrt, ak.eps);
#pragma unroll
        for (int j = 0; j < CWT; ++j) dn[j] = pm[j] * rcp_approx(dn[j]);
#pragma unroll
        for (int j = 0; j < CWT; ++j) pw[j] = fmaf(-ak.step_size, dn[j], pw[j]);
#else
#pragma unroll
        for (int j = 0; j < CWT; ++j) { dn[j] = gw[j]; pw[j] += dn[j]; }
#endif
#ifndef K3X_NO_E2ST
#pragma unroll
        for (int j = 0; j < CWT; ++j) {
          if (j < ecnt) {
            pW[(size_t)j * H] = pw[j];
            __stcs(pM + (size_t)j * H, pm[j]);
            __stcs(pV + (size_t)j * H, pv[j]);
          }
        }
#else
        if (pw[0] + pm[1] + pv[2] == 1.2345e30f) pW[0] = pw[3];      // keep the values alive
#endif
      } else {
#pragma unroll
        for (int j = 0; j < CWT; ++j)
          if (j < ecnt) pG[(size_t)j * H] = gw[j];
      }
      if (warp == NWE) K3X_MARK(jt, 7);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (tid == 0) {
    double tot = 0.0;
    for (int w = 0; w < NWE; ++w) tot += (double)red[w];
    atomicAdd(loss_sum, tot);
  }
  if (warp == 0) K3X_MARK(39, 8);
  if (warp == 2 * NWE) tmem_dealloc(tmem, TMEM_COLS);
  trace_mark(TR_K3, 1);
}

// ---------------------------------------------------------------------------------------------
// self-test kernel: one GEMM form at a time, operands filled from global, TMEM dumped to global
//   mode 1 (G1 form, A and B in smem):  D[128,32]  = A[128,104]      . Bm[32,104]^T
//   mode 2 (G2 form, A in TMEM):        D[128,112] = A[128,32]       . Bm[112,32]^T
//   mode 3 (G3 form, A in TMEM):        D[128,32]  = A[128,128]      . Bm[32,128]^T
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT, 1) tc_selftest_kernel(int mode_in, const float* __restrict__ A,
                                                            const float* __restrict__ Bm, float* __restrict__ D,
                                                            int split) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ uint64_t bar_mma;
  __shared__ uint32_t tmem_base_s;
  const Geom g = make_geom(100);
  int mode = mode_in;
  unsigned char* hb_hi = smem;
  unsigned char* hb_lo = hb_hi + g.hb_bytes;
  unsigned char* wb_hi = hb_lo + g.hb_bytes;
  unsigned char* wb_lo = wb_hi + g.wb_bytes;
  unsigned char* wt_hi = wb_lo + g.wb_bytes;
  unsigned char* wt_lo = wt_hi + g.wt_bytes;
  unsigned char* dt_hi = wt_lo + g.wt_bytes;
  unsigned char* dt_lo = dt_hi + g.dt_bytes;
  const bool with_lo = (split == 3);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q4 = warp & 3, cpart = warp >> 2;
  if (warp == 0) tmem_alloc(&tmem_base_s, TMEM_COLS);
  if (tid == 0) {
    mbar_init(&bar_mma, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int q = tid; q < (int)(smem_bytes(g) - 256) / 16; q += NT) reinterpret_cast<float4*>(smem)[q] = make_float4(0, 0, 0, 0);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const uint32_t lane_addr = tmem + ((uint32_t)(q4 * 32) << 16);
  const int row = q4 * 32 + lane;
  auto split_store = [&](unsigned char* hi, unsigned char* lo, int r, int c, uint32_t lbo, uint32_t sbo, float x) {
    uint32_t off = (uint32_t)(r >> 3) * sbo + (uint32_t)(c >> 2) * lbo + (uint32_t)(r & 7) * 16u + (uint32_t)(c & 3) * 4u;
    float h = tf32_hi(x);
    *reinterpret_cast<float*>(hi + off) = h;
    if (with_lo) *reinterpret_cast<float*>(lo + off) = x - h;
  };
  // modes 6 / 7 (+16*variant): the B operand of the G2 / G3 form MN-major (N contiguous) in the SWIZZLE_128B_BASE32B
  // layout: rows of 128 bytes (32 N-elements) per K index, the four 32-byte chunks of a row XOR-ed with (K index & 3)
  const int variant = mode >> 4;
  mode &= 15;
  unsigned char* pb_hi = smem;                 // probe buffers (the Hb region is unused in these modes)
  unsigned char* pb_lo = smem + 16384;
  if (mode == 6 || mode == 7) {
    const int acols = (mode == 6) ? TN : BM;
    const uint32_t th = (mode == 6) ? TM_DZH : TM_HTH, tl = (mode == 6) ? TM_DZL : TM_HTL;
    for (int c = cpart; c < acols / CW; c += NT / 128) {
      float hi[CW], lo[CW];
#pragma unroll
      for (int j = 0; j < CW; ++j) {
        float x = A[(size_t)row * acols + c * CW + j];
        hi[j] = tf32_hi(x);
        lo[j] = x - hi[j];
      }
      tmem_st8(lane_addr + th + c * CW, hi);
      if (with_lo) tmem_st8(lane_addr + tl + c * CW, lo);
    }
    tmem_st_wait();
    const int nN = (mode == 6) ? g.Np : TN, nK = (mode == 6) ? TN : BM;
    for (int q = tid; q < nN * nK; q += NT) {
      const int n = q / nK, kk = q % nK;
      const int blk = n >> 5, nn = n & 31;
      const int sw = (variant == 2) ? 0 : (kk & 3);
      const uint32_t off = (uint32_t)blk * 4096u + (uint32_t)kk * 128u + (uint32_t)(((nn >> 3) ^ sw) * 32) + (uint32_t)(nn & 7) * 4u;
      const float x = Bm[q], h = tf32_hi(x);
      *reinterpret_cast<float*>(pb_hi + off) = h;
      if (with_lo) *reinterpret_cast<float*>(pb_lo + off) = x - h;
    }
  } else if (mode == 1) {
    for (int q = tid; q < BM * g.Kp; q += NT) split_store(hb_hi, hb_lo, q / g.Kp, q % g.Kp, CORE, g.hb_sbo, A[q]);
    for (int q = tid; q < TN * g.Kp; q += NT) split_store(wb_hi, wb_lo, q / g.Kp, q % g.Kp, CORE, g.wb_sbo, Bm[q]);
  } else {
    const int acols = (mode == 2) ? TN : BM;
    const uint32_t th = (mode == 2) ? TM_DZH : TM_HTH, tl = (mode == 2) ? TM_DZL : TM_HTL;
    for (int c = cpart; c < acols / CW; c += NT / 128) {
      float hi[CW], lo[CW];
#pragma unroll
      for (int j = 0; j < CW; ++j) {
        float x = A[(size_t)row * acols + c * CW + j];
        hi[j] = tf32_hi(x);
        lo[j] = x - hi[j];
      }
      tmem_st8(lane_addr + th + c * CW, hi);
      if (with_lo) tmem_st8(lane_addr + tl + c * CW, lo);
    }
    tmem_st_wait();
    if (mode == 2)
      for (int q = tid; q < g.Np * TN; q += NT) split_store(wt_hi, wt_lo, q / TN, q % TN, g.wt_lbo, g.wt_sbo, Bm[q]);
    else
      for (int q = tid; q < TN * BM; q += NT) split_store(dt_hi, dt_lo, q / BM, q % BM, g.dt_lbo, g.dt_sbo, Bm[q]);
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    const SmemOp o_hb = make_op(hb_hi, hb_lo, CORE, g.hb_sbo, 2 * CORE), o_wb = make_op(wb_hi, wb_lo, CORE, g.wb_sbo, 2 * CORE);
    const SmemOp o_wt = make_op(wt_hi, wt_lo, g.wt_lbo, g.wt_sbo, 2 * g.wt_lbo);
    const SmemOp o_dt = make_op(dt_hi, dt_lo, g.dt_lbo, g.dt_sbo, 2 * g.dt_lbo);
    const bool leader = elect_one();
    if (leader && (mode == 6 || mode == 7)) {
      uint32_t lbo = 4096u, sbo = 512u;
      if (variant == 1) { lbo = 512u; sbo = 4096u; }
      if (variant == 3) sbo = 1024u;
      SmemOp o;
      o.hi = make_desc_sw(smem_u32(pb_hi), lbo, sbo, 1u);
      o.lo = make_desc_sw(smem_u32(pb_lo), lbo, sbo, 1u);
      o.step16 = 1024u >> 4;                       // 8 K rows of 128 bytes per k-step
      if (mode == 6) {
        if (split == 3) issue_gemm_ts<3>(tmem + TM_DH, tmem + TM_DZH, tmem + TM_DZL, o, TN / 8, make_idesc(BM, g.Np, 0, 1), 0u);
        else issue_gemm_ts<1>(tmem + TM_DH, tmem + TM_DZH, tmem + TM_DZL, o, TN / 8, make_idesc(BM, g.Np, 0, 1), 0u);
      } else {
        if (split == 3) issue_gemm_ts<3>(tmem + TM_DW, tmem + TM_HTH, tmem + TM_HTL, o, BM / 8, make_idesc(BM, TN, 0, 1), 0u);
        else issue_gemm_ts<1>(tmem + TM_DW, tmem + TM_HTH, tmem + TM_HTL, o, BM / 8, make_idesc(BM, TN, 0, 1), 0u);
      }
      mma_commit(&bar_mma);
    } else if (leader) {
      if (split == 3) {
        if (mode == 1) issue_gemm<3>(tmem + TM_Z, o_hb, o_wb, g.Kp / 8, make_idesc(BM, TN, 0, 0), 0u);
        else if (mode == 2) issue_gemm_ts<3>(tmem + TM_DH, tmem + TM_DZH, tmem + TM_DZL, o_wt, TN / 8, make_idesc(BM, g.Np, 0, 0), 0u);
        else issue_gemm_ts<3>(tmem + TM_DW, tmem + TM_HTH, tmem + TM_HTL, o_dt, BM / 8, make_idesc(BM, TN, 0, 0), 0u);
      } else {
        if (mode == 1) issue_gemm<1>(tmem + TM_Z, o_hb, o_wb, g.Kp / 8, make_idesc(BM, TN, 0, 0), 0u);
        else if (mode == 2) issue_gemm_ts<1>(tmem + TM_DH, tmem + TM_DZH, tmem + TM_DZL, o_wt, TN / 8, make_idesc(BM, g.Np, 0, 0), 0u);
        else issue_gemm_ts<1>(tmem + TM_DW, tmem + TM_HTH, tmem + TM_HTL, o_dt, BM / 8, make_idesc(BM, TN, 0, 0), 0u);
      }
      mma_commit(&bar_mma);
    }
    __syncwarp();
  }
  mbar_wait_backoff(&bar_mma, 0);
  tc_fence_after();
  const int ncols = (mode == 2 || mode == 6) ? g.Np : TN;
  const uint32_t tsrc = (mode == 1) ? TM_Z : ((mode == 2 || mode == 6) ? TM_DH : TM_DW);
  for (int c = cpart; c < ncols / CW; c += NT / 128) {
    float d[CW];
    tmem_ld8(lane_addr + tsrc + c * CW, d);
#pragma unroll
    for (int j = 0; j < CW; ++j) D[(size_t)row * ncols + c * CW + j] = d[j];
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, TMEM_COLS);
}

}  // namespace tc

// smem of the pipelined kernel: Hb hi/lo (round8(B) rows) + Wb hi/lo + Wtb hi/lo + Dtb hi/lo + E2 stage
static size_t tc2_smem_bytes(const tc::Geom& g, int B) {
  size_t hb_eff = (size_t)(((B + 7) & ~7) / 8) * g.hb_sbo;
  size_t n = 2 * hb_eff + 2 * (size_t)g.wb_bytes + 2 * (size_t)g.wt_bytes + 2 * (size_t)g.dt_bytes +
             3 * (size_t)tc::TN * g.H * 4 + 3 * tc::TN * 4;
  // the M = 128 operand view of Hb reaches 16 row groups from the start of its lo half
  size_t reach = hb_eff + 16 * (size_t)g.hb_sbo;
  return std::max(n, reach);
}
// Envelope of the pipelined kernel: TMEM budget, shared-memory budget, bias lanes inside one warp.
static bool tc2_supported(int B, int H) {
  tc::Geom g = tc::make_geom(H);
  int BK = (B + 7) & ~7;
  if (B > tc::BM || g.Np + 2 * BK > 320) return false;
  if ((H & 31) + 1 + TC2_CW > 32) return false;   // bias lanes H+1..H+CW live in the warp of lane H
  return tc2_smem_bytes(g, B) <= 227 * 1024 - 256;
}

// largest row chunk the pipelined kernel takes for this n_hidden (multiple of 8; 0: shape outside its envelope)
int tc2_max_rows(int H) {
  if ((H & 3) != 0 || H + 1 > 128) return 0;
  for (int b = tc::BM; b >= 8; b -= 8)
    if (tc2_supported(b, H)) return b;
  return 0;
}

template <int MODE>
static int launch_tc2(const float* h2, int B, int H, float* Wd3, float* bd3, float* mW, float* vW, float* mb, float* vb,
                      int v_begin, int Vloc, const int32_t* indptr, const int32_t* indices, double n_total,
                      const aae_step_state* st, float* dh2, double* loss_sum, int split, float* gW, float* gB,
                      cudaStream_t s) {
  tc::Geom g = tc::make_geom(H);
  int n_tiles = (Vloc + tc::TN - 1) / tc::TN;
  int grid = std::min(n_tiles, sm_count());
  size_t smem = tc2_smem_bytes(g, B);
  void (*kern)(const float*, int, int, float*, float*, float*, float*, float*, float*, int, int, const int32_t*,
               const int32_t*, float, const aae_step_state*, float*, double*, int, float*, float*);
  if (MODE == 0 && split != 3)
    kern = (H == 100) ? tc::dec_out_train_tc2_kernel<1, 100, TC2_CW, 0> : tc::dec_out_train_tc2_kernel<1, 0, TC2_CW, 0>;
  else
    kern = (H == 100) ? tc::dec_out_train_tc2_kernel<3, 100, TC2_CW, MODE> : tc::dec_out_train_tc2_kernel<3, 0, TC2_CW, MODE>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) {
    set_error("dec_out_train(tc2): smem %zu: %s", smem, cudaGetErrorString(e));
    return AAE_E_CUDA;
  }
  kern<<<grid, tc::Tc2Cfg<TC2_CW>::NTHR, smem, s>>>(h2, B, H, Wd3, bd3, mW, vW, mb, vb, v_begin, Vloc, indptr, indices,
                                                   (float)(1.0 / n_total), st, dh2, loss_sum, (int)smem, gW, gB);
  return check_launch("dec_out_train(tc2)");
}

int dec_out_train_tc(const float* h2, int B, int H, float* Wd3, float* bd3, float* mW, float* vW, float* mb, float* vb,
                     int v_begin, int Vloc, const int32_t* indptr, const int32_t* indices, double n_total,
                     const aae_step_state* st, float* dh2, double* loss_sum, int split, bool pipelined,
                     float* gwork, cudaStream_t s) {
  if (!tc_supported(B, H, "dec_out_train")) return AAE_E_UNSUPPORTED;
  tc::Geom g = tc::make_geom(H);
  int n_tiles = (Vloc + tc::TN - 1) / tc::TN;
  int grid = std::min(n_tiles, sm_count());
  const bool aligned16 = ((reinterpret_cast<uintptr_t>(Wd3) | reinterpret_cast<uintptr_t>(mW) |
                           reinterpret_cast<uintptr_t>(vW) | reinterpret_cast<uintptr_t>(bd3) |
                           reinterpret_cast<uintptr_t>(mb) | reinterpret_cast<uintptr_t>(vb)) & 15) == 0;   // TMA bulk copies
  if (pipelined && aligned16 && tc2_supported(B, H))
    return launch_tc2<0>(h2, B, H, Wd3, bd3, mW, vW, mb, vb, v_begin, Vloc, indptr, indices, n_total, st, dh2, loss_sum,
                         split, nullptr, nullptr, s);
  const int rows = (pipelined && aligned16) ? tc2_max_rows(H) : 0;
  if (B > tc::BM || (rows > 0 && B > rows && gwork && split == 3)) {
    // Batches beyond one row chunk (the reference's scripts use 500, 1000, 10000: main.py:76, mpd.py:75-76,
    // aminer.py:62): one launch of the pipelined kernel per chunk of <= `rows` rows with the W' tile walk unchanged;
    // the chunks' weight gradients are summed in `gwork` ([Vloc,H] + [Vloc] floats) and the last chunk applies Adam
    // once with the total, exactly as the reference's single backward over the whole batch does.
    if (!(pipelined && aligned16 && rows > 0 && gwork && split == 3)) {
      set_error("dec_out_train: batch %d needs the chunked tensor-core path (3xTF32, gradient scratch, 16-byte aligned "
                "tensors, n_hidden inside the pipelined kernel's envelope); use impl=simt", B);
      return AAE_E_UNSUPPORTED;
    }
    const int n_chunks = (B + rows - 1) / rows;
    int per = (B + n_chunks - 1) / n_chunks;
    per = std::min(rows, (per + 7) & ~7);
    float* gW = gwork;
    float* gB = gwork + (size_t)Vloc * H;
    for (int c = 0, b0 = 0; b0 < B; ++c, b0 += per) {
      const int nb = std::min(per, B - b0);
      const bool first = (b0 == 0), last = (b0 + nb >= B);
      int rc;
#define TC2_CHUNK(M)                                                                                                    \
  launch_tc2<M>(h2 + (size_t)b0 * H, nb, H, Wd3, bd3, mW, vW, mb, vb, v_begin, Vloc, indptr + b0, indices, n_total, st, \
                dh2 + (size_t)b0 * H, loss_sum, 3, gW, gB, s)
      if (first) rc = TC2_CHUNK(1);
      else if (last) rc = TC2_CHUNK(3);
      else rc = TC2_CHUNK(2);
#undef TC2_CHUNK
      if (rc) return rc;
    }
    return AAE_OK;
  }
  size_t smem = tc::smem_bytes(g);
  auto kern = (split == 3) ? tc::dec_out_train_tc_kernel<3> : tc::dec_out_train_tc_kernel<1>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) {
    set_error("dec_out_train(tc): smem %zu: %s", smem, cudaGetErrorString(e));
    return AAE_E_CUDA;
  }
  kern<<<grid, tc::NT, smem, s>>>(h2, B, H, Wd3, bd3, mW, vW, mb, vb, v_begin, Vloc, indptr, indices,
                                  (float)(1.0 / n_total), st, dh2, loss_sum);
  return check_launch("dec_out_train(tc)");
}
}  // namespace aae

extern "C" int aae_tc_selftest(int mode, const float* A, const float* Bm, float* D, int split, void* stream) {
  using namespace aae;
  tc::Geom g = tc::make_geom(100);
  size_t smem = tc::smem_bytes(g);
  cudaError_t e = cudaFuncSetAttribute(tc::tc_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) {
    set_error("tc_selftest: %s", cudaGetErrorString(e));
    return AAE_E_CUDA;
  }
  tc::tc_selftest_kernel<<<1, tc::NT, smem, as_stream(stream)>>>(mode, A, Bm, D, split);
  return check_launch("tc_selftest");
}

#ifdef K3X_TRACE
extern "C" int aae_k3x_trace_read(long long* out) {
  return (int)cudaMemcpyFromSymbol(out, aae::tc::k3x_tr, sizeof(long long) * 32 * 16);
}
#endif
