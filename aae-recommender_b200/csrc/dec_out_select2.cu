// K5 v2: predict's candidate filter fed by TMA, W' tiles multicast across a thread-block cluster.
//
// The first K5 (dec_out_select.cu, dec_out_select_kernel) ran every logit through the fp32-accurate 3xTF32 split and fed
// the tensor core from register-staged loads: each of the row-chunk CTAs that walk the same W' tile fetched it from
// L2 and converted it to operand layout by itself, and the kernel was bound by that loader, not by the MMAs
// (single-pass TF32 was no faster).  An exact top-k does not need exact logits for all B x V pairs -- only for the
// ~1.4 k candidates per row that survive a threshold:
//   * this kernel computes single-pass TF32 logits (kind::tf32 reads the upper 19 bits of the fp32 container, so the
//     RAW fp32 tile is the operand: no conversion pass at all) and keeps items whose logit exceeds tau_b - margin_b,
//     margin_b a rigorous bound of the TF32 error of row b (topk.cu);
//   * the survivors are re-scored exactly in fp32 and ranked (topk.cu), and a row whose k-th exact score does not
//     clear tau_b is reported in n_bad (the caller falls back to the exact dense path): the result is exact.
// Feed: W' = [Wd3 | bd3 | 0] is kept as a padded [Vloc, 104] fp32 matrix (aae_pad_weights; 416-byte rows) described by
// two 2-D tensor maps (three boxes of 32 floats x 128/CY rows, SWIZZLE_128B, for k = 0..95 and one box of 8 floats,
// SWIZZLE_32B, for k = 96..103: a 52 KB stage holds K = 104 exactly, so four stages fit).  A
// cluster of CY CTAs (CY row chunks of 128 query rows) shares every tile: CTA r loads rows [r*128/CY, (r+1)*128/CY) of
// each of the 4 K-boxes and MULTICASTS them into the same stage of all CY CTAs (cp.async.bulk.tensor ...
// .multicast::cluster), so a tile crosses L2 -> SM once per cluster instead of once per CTA.  Stage hand-over: full[s]
// (transaction bytes of the whole tile) and empty[s] (one tcgen05.commit.multicast arrival from each CTA of the
// cluster: every consumer is done with the stage).
// Roles per CTA: warps 0-15 epilogue (TMEM lane quarter = warp % 4, 32-column part = warp / 4), warp 16 MMA issuer,
// warp 17 TMA producer.  TMEM: accumulators 2 x 128 columns | A operand (H2' chunk, tf32, lane = query row) 104.
//
// Replaces the dense lin3 of predict (aae.py:866-868) and the front half of remove_non_missing + argtopk
// (evaluation.py:183-199, 20-58), like the first K5.
#include <cuda.h>
#include <cooperative_groups.h>
#include <algorithm>
#include <map>
#include <mutex>
#include <tuple>
#include "tcgen05.cuh"
#include "dec_out.cuh"

namespace aae {
namespace s2 {
namespace cg = cooperative_groups;

constexpr int BM = 128;                 // query rows per chunk (MMA M)
constexpr int PN = 128;                 // items per tile (MMA N)
constexpr int KP = 104;                 // padded K of W' rows (n_hidden 100 + bias + 3 zeros): 13 MMA K-steps
constexpr int KBOX = 32;                // floats per row of a big TMA box (128 bytes: one SWIZZLE_128B atom row)
constexpr int NBOX = 3;                 // big K boxes per tile (k = 0..95)
constexpr int KTAIL = KP - NBOX * KBOX; // 8 floats (k = 96..103): one SWIZZLE_32B box, exactly one MMA K-step
constexpr int BOX_BYTES = PN * KBOX * 4;               // 16 KB
constexpr int TAIL_BYTES = PN * KTAIL * 4;             // 4 KB
constexpr int STAGE_BYTES = NBOX * BOX_BYTES + TAIL_BYTES;   // 52 KB: K = 104 exactly, no zero-filled padding in smem
constexpr int NSTAGE = 4;
constexpr int NWE = 16;                 // epilogue warps
constexpr int NT = 32 * (NWE + 2);      // + MMA warp + TMA warp
constexpr int CW = PN / 4;              // accumulator columns per epilogue thread
constexpr uint32_t T_ACC = 0, T_A = 256, TMEM_COLS = 512;

struct Sel2Args {
  const float* h2; int B, H;
  int Vloc, v_begin;
  int tile_stride, n_sel;              // tiles visited: j * tile_stride, j < n_sel
  int filter;                          // 0: dense approximate scores (threshold sample), 1: threshold filter
  float* out; long long ldo; int out_by_visit;
  const float* tau; int32_t* cnt; int32_t* cand_idx; int cap_sub;
};

template <int CY>
__global__ void __launch_bounds__(NT, 1) dec_out_select2_kernel(const __grid_constant__ CUtensorMap wmap,
                                                                const __grid_constant__ CUtensorMap wmap_tail,
                                                                Sel2Args a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // SWIZZLE_128B needs 1024-byte aligned stages: align the dynamic window by hand (the launcher adds the slack)
  unsigned char* stages = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t bar_full[NSTAGE], bar_empty[NSTAGE], bar_acc_full[2], bar_acc_empty[2];
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rank = (CY > 1) ? (int)(blockIdx.y % CY) : 0;          // cluster dims (1, CY, 1)
  constexpr uint16_t kMask = (uint16_t)((1u << CY) - 1u);
  const int n_chunks = (a.B + BM - 1) / BM;
  const int n_groups = (n_chunks + CY - 1) / CY;
  const int groups_per_pass = (int)gridDim.y / CY;
  const int n_my = ((int)blockIdx.x < a.n_sel) ? (a.n_sel - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  // Cluster rows that work on different row-chunk groups at the same time walk the tiles in rotated order: the same
  // W' lines requested by 16 clusters in the same microsecond serialise on their L2 slices (measured: 1.37 us per tile
  // against 0.88 us when the clusters read different tiles); HBM has the bandwidth to stream W' once per cluster row.
  const int rot = (groups_per_pass > 1 && n_my > 0) ? (int)(((long long)((int)blockIdx.y / CY) * n_my) / groups_per_pass) : 0;

  if (warp == NWE) tmem_alloc(&tmem_base_s, TMEM_COLS);
  if (tid == 0) {
    for (int s = 0; s < NSTAGE; ++s) {
      mbar_init(&bar_full[s], 1);
      mbar_init(&bar_empty[s], CY);              // one tcgen05.commit arrival from every CTA of the cluster
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&bar_acc_full[b], 1);
      mbar_init(&bar_acc_empty[b], NWE);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&wmap) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&wmap_tail) : "memory");
  }
  tc_fence_before();
  __syncthreads();
  if (CY > 1) cg::this_cluster().sync();         // every CTA's barriers exist before a peer multicasts into them
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const uint32_t idesc = make_idesc(BM, PN);
  // pipeline positions (continue across chunk groups)
  uint32_t it_p = 0, it_m = 0, it_e = 0;          // tiles produced / issued / drained so far

  for (int grp = (int)blockIdx.y / CY; grp < n_groups; grp += groups_per_pass) {
    const int chunk = grp * CY + rank;
    const int b0 = chunk * BM;
    const int nb = max(0, min(BM, a.B - b0));      // 0: an idle CTA padding the cluster (it still feeds and drains)
    __syncthreads();                               // the previous group's accumulators are drained: A may be rebuilt
    if (warp < NWE) {
      // H2' chunk -> TMEM (A operand: lane = query row, column = k), truncated to tf32 like the raw B operand
      const int q4 = warp & 3, cpart = warp >> 2;
      const uint32_t lane_addr = tmem + ((uint32_t)(q4 * 32) << 16);
      const int brow = q4 * 32 + lane;
      for (int c = cpart; c < KP / 8; c += 4) {
        float hi[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int kk = c * 8 + j;
          float x = 0.f;
          if (brow < nb) x = (kk < a.H) ? __ldg(a.h2 + (size_t)(b0 + brow) * a.H + kk) : (kk == a.H ? 1.0f : 0.f);
          hi[j] = tf32_hi(x);
        }
        tmem_st8(lane_addr + T_A + c * 8, hi);
      }
      tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    if (warp == NWE + 1) {
      // ================= TMA producer =================
      if (elect_one()) {
        for (int i = 0; i < n_my; ++i, ++it_p) {
          const int s = (int)(it_p % NSTAGE);
          const uint32_t use = it_p / NSTAGE;
          mbar_wait_spin(&bar_empty[s], (use & 1u) ^ 1u);          // every CTA of the cluster has released the stage
          mbar_arrive_expect_tx(&bar_full[s], STAGE_BYTES);   // the whole tile lands here (all slices, all senders)
          int j = i + rot;
          if (j >= n_my) j -= n_my;
          const int row0 = ((int)blockIdx.x + j * (int)gridDim.x) * a.tile_stride * PN + rank * (PN / CY);
          unsigned char* dst = stages + (size_t)s * STAGE_BYTES + (size_t)rank * (PN / CY) * (KBOX * 4);
#pragma unroll
          for (int j = 0; j < NBOX; ++j) {
            if (CY > 1) tma_load_mc(dst + j * BOX_BYTES, &wmap, j * KBOX, row0, &bar_full[s], kMask);
            else tma_load(dst + j * BOX_BYTES, &wmap, j * KBOX, row0, &bar_full[s]);
          }
          unsigned char* dst_t = stages + (size_t)s * STAGE_BYTES + NBOX * BOX_BYTES + (size_t)rank * (PN / CY) * (KTAIL * 4);
          if (CY > 1) tma_load_mc(dst_t, &wmap_tail, NBOX * KBOX, row0, &bar_full[s], kMask);
          else tma_load(dst_t, &wmap_tail, NBOX * KBOX, row0, &bar_full[s]);
        }
      }
      __syncwarp();
    } else if (warp == NWE) {
      // ================= MMA issuer =================
      for (int i = 0; i < n_my; ++i, ++it_m) {
        const int s = (int)(it_m % NSTAGE), acc = (int)(it_m & 1u);
        mbar_wait_spin(&bar_full[s], (it_m / NSTAGE) & 1u);
        mbar_wait_spin(&bar_acc_empty[acc], ((it_m >> 1) & 1u) ^ 1u);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sbase = smem_u32(stages + (size_t)s * STAGE_BYTES);
#pragma unroll
          for (int kk = 0; kk < KP / 8; ++kk) {
            const uint64_t bdesc = (kk < NBOX * 4)
                ? make_desc_sw128(sbase + (uint32_t)(kk >> 2) * BOX_BYTES + (uint32_t)(kk & 3) * 32u)
                : make_desc_sw32(sbase + (uint32_t)NBOX * BOX_BYTES);
            mma_tf32_ts(tmem + T_ACC + (uint32_t)(acc * PN), tmem + T_A + 8 * kk, bdesc, idesc, kk ? 1u : 0u);
          }
          mma_commit(&bar_acc_full[acc]);
          if (CY > 1) mma_commit_mc(&bar_empty[s], kMask);
          else mma_commit(&bar_empty[s]);
        }
        __syncwarp();
      }
    } else {
      // ================= epilogue =================
      const int q4 = warp & 3, cpart = warp >> 2;
      const uint32_t lane_addr = tmem + ((uint32_t)(q4 * 32) << 16);
      const int brow = q4 * 32 + lane;
      const bool rowv = brow < nb;
      float tau = __int_as_float(0x7f800000);
      if (a.filter && rowv) tau = a.tau[b0 + brow];
      const int nsub = (int)gridDim.x * 4, sub = (int)blockIdx.x * 4 + cpart;
      const size_t sub_base = ((size_t)(b0 + brow) * nsub + sub) * (size_t)a.cap_sub;
      int my_cnt = 0;
      const int c0 = cpart * CW;
      for (int i = 0; i < n_my; ++i, ++it_e) {
        const int acc = (int)(it_e & 1u);
        int jt = i + rot;
        if (jt >= n_my) jt -= n_my;
        const int v0 = ((int)blockIdx.x + jt * (int)gridDim.x) * a.tile_stride * PN;
        mbar_wait_spin(&bar_acc_full[acc], (it_e >> 1) & 1u);
        tc_fence_after();
        uint32_t zr[CW];
        TmemIO<16>::ld_issue(lane_addr + T_ACC + (uint32_t)(acc * PN + c0), zr);
        TmemIO<16>::ld_issue(lane_addr + T_ACC + (uint32_t)(acc * PN + c0 + 16), zr + 16);
        tmem_ld_wait32(zr);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_acc_empty[acc]);       // this warp's quarter x part is in registers
        const int vm = a.Vloc - v0 - c0;                         // valid columns among this thread's 32
        if (a.filter) {
          float zmax = __uint_as_float(zr[0]);
#pragma unroll
          for (int j = 1; j < CW; ++j) zmax = fmaxf(zmax, __uint_as_float(zr[j]));
          if (zmax > tau) {
#pragma unroll
            for (int j = 0; j < CW; ++j) {
              if (__uint_as_float(zr[j]) > tau && j < vm) {
                if (my_cnt < a.cap_sub) a.cand_idx[sub_base + my_cnt] = a.v_begin + v0 + c0 + j;
                ++my_cnt;
              }
            }
          }
        } else if (rowv) {
          const int colbase = a.out_by_visit ? ((int)blockIdx.x + jt * (int)gridDim.x) * PN : v0;
          float* orow = a.out + (size_t)(b0 + brow) * a.ldo + colbase + c0;
          if (vm >= CW && ((reinterpret_cast<uintptr_t>(orow) & 15) == 0)) {
#pragma unroll
            for (int j = 0; j < CW; j += 4)
              __stcs(reinterpret_cast<float4*>(orow + j),
                     make_float4(__uint_as_float(zr[j]), __uint_as_float(zr[j + 1]), __uint_as_float(zr[j + 2]),
                                 __uint_as_float(zr[j + 3])));
          } else {
#pragma unroll
            for (int j = 0; j < CW; ++j)
              if (j < vm) orow[j] = __uint_as_float(zr[j]);
          }
        }
      }
      if (a.filter && rowv) a.cnt[(size_t)(b0 + brow) * nsub + sub] = my_cnt;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CY > 1) cg::this_cluster().sync();         // no CTA leaves while a peer may still multicast into its stages
  if (warp == NWE) tmem_dealloc(tmem, TMEM_COLS);
}

// W' = [Wd3 | bd3 | 0 0 0] as a padded [Vloc, KP] matrix + the largest row norm (for the TF32 error bound)
__global__ void __launch_bounds__(256) pad_weights_kernel(const float* __restrict__ Wd3, const float* __restrict__ bd3,
                                                          int Vloc, int H, float* __restrict__ Wp,
                                                          float* __restrict__ wmax) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  float best = 0.f;
  for (int v = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < Vloc; v += warps) {
    float ss = 0.f;
    for (int k = lane; k < KP; k += 32) {
      const float x = (k < H) ? Wd3[(size_t)v * H + k] : (k == H ? bd3[v] : 0.f);
      Wp[(size_t)v * KP + k] = x;
      ss = fmaf(x, x, ss);
    }
    ss = warp_sum(ss);
    best = fmaxf(best, ss);
  }
  if (lane == 0 && best > 0.f) atomicMax(reinterpret_cast<int*>(wmax), __float_as_int(sqrtf(best) * 1.000001f));
}

}  // namespace s2

// ---- host side ---------------------------------------------------------------------------------------------------
static std::mutex g_map_mutex;
static std::map<std::tuple<const void*, int, int>, CUtensorMap> g_maps;

static int get_tensor_map(const float* Wp, int Vloc, int cy, bool tail, CUtensorMap* out) {
  std::lock_guard<std::mutex> lock(g_map_mutex);
  auto key = std::make_tuple((const void*)Wp, Vloc, tail ? -cy : cy);
  auto it = g_maps.find(key);
  if (it != g_maps.end()) { *out = it->second; return AAE_OK; }
  CUtensorMap m;
  const cuuint64_t gdim[2] = {(cuuint64_t)s2::KP, (cuuint64_t)Vloc};
  const cuuint64_t gstride[1] = {(cuuint64_t)s2::KP * sizeof(float)};
  const cuuint32_t box[2] = {(cuuint32_t)(tail ? s2::KTAIL : s2::KBOX), (cuuint32_t)(s2::PN / cy)};
  const cuuint32_t estr[2] = {1, 1};
  // The driver entry point is looked up through the runtime (cudaGetDriverEntryPoint), so the library has no link-time
  // dependency on libcuda.so.1 and still loads on a machine without a driver (CPU-side ABI tests, the build check).
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t ce = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (ce != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
      set_error("cuTensorMapEncodeTiled is not available from this driver (%s)", cudaGetErrorString(ce));
      cudaGetLastError();
      return AAE_E_CUDA;
    }
    encode = reinterpret_cast<EncodeFn>(fn);
  }
  CUresult r = encode(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(Wp), gdim, gstride, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, tail ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
    return AAE_E_CUDA;
  }
  if (g_maps.size() > 64) g_maps.clear();
  g_maps[key] = m;
  *out = m;
  return AAE_OK;
}

static int pick_cy(int B) {
  const int n_chunks = (B + s2::BM - 1) / s2::BM;
  // clusters of 4: measured at V=2M -- B=1000: 1.79 / 1.43 / 1.38 / 1.38 ms and B=4000: 6.76 / 5.65 / 5.23 / 5.92 ms for
  // cluster sizes 1 / 2 / 4 / 8 (clusters of 8 leave 28 of the 148 SMs without work: 15 clusters fit)
  int cy = 1;
  while (cy < 4 && cy * 2 <= n_chunks) cy *= 2;
  const char* e = getenv("AAE_B200_K5_CLUSTER");
  if (e) cy = std::max(1, std::min(8, atoi(e)));
  return cy;
}

template <int CY>
static int grid_for(int B, int n_sel, int* gx, int* gy) {
  const int n_chunks = (B + s2::BM - 1) / s2::BM;
  const int n_groups = (n_chunks + CY - 1) / CY;
  const size_t smem = (size_t)s2::NSTAGE * s2::STAGE_BYTES + 1024;
  auto kern = s2::dec_out_select2_kernel<CY>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) { set_error("dec_out_select2: smem %zu: %s", smem, cudaGetErrorString(e)); return AAE_E_CUDA; }
  int max_clusters = sm_count() / CY;
  if (CY > 1) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(1, CY, 1);
    cfg.blockDim = dim3(s2::NT, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 1; attr[0].val.clusterDim.y = CY; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) == cudaSuccess && n > 0) max_clusters = n;
    else cudaGetLastError();
  }
  const int gyc = std::max(1, std::min(n_groups, max_clusters));              // cluster rows
  *gy = gyc * CY;
  *gx = std::max(1, std::min(n_sel, max_clusters / gyc));
  return AAE_OK;
}

void dec_out_select2_grid(int B, int n_sel, int* gx, int* gy) {
  switch (pick_cy(B)) {
    case 8: grid_for<8>(B, n_sel, gx, gy); break;
    case 4: grid_for<4>(B, n_sel, gx, gy); break;
    case 2: grid_for<2>(B, n_sel, gx, gy); break;
    default: grid_for<1>(B, n_sel, gx, gy); break;
  }
}

template <int CY>
static int launch_select2(const CUtensorMap& map, const CUtensorMap& map_tail, const s2::Sel2Args& a, cudaStream_t s) {
  int gx = 1, gy = 1;
  int rc = grid_for<CY>(a.B, a.n_sel, &gx, &gy);
  if (rc) return rc;
  const size_t smem = (size_t)s2::NSTAGE * s2::STAGE_BYTES + 1024;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(gx, gy, 1);
  cfg.blockDim = dim3(s2::NT, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1; attr[0].val.clusterDim.y = CY; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, s2::dec_out_select2_kernel<CY>, map, map_tail, a);
  if (e != cudaSuccess) { set_error("dec_out_select2<%d>: %s", CY, cudaGetErrorString(e)); return AAE_E_CUDA; }
  return check_launch("dec_out_select2");
}

// K5 v2 launcher: approximate (single-pass TF32) dense scores of the visited tiles (filter == 0) or the threshold filter.
int dec_out_select2(const float* h2, int B, int H, const float* Wp, int Vloc, int v_begin, int tile_stride, int n_sel,
                    int filter, float* out, int64_t ldo, int out_by_visit, const float* tau, int32_t* cnt,
                    int32_t* cand_idx, int cap_sub, cudaStream_t s) {
  if (H + 1 > s2::KP) { set_error("dec_out_select2: n_hidden %d > %d", H, s2::KP - 1); return AAE_E_UNSUPPORTED; }
  const int cy = pick_cy(B);
  CUtensorMap map, map_tail;
  int rc = get_tensor_map(Wp, Vloc, cy, false, &map);
  if (rc) return rc;
  rc = get_tensor_map(Wp, Vloc, cy, true, &map_tail);
  if (rc) return rc;
  s2::Sel2Args a;
  a.h2 = h2; a.B = B; a.H = H; a.Vloc = Vloc; a.v_begin = v_begin; a.tile_stride = tile_stride; a.n_sel = n_sel;
  a.filter = filter; a.out = out; a.ldo = ldo; a.out_by_visit = out_by_visit; a.tau = tau; a.cnt = cnt;
  a.cand_idx = cand_idx; a.cap_sub = cap_sub;
  switch (cy) {
    case 8: return launch_select2<8>(map, map_tail, a, s);
    case 4: return launch_select2<4>(map, map_tail, a, s);
    case 2: return launch_select2<2>(map, map_tail, a, s);
    default: return launch_select2<1>(map, map_tail, a, s);
  }
}

bool select2_supported(int H) { return H + 1 <= s2::KP && (H & 3) == 0; }

}  // namespace aae

using namespace aae;

extern "C" {

int64_t aae_pad_weights_floats(int Vloc, int H) {
  if (Vloc <= 0 || !select2_supported(H)) return 0;
  return (int64_t)Vloc * s2::KP + 64;       // + the row-norm maximum (one float, kept 256-byte aligned behind the matrix)
}

int aae_pad_weights(const float* Wd3, const float* bd3, int Vloc, int H, float* Wp, float* wmax, void* stream) {
  AAE_REQUIRE(Wd3 && bd3 && Wp && wmax, "null pointer");
  AAE_REQUIRE(Vloc > 0 && select2_supported(H), "shape outside the TMA-fed filter's envelope");
  AAE_REQUIRE((reinterpret_cast<uintptr_t>(Wp) & 15) == 0, "Wp must be 16-byte aligned");
  cudaStream_t s = as_stream(stream);
  cudaMemsetAsync(wmax, 0, sizeof(float), s);
  s2::pad_weights_kernel<<<std::min(8 * sm_count(), std::max(1, cdiv((int64_t)Vloc * 32, 256))), 256, 0, s>>>(
      Wd3, bd3, Vloc, H, Wp, wmax);
  return check_launch("pad_weights");
}

}  // extern "C"
