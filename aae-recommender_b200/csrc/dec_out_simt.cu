// K3 (fp32 CUDA-core variant) -- the n_items-wide decoder output layer.
// Training: logits, sigmoid, BCE, dZ, dh2 += dZ.W, dW = dZ^T.h2 and Adam on W/bias in ONE pass over
// Wd3 (the [B,V] logit matrix never exists in HBM).  Prediction: scores (logits or probabilities).
// This is the exact-fp32 correctness baseline and the path for shapes outside the tensor-core
// kernels' envelope; the tcgen05 kernels in dec_out_tc.cu (training) and dec_out_select.cu (scores) are the fast path.
// Reference: aaerec/aae.py:176-177 (lin3 + sigmoid), :693-695 (BCE), :703 (backward), :707 (dec_optim).
#include "dec_out.cuh"

namespace aae {

constexpr int TN = 32;         // items per tile
constexpr int DT = 256;        // threads
constexpr int ZLD = TN + 4;    // row pitch of the dZ tile (16-byte aligned rows)

__host__ __device__ inline int pad_ld(int H) {  // multiple of 4 with (ld/4) odd -> conflict-free float4 rows
  int ld = (H + 3) & ~3;
  if (((ld >> 2) & 1) == 0) ld += 4;
  return ld;
}

// targets of a tile: bit v of tmask[b] <=> item v0+v is in set b (rows sorted, binary search)
__device__ __forceinline__ uint32_t tile_targets(const int32_t* __restrict__ indices, int s, int e, int v0g) {
  int lo = s, hi = e;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (indices[mid] < v0g) lo = mid + 1; else hi = mid;
  }
  uint32_t m = 0;
  while (lo < e) {
    int d = indices[lo] - v0g;
    if (d >= TN) break;
    m |= 1u << d;
    ++lo;
  }
  return m;
}

template <int BC, int KB>
__global__ void __launch_bounds__(DT) dec_out_train_simt_kernel(
    const float* __restrict__ h2, int B, int H, float* __restrict__ Wd3, float* __restrict__ bd3,
    float* __restrict__ mW, float* __restrict__ vW, float* __restrict__ mb, float* __restrict__ vb, int v_begin,
    int Vloc, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices, float inv_n,
    const aae_step_state* __restrict__ st, float* __restrict__ dh2, double* __restrict__ loss_sum) {
  extern __shared__ __align__(16) float smem[];
  const int ldw = pad_ld(H);
  const int ldh = (H + 3) & ~3;
  float* Ws = smem;                       // [TN][ldw]
  float* Hs = Ws + TN * ldw;              // [BC][ldh]
  float* Zs = Hs + BC * ldh;              // [BC][TN+1]   dZ
  float* dbs = Zs + BC * ZLD;        // [TN]
  uint32_t* tmask = reinterpret_cast<uint32_t*>(dbs + TN);  // [BC]
  __shared__ float red[DT / 32];

  const int tid = threadIdx.x;
  const int tv = tid & 31, tb = tid >> 5;          // phase 1 mapping
  const int tk = tid & 127, tg = tid >> 7;         // phase 3/4/5 mapping (k, group)
  const int n_tiles = (Vloc + TN - 1) / TN;
  const int n_chunks = (B + BC - 1) / BC;
  const bool single = (n_chunks == 1);
  const AdamK ak = adam_load(st, 0);               // dec_optim uses gen_lr (aae.py:801)

  float dh2_acc[KB][BC / 2];
#pragma unroll
  for (int kb = 0; kb < KB; ++kb)
#pragma unroll
    for (int j = 0; j < BC / 2; ++j) dh2_acc[kb][j] = 0.f;
  float loss_local = 0.f;
  int loaded_chunk = -1;

  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int v0 = tile * TN;
    const int nv = min(TN, Vloc - v0);
    __syncthreads();
    // W tile -> smem (rows are contiguous in global)
    for (int q = tid; q < TN * ldh / 4; q += DT) {
      int r = q / (ldh / 4), c4 = q - r * (ldh / 4);
      float4 w = make_float4(0, 0, 0, 0);
      if (r < nv) {
        const float* src = Wd3 + (size_t)(v0 + r) * H + c4 * 4;
        if ((H & 3) == 0) w = *reinterpret_cast<const float4*>(src);
        else {
          w.x = (c4 * 4 + 0 < H) ? src[0] : 0.f; w.y = (c4 * 4 + 1 < H) ? src[1] : 0.f;
          w.z = (c4 * 4 + 2 < H) ? src[2] : 0.f; w.w = (c4 * 4 + 3 < H) ? src[3] : 0.f;
        }
      }
      *reinterpret_cast<float4*>(Ws + r * ldw + c4 * 4) = w;
    }
    if (tid < TN) dbs[tid] = 0.f;
    float dW_acc[KB][TN / 2];
#pragma unroll
    for (int kb = 0; kb < KB; ++kb)
#pragma unroll
      for (int j = 0; j < TN / 2; ++j) dW_acc[kb][j] = 0.f;

    for (int chunk = 0; chunk < n_chunks; ++chunk) {
      const int b0 = chunk * BC;
      const int nb = min(BC, B - b0);
      if (loaded_chunk != chunk) {
        __syncthreads();
        for (int q = tid; q < BC * ldh; q += DT) {
          int r = q / ldh, c = q - r * ldh;
          Hs[q] = (r < nb && c < H) ? h2[(size_t)(b0 + r) * H + c] : 0.f;
        }
        loaded_chunk = chunk;
      }
      if (tid < BC) {
        uint32_t m = 0;
        if (tid < nb) m = tile_targets(indices, indptr[b0 + tid], indptr[b0 + tid + 1], v_begin + v0);
        tmask[tid] = m;
      }
      __syncthreads();
      // ---- phase 1: logits for (b = tb + 8j, v = tv)
      float z[BC / 8];
#pragma unroll
      for (int j = 0; j < BC / 8; ++j) z[j] = 0.f;
      for (int k = 0; k < ldh; k += 4) {
        float4 w = *reinterpret_cast<const float4*>(Ws + tv * ldw + k);
#pragma unroll
        for (int j = 0; j < BC / 8; ++j) {
          float4 h = *reinterpret_cast<const float4*>(Hs + (tb + 8 * j) * ldh + k);
          z[j] = fmaf(w.x, h.x, z[j]);
          z[j] = fmaf(w.y, h.y, z[j]);
          z[j] = fmaf(w.z, h.z, z[j]);
          z[j] = fmaf(w.w, h.w, z[j]);
        }
      }
      // ---- phase 2: sigmoid + BCE + dZ
      float bias = (tv < nv) ? bd3[v0 + tv] : 0.f;
#pragma unroll
      for (int j = 0; j < BC / 8; ++j) {
        int b = tb + 8 * j;
        float dz = 0.f;
        if (b < nb && tv < nv) {
          bool pos = (tmask[b] >> tv) & 1u;
          loss_local += bce_term(z[j] + bias, pos, inv_n, dz);
        }
        Zs[b * ZLD + tv] = dz;
      }
      __syncthreads();
      // ---- bias gradient
      if (tid < TN) {
        float s = 0.f;
        for (int b = 0; b < nb; ++b) s += Zs[b * ZLD + tid];
        dbs[tid] += s;
      }
      // ---- phase 3: dW[v][k] += sum_b dZ[b][v] h2[b][k];  v = tg*16 + j
#pragma unroll
      for (int kb = 0; kb < KB; ++kb) {
        int k = kb * 128 + tk;
        if (k < H) {
          for (int b = 0; b < nb; ++b) {
            float h = Hs[b * ldh + k];
            const float4* zr = reinterpret_cast<const float4*>(Zs + b * ZLD + tg * (TN / 2));
#pragma unroll
            for (int j = 0; j < TN / 8; ++j) {
              float4 zq = zr[j];
              dW_acc[kb][4 * j + 0] = fmaf(zq.x, h, dW_acc[kb][4 * j + 0]);
              dW_acc[kb][4 * j + 1] = fmaf(zq.y, h, dW_acc[kb][4 * j + 1]);
              dW_acc[kb][4 * j + 2] = fmaf(zq.z, h, dW_acc[kb][4 * j + 2]);
              dW_acc[kb][4 * j + 3] = fmaf(zq.w, h, dW_acc[kb][4 * j + 3]);
            }
          }
        }
      }
      // ---- phase 4: dh2[b][k] += sum_v dZ[b][v] W[v][k];  b = tg + 2j
#pragma unroll
      for (int kb = 0; kb < KB; ++kb) {
        int k = kb * 128 + tk;
        if (k < H) {
          float wcol[TN];
#pragma unroll
          for (int v = 0; v < TN; ++v) wcol[v] = Ws[v * ldw + k];
#pragma unroll
          for (int j = 0; j < BC / 2; ++j) {
            int b = tg + 2 * j;
            float acc = 0.f;
            const float4* zr = reinterpret_cast<const float4*>(Zs + b * ZLD);
#pragma unroll
            for (int v = 0; v < TN / 4; ++v) {
              float4 zq = zr[v];
              acc = fmaf(zq.x, wcol[4 * v + 0], acc);
              acc = fmaf(zq.y, wcol[4 * v + 1], acc);
              acc = fmaf(zq.z, wcol[4 * v + 2], acc);
              acc = fmaf(zq.w, wcol[4 * v + 3], acc);
            }
            if (single) dh2_acc[kb][j] += acc;
            else if (b < nb) atomicAdd(dh2 + (size_t)(b0 + b) * H + k, acc);
          }
        }
      }
      __syncthreads();
    }
    // ---- phase 5: Adam on the tile (W rows from smem, moments streamed coalesced over k)
#pragma unroll
    for (int kb = 0; kb < KB; ++kb) {
      int k = kb * 128 + tk;
      if (k < H) {
#pragma unroll
        for (int j = 0; j < TN / 2; ++j) {
          int v = tg * (TN / 2) + j;
          if (v < nv) {
            size_t off = (size_t)(v0 + v) * H + k;
            float p = Ws[v * ldw + k], m = mW[off], vv = vW[off];
            adam_update(ak, dW_acc[kb][j], p, m, vv);
            Wd3[off] = p; mW[off] = m; vW[off] = vv;
          }
        }
      }
    }
    if (tid < nv) {
      float p = bd3[v0 + tid], m = mb[v0 + tid], vv = vb[v0 + tid];
      adam_update(ak, dbs[tid], p, m, vv);
      bd3[v0 + tid] = p; mb[v0 + tid] = m; vb[v0 + tid] = vv;
    }
  }
  // ---- flush dh2 (single-chunk case) and the loss
  if (single) {
#pragma unroll
    for (int kb = 0; kb < KB; ++kb) {
      int k = kb * 128 + tk;
      if (k < H) {
#pragma unroll
        for (int j = 0; j < BC / 2; ++j) {
          int b = tg + 2 * j;
          if (b < B && dh2_acc[kb][j] != 0.f) atomicAdd(dh2 + (size_t)b * H + k, dh2_acc[kb][j]);
        }
      }
    }
  }
  float s = warp_sum(loss_local);
  if ((tid & 31) == 0) red[tid >> 5] = s;
  __syncthreads();
  if (tid == 0) {
    double tot = 0.0;
    for (int w = 0; w < DT / 32; ++w) tot += (double)red[w];
    atomicAdd(loss_sum, tot);
  }
}

// scores: out[b][v] = (sigmoid)(h2[b,:].W[v,:] + bias[v])
template <int BC>
__global__ void __launch_bounds__(DT) dec_out_scores_simt_kernel(const float* __restrict__ h2, int B, int H,
                                                                 const float* __restrict__ Wd3,
                                                                 const float* __restrict__ bd3, int Vloc,
                                                                 int apply_sigmoid, float* __restrict__ out,
                                                                 int64_t ldo) {
  extern __shared__ __align__(16) float smem[];
  const int ldw = pad_ld(H);
  const int ldh = (H + 3) & ~3;
  float* Ws = smem;
  float* Hs = Ws + TN * ldw;
  const int tid = threadIdx.x, tv = tid & 31, tb = tid >> 5;
  const int n_tiles = (Vloc + TN - 1) / TN;
  const int n_chunks = (B + BC - 1) / BC;
  // grid.y splits the batch chunks so that large batches fill the machine
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int v0 = tile * TN;
    const int nv = min(TN, Vloc - v0);
    __syncthreads();
    for (int q = tid; q < TN * ldh / 4; q += DT) {
      int r = q / (ldh / 4), c4 = q - r * (ldh / 4);
      float4 w = make_float4(0, 0, 0, 0);
      if (r < nv) {
        const float* src = Wd3 + (size_t)(v0 + r) * H + c4 * 4;
        if ((H & 3) == 0) w = *reinterpret_cast<const float4*>(src);
        else {
          w.x = (c4 * 4 + 0 < H) ? src[0] : 0.f; w.y = (c4 * 4 + 1 < H) ? src[1] : 0.f;
          w.z = (c4 * 4 + 2 < H) ? src[2] : 0.f; w.w = (c4 * 4 + 3 < H) ? src[3] : 0.f;
        }
      }
      *reinterpret_cast<float4*>(Ws + r * ldw + c4 * 4) = w;
    }
    float bias = (tv < nv) ? bd3[v0 + tv] : 0.f;
    for (int chunk = blockIdx.y; chunk < n_chunks; chunk += gridDim.y) {
      const int b0 = chunk * BC;
      const int nb = min(BC, B - b0);
      __syncthreads();
      for (int q = tid; q < BC * ldh; q += DT) {
        int r = q / ldh, c = q - r * ldh;
        Hs[q] = (r < nb && c < H) ? h2[(size_t)(b0 + r) * H + c] : 0.f;
      }
      __syncthreads();
      float z[BC / 8];
#pragma unroll
      for (int j = 0; j < BC / 8; ++j) z[j] = 0.f;
      for (int k = 0; k < ldh; k += 4) {
        float4 w = *reinterpret_cast<const float4*>(Ws + tv * ldw + k);
#pragma unroll
        for (int j = 0; j < BC / 8; ++j) {
          float4 h = *reinterpret_cast<const float4*>(Hs + (tb + 8 * j) * ldh + k);
          z[j] = fmaf(w.x, h.x, z[j]);
          z[j] = fmaf(w.y, h.y, z[j]);
          z[j] = fmaf(w.z, h.z, z[j]);
          z[j] = fmaf(w.w, h.w, z[j]);
        }
      }
#pragma unroll
      for (int j = 0; j < BC / 8; ++j) {
        int b = tb + 8 * j;
        if (b < nb && tv < nv) {
          float s = z[j] + bias;
          if (apply_sigmoid) s = 1.0f / (1.0f + expf(-s));
          out[(size_t)(b0 + b) * ldo + v0 + tv] = s;
        }
      }
    }
  }
}

template <int BC, int KB>
static int launch_train(const float* h2, int B, int H, float* Wd3, float* bd3, float* mW, float* vW, float* mb,
                        float* vb, int v_begin, int Vloc, const int32_t* indptr, const int32_t* indices, float inv_n,
                        const aae_step_state* st, float* dh2, double* loss_sum, cudaStream_t s) {
  size_t smem = sizeof(float) * ((size_t)TN * pad_ld(H) + (size_t)BC * ((H + 3) & ~3) + (size_t)BC * ZLD + TN + BC);
  auto kern = dec_out_train_simt_kernel<BC, KB>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) {
    set_error("dec_out_train(simt): smem %zu: %s", smem, cudaGetErrorString(e));
    return AAE_E_CUDA;
  }
  int n_tiles = (Vloc + TN - 1) / TN;
  int grid = std::min(n_tiles, 2 * sm_count());
  kern<<<grid, DT, smem, s>>>(h2, B, H, Wd3, bd3, mW, vW, mb, vb, v_begin, Vloc, indptr, indices, inv_n, st, dh2,
                              loss_sum);
  return check_launch("dec_out_train(simt)");
}

int dec_out_train_simt(const float* h2, int B, int H, float* Wd3, float* bd3, float* mW, float* vW, float* mb,
                       float* vb, int v_begin, int Vloc, const int32_t* indptr, const int32_t* indices, double n_total,
                       const aae_step_state* st, float* dh2, double* loss_sum, cudaStream_t s) {
  float inv_n = (float)(1.0 / n_total);
  if (H <= 128)
    return launch_train<128, 1>(h2, B, H, Wd3, bd3, mW, vW, mb, vb, v_begin, Vloc, indptr, indices, inv_n, st, dh2,
                                loss_sum, s);
  if (H <= 256)
    return launch_train<64, 2>(h2, B, H, Wd3, bd3, mW, vW, mb, vb, v_begin, Vloc, indptr, indices, inv_n, st, dh2,
                               loss_sum, s);
  if (H <= 512)
    return launch_train<32, 4>(h2, B, H, Wd3, bd3, mW, vW, mb, vb, v_begin, Vloc, indptr, indices, inv_n, st, dh2,
                               loss_sum, s);
  set_error("dec_out_train: n_hidden %d > 512 is outside the supported envelope", H);
  return AAE_E_UNSUPPORTED;
}

int dec_out_scores_simt(const float* h2, int B, int H, const float* Wd3, const float* bd3, int Vloc, int apply_sigmoid,
                        float* out, int64_t ldo, cudaStream_t s) {
  if (H > 512) {
    set_error("dec_out_scores: n_hidden %d > 512 is outside the supported envelope", H);
    return AAE_E_UNSUPPORTED;
  }
  int n_tiles = (Vloc + TN - 1) / TN;
  int gx = std::min(n_tiles, 2 * sm_count());
  if (H <= 128) {
    constexpr int BC = 128;
    size_t smem = sizeof(float) * ((size_t)TN * pad_ld(H) + (size_t)BC * ((H + 3) & ~3));
    auto kern = dec_out_scores_simt_kernel<BC>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int n_chunks = (B + BC - 1) / BC;
    int gy = std::max(1, std::min(n_chunks, (4 * sm_count() + gx - 1) / gx));
    kern<<<dim3(gx, gy), DT, smem, s>>>(h2, B, H, Wd3, bd3, Vloc, apply_sigmoid, out, ldo);
  } else {
    constexpr int BC = 32;
    size_t smem = sizeof(float) * ((size_t)TN * pad_ld(H) + (size_t)BC * ((H + 3) & ~3));
    auto kern = dec_out_scores_simt_kernel<BC>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int n_chunks = (B + BC - 1) / BC;
    int gy = std::max(1, std::min(n_chunks, (4 * sm_count() + gx - 1) / gx));
    kern<<<dim3(gx, gy), DT, smem, s>>>(h2, B, H, Wd3, bd3, Vloc, apply_sigmoid, out, ldo);
  }
  return check_launch("dec_out_scores(simt)");
}

}  // namespace aae
