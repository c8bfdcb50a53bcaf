// Ranking tail: masked top-k over the item vocabulary, one CTA per query row.
// Replaces remove_non_missing + argtopk (aaerec/evaluation.py:183-199, 20-58) for the consumers
// that only need the k best unknown items (metrics at k in {1,5,10,20}, MPD submission k=500,
// eval/mpd/make_submission.py:36-53).  Min-max scaling is monotone per row, so ranking the raw
// scores gives the same order; known items are pushed to the bottom (the reference sets them to
// the row minimum, 0 after scaling).
//
// Algorithm (single HBM pass per row in the common case): sort a strided sample of the row in
// shared memory, take its j-th largest value as a threshold that is expected to keep ~max(6k,2048)
// elements, stream the row once collecting (key,index) pairs above the threshold, bitonic-sort
// the candidates in shared memory, emit the first k.  Too few / too many candidates -> retry with
// a lower / higher sample rank; pathological rows (huge tie groups) fall back to an exact
// bit-by-bit radix bisection.
#include <float.h>
#include <math.h>
#include <algorithm>
#include "dec_out.cuh"

namespace aae {

constexpr int TK_THREADS = 1024;
constexpr int TK_SAMPLE = 4096;
constexpr int TK_CAP = 8192;

__device__ __forceinline__ uint32_t f2key(float f) {
  uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
  uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(b);
}

__global__ void mask_known_kernel(float* __restrict__ scores, int64_t lds, int B, int Vloc, int v_begin,
                                  const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices) {
  int nnz = indptr[B];
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += gridDim.x * blockDim.x) {
    // row of entry e: binary search in indptr
    int lo = 0, hi = B;
    while (lo < hi) {
      int mid = (lo + hi) >> 1;
      if (indptr[mid + 1] <= e) lo = mid + 1; else hi = mid;
    }
    int i = indices[e] - v_begin;
    if (i >= 0 && i < Vloc) scores[(size_t)lo * lds + i] = -FLT_MAX;
  }
}

// Candidate filter of a ranking call (aae_rank_filter): the columns are the ascending global ids ids[0..n) (NULL:
// v_begin + column), and excluded (row, id) pairs come as a CSR with sorted rows (NULL: none).
struct RankFilt {
  const int32_t* ids; const int32_t* xp; const int32_t* xi;
};
// true iff global id g is in CSR row `row` (sorted columns)
__device__ __forceinline__ bool csr_has(const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices, int row,
                                        int g) {
  int lo = indptr[row], hi = indptr[row + 1];
  const int end = hi;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(indices + mid) < g) lo = mid + 1; else hi = mid;
  }
  return lo < end && __ldg(indices + lo) == g;
}
// column of global id g, or -1 when g is not a column
__device__ __forceinline__ int col_of(const int32_t* __restrict__ ids, int n, int v_begin, int g) {
  if (!ids) return (g >= v_begin && g - v_begin < n) ? g - v_begin : -1;
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(ids + mid) < g) lo = mid + 1; else hi = mid;
  }
  return (lo < n && __ldg(ids + lo) == g) ? lo : -1;
}
// mask_known_kernel on a filtered column set: scores[row, col_of(id)] = fill for every CSR entry whose id is a column
// (fill = -FLT_MAX for the known items, -INFINITY for the exclusions)
__global__ void mask_cols_kernel(float* __restrict__ scores, int64_t lds, int B, int n, int v_begin,
                                 const int32_t* __restrict__ ids, const int32_t* __restrict__ indptr,
                                 const int32_t* __restrict__ indices, float fill) {
  const int nnz = indptr[B];
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += gridDim.x * blockDim.x) {
    int lo = 0, hi = B;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (indptr[mid + 1] <= e) lo = mid + 1; else hi = mid;
    }
    const int c = col_of(ids, n, v_begin, indices[e]);
    if (c >= 0) scores[(size_t)lo * lds + c] = fill;
  }
}
// Compact copy of the eligible rows of an item shard: Wd3c[j,:] = Wd3[ids[j] - v_begin, :], bd3c[j] = bd3[...]; one warp
// per row (float4 when H % 4 == 0).  An id outside the shard reads nothing (its row becomes zeros with bias -inf); ids
// outside the shard or not above their predecessor are counted in *n_bad_ids.
__global__ void gather_item_rows_kernel(const float* __restrict__ Wd3, const float* __restrict__ bd3, int H, int Vloc,
                                        int v_begin, const int32_t* __restrict__ ids, int A, float* __restrict__ Wd3c,
                                        float* __restrict__ bd3c, int32_t* __restrict__ n_bad_ids) {
  const int lane = threadIdx.x & 31;
  const int nw = (gridDim.x * blockDim.x) >> 5;
  for (int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < A; j += nw) {
    const int r = ids[j] - v_begin;
    const bool in = r >= 0 && r < Vloc;
    if (lane == 0 && (!in || (j > 0 && ids[j - 1] >= ids[j]))) atomicAdd(n_bad_ids, 1);
    float* dst = Wd3c + (size_t)j * H;
    if ((H & 3) == 0) {
      const float4* src = reinterpret_cast<const float4*>(Wd3 + (size_t)(in ? r : 0) * H);
      for (int c = lane; c < (H >> 2); c += 32)
        reinterpret_cast<float4*>(dst)[c] = in ? __ldg(src + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
      for (int c = lane; c < H; c += 32) dst[c] = in ? __ldg(Wd3 + (size_t)r * H + c) : 0.f;
    }
    if (lane == 0) bd3c[j] = in ? __ldg(bd3 + r) : -INFINITY;
  }
}

// descending bitonic sort of n (power of two) 64-bit composites in shared memory
__device__ void bitonic_desc(unsigned long long* a, int n) {
  for (int size = 2; size <= n; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int t = threadIdx.x; t < (n >> 1); t += blockDim.x) {
        int lo = 2 * t - (t & (stride - 1));
        int hi = lo + stride;
        bool desc = ((lo & size) == 0);
        unsigned long long x = a[lo], y = a[hi];
        if ((x < y) == desc) { a[lo] = y; a[hi] = x; }
      }
    }
  }
  __syncthreads();
}

__device__ __forceinline__ unsigned long long compose(uint32_t key, uint32_t idx) {
  return ((unsigned long long)key << 32) | (unsigned long long)(0xFFFFFFFFu - idx);
}

// collect every element of the row with key > thr (or >= thr) into buf; returns the count in *cnt
__device__ void collect(const float* __restrict__ row, int n, uint32_t thr, bool inclusive, unsigned long long* buf,
                        int* cnt) {
  int lane = threadIdx.x & 31;
  for (int base = 0; base < n; base += blockDim.x) {
    int i = base + threadIdx.x;
    bool take = false;
    uint32_t key = 0;
    if (i < n) {
      key = f2key(__ldcs(row + i));
      take = inclusive ? (key >= thr) : (key > thr);
    }
    unsigned bal = __ballot_sync(0xffffffffu, take);
    if (bal) {
      int pos = 0;
      if (lane == 0) pos = atomicAdd(cnt, __popc(bal));
      pos = __shfl_sync(0xffffffffu, pos, 0);
      if (take) {
        int p = pos + __popc(bal & ((1u << lane) - 1));
        if (p < TK_CAP) buf[p] = compose(key, (uint32_t)i);
      }
    }
  }
  __syncthreads();
}

__device__ int block_count_ge(const float* __restrict__ row, int n, uint32_t thr, int* scratch) {
  if (threadIdx.x == 0) *scratch = 0;
  __syncthreads();
  int c = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) c += (f2key(row[i]) >= thr);
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(scratch, c);
  __syncthreads();
  int r = *scratch;
  __syncthreads();
  return r;
}

// idx_map == nullptr: candidates are row positions (+ idx_offset); else idx_out = idx_map[row, pos]
// FILT: the id found that way is a column of a filtered set: emitted as ids[id] (ids NULL: as is); entries scored
// -INFINITY (excluded) and the padding of rows shorter than k are emitted as (-1, -INFINITY)
template <bool FILT>
__global__ void __launch_bounds__(TK_THREADS, 1) row_topk_kernel(const float* __restrict__ scores, int64_t lds, int n,
                                                                 int k, int idx_offset,
                                                                 const int32_t* __restrict__ idx_map,
                                                                 const int32_t* __restrict__ n_valid,
                                                                 int skip_upto, int32_t* __restrict__ idx_out,
                                                                 float* __restrict__ val_out,
                                                                 const int32_t* __restrict__ ids) {
  extern __shared__ __align__(16) unsigned char sm_raw[];
  unsigned long long* buf = reinterpret_cast<unsigned long long*>(sm_raw);          // [TK_CAP]
  uint32_t* samp = reinterpret_cast<uint32_t*>(buf + TK_CAP);                       // [TK_SAMPLE] (as u64 pairs)
  __shared__ int cnt;
  __shared__ int scratch;
  const int rowi = blockIdx.x;
  const float* row = scores + (size_t)rowi * lds;
  if (n_valid) n = max(0, min(n, n_valid[rowi]));     // only the first n_valid[row] entries of the row are live
  if (n <= skip_upto) return;                         // rows this short are ranked by cand_sort_small_kernel
  const int kk = min(k, n);
  int total = 0;
  const bool direct_ids = idx_map != nullptr && n <= TK_CAP;   // composites carry the item id itself
  if (n <= TK_CAP) {
    for (int i = threadIdx.x; i < TK_CAP; i += blockDim.x)
      buf[i] = (i < n) ? compose(f2key(row[i]), direct_ids ? (uint32_t)idx_map[(size_t)rowi * lds + i] : (uint32_t)i)
                       : 0ull;
    total = n;
    __syncthreads();
  } else {
    // ---- sample, sort, pick a threshold
    unsigned long long* sbuf = reinterpret_cast<unsigned long long*>(samp);
    double stride = (double)n / TK_SAMPLE;
    for (int s = threadIdx.x; s < TK_SAMPLE; s += blockDim.x) {
      int p = min(n - 1, (int)(s * stride));
      sbuf[s] = compose(f2key(row[p]), 0u);
    }
    bitonic_desc(sbuf, TK_SAMPLE);
    int target = max(6 * kk, 2048);
    int j = max(2, (int)((double)target * TK_SAMPLE / n + 0.5));
    j = min(j, TK_SAMPLE - 1);
    bool ok = false;
    for (int attempt = 0; attempt < 5 && !ok; ++attempt) {
      uint32_t thr = (uint32_t)(sbuf[j] >> 32);
      if (threadIdx.x == 0) cnt = 0;
      __syncthreads();
      collect(row, n, thr, false, buf, &cnt);
      total = cnt;
      __syncthreads();
      if (total >= kk && total <= TK_CAP) ok = true;
      else if (total > TK_CAP) j = max(0, j / 2 - (j <= 1));
      else j = min(TK_SAMPLE - 1, 2 * j + 2);
    }
    if (!ok) {
      // ---- exact fallback: largest threshold T with count(key >= T) >= kk, bit by bit
      uint32_t T = 0;
      for (int bit = 31; bit >= 0; --bit) {
        uint32_t cand = T | (1u << bit);
        if (block_count_ge(row, n, cand, &scratch) >= kk) T = cand;
      }
      if (threadIdx.x == 0) cnt = 0;
      __syncthreads();
      collect(row, n, T, false, buf, &cnt);          // strictly greater: fewer than kk of them
      int gt = min(cnt, TK_CAP);
      __syncthreads();
      // fill with ties (== T) in index order (serial over chunks; ties are exempt from parity)
      if (threadIdx.x == 0) {
        int need = kk - gt, got = 0;
        for (int i = 0; i < n && got < need; ++i)
          if (f2key(row[i]) == T) { buf[gt + got] = compose(T, (uint32_t)i); ++got; }
        cnt = gt + got;
      }
      __syncthreads();
      total = cnt;
    }
    for (int i = total + threadIdx.x; i < TK_CAP; i += blockDim.x) buf[i] = 0ull;
    __syncthreads();
  }
  int npow = 1;
  while (npow < total) npow <<= 1;
  npow = max(npow, 2);
  bitonic_desc(buf, npow);
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    int32_t id = -1;
    float val = FILT ? -INFINITY : -FLT_MAX;
    if (i < kk) {
      unsigned long long c = buf[i];
      uint32_t pos = 0xFFFFFFFFu - (uint32_t)(c & 0xFFFFFFFFull);
      id = direct_ids ? (int32_t)pos : (idx_map ? idx_map[(size_t)rowi * lds + pos] : (int32_t)pos + idx_offset);
      val = key2f((uint32_t)(c >> 32));
      if (FILT) id = (val == -INFINITY || id < 0) ? -1 : (ids ? ids[id] : id);
    }
    idx_out[(size_t)rowi * k + i] = id;
    if (val_out) val_out[(size_t)rowi * k + i] = val;
  }
}

// Candidate sub-lists of the fused predict path -> one compact list per row, ready for the final sort.  Row b owns
// nsub private sub-lists of cap_sub slots (written without atomics by the filter epilogue, counts in cnt[b*nsub+s]);
// they are concatenated in sub-list order (deterministic), known items of the row (sorted CSR columns) are pushed to
// the bottom.  Rows with an overflowed sub-list, more than cap_out candidates or fewer than k unknown ones are counted
// in n_bad (the caller then re-ranks the batch through the dense path -- exactness never depends on the threshold
// estimate).  One CTA per row.
// RESCORE (K5 v2): the sub-lists hold item ids only (they passed an approximate single-pass TF32 filter); every unknown
// candidate is scored here exactly in fp32 -- one warp per candidate: z = h2'[b,:] . Wd3[item,:] + bd3[item], lanes over
// the float4 columns, fixed reduction order -- so the final ranking never sees an approximate value.
struct RescoreArgs {
  const float* h2; const float* Wd3; const float* bd3; int H; int v_begin;
};
// FILT: the candidate ids are columns of a filtered set (global id f.ids[id], or id itself when f.ids is NULL): known
// items are looked up by global id, excluded candidates are dropped (value -INFINITY, not counted as returnable); the
// ids stay columns (the final sort translates them), so that re-scoring reads compact row `id`.
constexpr int FIN_THREADS = 256;
template <bool RESCORE, bool FILT>
__global__ void __launch_bounds__(FIN_THREADS) cand_finish_kernel(const float* __restrict__ cand_val,
                                                                  const int32_t* __restrict__ cand_idx,
                                                                  const int32_t* __restrict__ cnt, int nsub, int cap_sub,
                                                                  float* __restrict__ out_val, int32_t* __restrict__ out_idx,
                                                                  int cap_out, int32_t* __restrict__ tot, int B, int k,
                                                                  const int32_t* __restrict__ indptr,
                                                                  const int32_t* __restrict__ indices, int32_t* n_bad,
                                                                  RescoreArgs ra, RankFilt f) {
  extern __shared__ int off_s[];                 // [nsub + 1] exclusive prefix of the sub-list counts (+ h2 row if RESCORE)
  __shared__ int warp_s[FIN_THREADS / 32];
  __shared__ int valid_s, over_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per = (nsub + FIN_THREADS - 1) / FIN_THREADS;
  for (int row = blockIdx.x; row < B; row += gridDim.x) {
    if (tid == 0) { valid_s = 0; over_s = 0; }
    __syncthreads();
    // block-wide exclusive scan of min(cnt, cap_sub)
    int mine = 0, over = 0;
    for (int q = 0; q < per; ++q) {
      const int sidx = tid * per + q;
      if (sidx < nsub) {
        const int c = cnt[(size_t)row * nsub + sidx];
        over |= (c > cap_sub);
        mine += min(c, cap_sub);
      }
    }
    int incl = mine;
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += y;
    }
    if (lane == 31) warp_s[warp] = incl;
    if (over) over_s = 1;
    __syncthreads();
    int wbase = 0;
    for (int w = 0; w < warp; ++w) wbase += warp_s[w];
    int run = wbase + incl - mine;
    for (int q = 0; q < per; ++q) {
      const int sidx = tid * per + q;
      if (sidx < nsub) {
        off_s[sidx] = run;
        run += min(cnt[(size_t)row * nsub + sidx], cap_sub);
      }
    }
    if (tid == FIN_THREADS - 1) off_s[nsub] = run;
    __syncthreads();
    const int total = off_s[nsub];
    const bool fits = total <= cap_out;
    const int p0 = indptr ? indptr[row] : 0, p1 = indptr ? indptr[row + 1] : 0;
    int valid = 0;
    if (fits) {
      for (int q = tid; q < nsub * cap_sub; q += FIN_THREADS) {
        const int sidx = q / cap_sub, sl = q - sidx * cap_sub;
        const int o0 = off_s[sidx];
        if (sl >= off_s[sidx + 1] - o0) continue;
        const size_t src = ((size_t)row * nsub + sidx) * cap_sub + sl;
        const int id = cand_idx[src];
        float v = RESCORE ? 0.f : cand_val[src];
        const int g = (FILT && f.ids) ? __ldg(f.ids + id) : id;
        int lo = p0, hi = p1;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (__ldg(indices + mid) < g) lo = mid + 1; else hi = mid;
        }
        if (FILT && f.xp && csr_has(f.xp, f.xi, row, g)) v = -INFINITY;
        else if (lo < p1 && __ldg(indices + lo) == g) v = -FLT_MAX;
        else ++valid;
        out_val[(size_t)row * cap_out + o0 + sl] = v;
        out_idx[(size_t)row * cap_out + o0 + sl] = id;
      }
    }
    for (int o = 16; o > 0; o >>= 1) valid += __shfl_xor_sync(0xffffffffu, valid, o);
    if (lane == 0 && valid) atomicAdd(&valid_s, valid);
    if (RESCORE) {
      float* hrow = reinterpret_cast<float*>(off_s + ((nsub + 4) & ~3));     // 16-byte aligned behind the prefix
      for (int c = tid; c < ra.H; c += FIN_THREADS) hrow[c] = ra.h2[(size_t)row * ra.H + c];
    }
    __syncthreads();
    if (RESCORE && fits) {
      // EIGHT LANES per candidate (four candidates per warp pass): the lanes of a group read consecutive float4 of the
      // candidate's 400-byte Wd3 row, so a warp-wide load touches 4 rows x 128 contiguous bytes (4 wavefronts) instead of
      // 32 rows x 16 bytes (32 wavefronts: one thread per candidate was bound by the L1 wavefront rate, 329 us for 1000
      // rows whatever the unrolling); the h2 row is a shared-memory broadcast; fixed reduction order (deterministic).
      const float* hrow = reinterpret_cast<const float*>(off_s + ((nsub + 4) & ~3));
      const float4* h4 = reinterpret_cast<const float4*>(hrow);
      const int H4 = ra.H >> 2;
      const int sub = lane >> 3, l8 = lane & 7;
      for (int c0 = warp * 4; c0 < total; c0 += (FIN_THREADS / 32) * 4) {
        const int c = c0 + sub;
        const size_t o = (size_t)row * cap_out + c;
        // -FLT_MAX: a known item, stays at the bottom; -INFINITY: an excluded one
        const bool live = c < total && out_val[o] != -FLT_MAX && (!FILT || out_val[o] != -INFINITY);
        float acc = 0.f;
        int item = 0;
        if (live) {
          item = out_idx[o] - ra.v_begin;
          const float4* wrow = reinterpret_cast<const float4*>(ra.Wd3 + (size_t)item * ra.H);
          for (int c4 = l8; c4 < H4; c4 += 8) {
            const float4 w = __ldg(wrow + c4);
            const float4 h = h4[c4];
            acc = fmaf(w.x, h.x, acc); acc = fmaf(w.y, h.y, acc); acc = fmaf(w.z, h.z, acc); acc = fmaf(w.w, h.w, acc);
          }
        }
        acc += __shfl_xor_sync(0xffffffffu, acc, 4);
        acc += __shfl_xor_sync(0xffffffffu, acc, 2);
        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
        if (live && l8 == 0) out_val[o] = acc + __ldg(ra.bd3 + item);
      }
    }
    if (tid == 0) {
      tot[row] = fits ? total : 0;
      if (over_s || !fits || valid_s < k) atomicAdd(n_bad, 1);
    }
    __syncthreads();
  }
}

// K5 v2: filter threshold of row b = tau_b - (bound of the single-pass TF32 error of the row's logits).
// Both operands are truncated to tf32 (10 explicit mantissa bits: relative error < 2^-10 each), so
// |z_tf32 - z| <= (2^-9 + 2^-20) * sum_k |h'_k w'_k| + accumulation error <= 2.1 * 2^-10 * ||h'_b|| * max_v ||w'_v||
// (Cauchy-Schwarz; h' = [h2 | 1], w' = [Wd3 | bd3]).  One warp per row.
__global__ void __launch_bounds__(256) tau_margin_kernel(const float* __restrict__ thr, int thr_stride,
                                                         const float* __restrict__ h2, int B, int H,
                                                         const float* __restrict__ wmax, float* __restrict__ tau_f) {
  const int lane = threadIdx.x & 31;
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= B) return;
  float ss = 0.f;
  for (int c = lane; c < H; c += 32) {
    const float x = h2[(size_t)row * H + c];
    ss = fmaf(x, x, ss);
  }
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if (lane == 0) {
    const float margin = 2.1f * 0.0009765625f * sqrtf(ss + 1.0f) * (*wmax);
    tau_f[row] = thr[(size_t)row * thr_stride] - margin;
  }
}
// The ranking is exact iff every item whose exact score reaches the k-th exact score passed the filter.  An item with
// exact score z has a TF32 score >= z - margin, and the filter kept everything above tau - margin: rows whose k-th exact
// score does not clear tau are reported (the caller re-ranks them through the exact dense path).
__global__ void check_kth_kernel(const float* __restrict__ val, int k, const float* __restrict__ thr, int thr_stride,
                                 const int32_t* __restrict__ tot, int B, int32_t* n_bad) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= B || tot[row] == 0) return;                 // tot == 0: already counted by cand_finish
  if (!(val[(size_t)row * k + (k - 1)] > thr[(size_t)row * thr_stride])) atomicAdd(n_bad, 1);
}

// Final ranking of a short candidate list (the common case of the fused predict path: ~1.4 k live candidates per row):
// 256 threads and 16 KB of shared memory per row instead of 1024 threads and 96 KB, so that eight rows are sorted per
// SM at a time.  Rows with more than CS_CAP live candidates are left to row_topk_kernel (skip_upto = CS_CAP there).
// Composites carry the item id: descending score, ties by lower id -- the same order as row_topk_kernel.
// FILT: ids are translated and excluded / padding entries emitted as in row_topk_kernel<true>.
constexpr int CS_THREADS = 256, CS_CAP = 2048;
template <bool FILT>
__global__ void __launch_bounds__(CS_THREADS) cand_sort_small_kernel(const float* __restrict__ val,
                                                                     const int32_t* __restrict__ idx, int64_t lds,
                                                                     const int32_t* __restrict__ n_valid, int k,
                                                                     int32_t* __restrict__ idx_out,
                                                                     float* __restrict__ val_out,
                                                                     const int32_t* __restrict__ ids) {
  __shared__ unsigned long long buf[CS_CAP];
  const int rowi = blockIdx.x;
  const int n = n_valid[rowi];
  if (n > CS_CAP) return;
  int npow = 2;
  while (npow < n) npow <<= 1;
  for (int i = threadIdx.x; i < npow; i += CS_THREADS)
    buf[i] = (i < n) ? compose(f2key(val[(size_t)rowi * lds + i]), (uint32_t)idx[(size_t)rowi * lds + i]) : 0ull;
  bitonic_desc(buf, npow);
  const int kk = min(k, n);
  for (int i = threadIdx.x; i < k; i += CS_THREADS) {
    int32_t id = -1;
    float v = FILT ? -INFINITY : -FLT_MAX;
    if (i < kk) {
      const unsigned long long c = buf[i];
      id = (int32_t)(0xFFFFFFFFu - (uint32_t)(c & 0xFFFFFFFFull));
      v = key2f((uint32_t)(c >> 32));
      if (FILT) id = v == -INFINITY ? -1 : (ids ? ids[id] : id);
    }
    idx_out[(size_t)rowi * k + i] = id;
    if (val_out) val_out[(size_t)rowi * k + i] = v;
  }
}

// k-way merge of per-shard top-k lists that an all-gather left in [world][B][kpad] order (item-sharded predict): one
// CTA per row gathers its world * kpad <= CS_CAP candidates from the segments and sorts them in shared memory.
__global__ void __launch_bounds__(CS_THREADS) seg_merge_small_kernel(const float* __restrict__ val,
                                                                     const int32_t* __restrict__ idx, int world, int B,
                                                                     int kpad, int k, int32_t* __restrict__ idx_out,
                                                                     float* __restrict__ val_out) {
  __shared__ unsigned long long buf[CS_CAP];
  const int rowi = blockIdx.x;
  const int n = world * kpad;
  int npow = 2;
  while (npow < n) npow <<= 1;
  for (int i = threadIdx.x; i < npow; i += CS_THREADS) {
    unsigned long long c = 0ull;
    if (i < n) {
      const int r = i / kpad, j = i - r * kpad;
      const size_t src = ((size_t)r * B + rowi) * kpad + j;
      const int32_t id = idx[src];
      c = (id >= 0) ? compose(f2key(val[src]), (uint32_t)id) : 0ull;
    }
    buf[i] = c;
  }
  bitonic_desc(buf, npow);
  for (int i = threadIdx.x; i < k; i += CS_THREADS) {
    const unsigned long long c = buf[i];
    int32_t id = -1;
    float v = -FLT_MAX;
    if (c != 0ull) {
      id = (int32_t)(0xFFFFFFFFu - (uint32_t)(c & 0xFFFFFFFFull));
      v = key2f((uint32_t)(c >> 32));
    }
    idx_out[(size_t)rowi * k + i] = id;
    if (val_out) val_out[(size_t)rowi * k + i] = v;
  }
}

// Threshold of the fused predict path: (approximately) the J-th largest of the row's S sample scores.  Every
// thread keeps the 4 largest of its strided share in registers, the 256 x 4 survivors are sorted in shared memory
// and the J-th is taken.  A thread that holds more than 4 of the row's top J makes the result slightly LOWER than
// the true order statistic -- a few more candidates pass the filter, nothing else: exactness is guarded by n_bad.
constexpr int KTH_THREADS = 256, KTH_KEEP = 4;
__global__ void __launch_bounds__(KTH_THREADS) row_kth_approx_kernel(const float* __restrict__ samp, int64_t lds, int S,
                                                                     int J, float* __restrict__ tau) {
  __shared__ unsigned long long buf[KTH_THREADS * KTH_KEEP];
  const float* row = samp + (size_t)blockIdx.x * lds;
  float t0 = -FLT_MAX, t1 = -FLT_MAX, t2 = -FLT_MAX, t3 = -FLT_MAX;      // t0 >= t1 >= t2 >= t3
  auto push = [&](float x) {
    if (x > t3) {
      if (x > t1) {
        t3 = t2; t2 = t1;
        if (x > t0) { t1 = t0; t0 = x; } else t1 = x;
      } else {
        if (x > t2) { t3 = t2; t2 = x; } else t3 = x;
      }
    }
  };
  if ((S & 3) == 0 && (lds & 3) == 0) {
    for (int i = threadIdx.x; i < (S >> 2); i += KTH_THREADS) {
      const float4 x = __ldcs(reinterpret_cast<const float4*>(row) + i);
      push(x.x); push(x.y); push(x.z); push(x.w);
    }
  } else {
    for (int i = threadIdx.x; i < S; i += KTH_THREADS) push(__ldcs(row + i));
  }
  buf[threadIdx.x * KTH_KEEP + 0] = compose(f2key(t0), 0u);
  buf[threadIdx.x * KTH_KEEP + 1] = compose(f2key(t1), 0u);
  buf[threadIdx.x * KTH_KEEP + 2] = compose(f2key(t2), 0u);
  buf[threadIdx.x * KTH_KEEP + 3] = compose(f2key(t3), 0u);
  bitonic_desc(buf, KTH_THREADS * KTH_KEEP);
  if (threadIdx.x == 0) tau[blockIdx.x] = key2f((uint32_t)(buf[min(J, KTH_THREADS * KTH_KEEP) - 1] >> 32));
}

// Plan of the fused predict + top-k path for one (Vloc, k): sample tiles, threshold rank, candidate capacity.
struct TopkPlan {
  int n_tiles, n_samp, stride, S, T, J, cap;
  int nsub, cap_sub;       // private candidate sub-lists per row (one per CTA column and 16-column tile part)
  bool ok;
};

static TopkPlan make_plan(int B, int Vloc, int k, bool v2 = false) {
  TopkPlan p;
  p.n_tiles = (Vloc + 127) / 128;
  p.n_samp = std::min(512, p.n_tiles / 8);
  p.ok = p.n_samp >= 32 && k <= 1024;          // Vloc >= 32641 (256 tiles); below that the dense path is as cheap
  p.stride = p.ok ? p.n_tiles / p.n_samp : 1;
  p.S = p.n_samp * 128;
  p.T = std::max(1024, std::min(4096, 4 * (k + 256)));
  p.cap = TK_CAP;
  p.J = p.ok ? std::max(8, (int)(((int64_t)p.T * p.S + Vloc - 1) / Vloc)) : 8;
  int gx = 1, gy = 1;
  if (v2) dec_out_select2_grid(B, p.n_tiles, &gx, &gy);
  else dec_out_select_grid(B, p.n_tiles, &gx, &gy);
  p.nsub = 4 * gx;
  // expected T / nsub candidates per sub-list; room for 8 sigma of a Poisson count, and for the worst clustering of
  // twice T candidates in consecutive items (32 per visited tile part)
  const double e = (double)p.T / p.nsub;
  const int stat = (int)(e + 8.0 * sqrt(e) + 8.0);
  const int clus = 32 * ((2 * p.T / 128 + gx - 1) / gx) + 8;
  p.cap_sub = std::max(stat, clus);
  return p;
}
static size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }


// ---------------------------------------------------------------------------------------------
// Rank of the gold items (SURVEY 8(f)-2; evaluation.py:70-164, 202-240 need, per test row, the positions of the
// held-out items in the descending ranking of remove_non_missing(predict(X), X)): rank - 1 = number of unknown
// items scored strictly higher (+ equal-score items with a lower id: the deterministic tie order of the top-k
// kernels).  Known items are -FLT_MAX in `scores` (mask_known_kernel) = the bottom of the ranking, where the
// reference's min-max scaling + zeroing puts them.
//   gold_scores_kernel : zg[p] = scores[row(p), gold[p]]  (NaN when the item belongs to another shard)
//   rank_count_kernel  : grid (column chunks, rows); each CTA counts, for up to RC_G gold items of its row at a
//                        time, the entries of its column chunk that rank before them; one atomicAdd per CTA and gold.
// The bodies take FILT: the columns are those of a filtered set (ids = ascending global id of each column, NULL:
// v_begin + column).  The gold items stay global ids; a gold's tie position is then lb = lower_bound(ids, gold), the
// number of columns with a lower id, so "column < lb" is "id < gold" also for a gold that is not a column.  The
// unfiltered kernels instantiate FILT = false and keep their names; the *_filt_kernel ones instantiate FILT = true.
// rank_count_body takes threadIdx.x from its kernel: read there, it carries the range the kernel's launch bounds give
// it, so the FILT = false instantiation compiles to the code of the kernel before it was split.
// ---------------------------------------------------------------------------------------------
template <bool FILT>
__device__ __forceinline__ void gold_scores_body(const float* __restrict__ scores, int64_t lds, int B, int Vloc,
                                                 int v_begin, const int32_t* __restrict__ gold_indptr,
                                                 const int32_t* __restrict__ gold_indices, float* __restrict__ zg,
                                                 const int32_t* __restrict__ ids) {
  const int n = gold_indptr[B];
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
    int lo = 0, hi = B;
    while (lo < hi) {
      int mid = (lo + hi) >> 1;
      if (gold_indptr[mid + 1] <= e) lo = mid + 1; else hi = mid;
    }
    const int i = FILT ? col_of(ids, Vloc, v_begin, gold_indices[e]) : gold_indices[e] - v_begin;
    zg[e] = (i >= 0 && i < Vloc) ? scores[(size_t)lo * lds + i] : __int_as_float(0x7fc00000);
  }
}
__global__ void gold_scores_kernel(const float* __restrict__ scores, int64_t lds, int B, int Vloc, int v_begin,
                                   const int32_t* __restrict__ gold_indptr, const int32_t* __restrict__ gold_indices,
                                   float* __restrict__ zg) {
  gold_scores_body<false>(scores, lds, B, Vloc, v_begin, gold_indptr, gold_indices, zg, nullptr);
}
__global__ void gold_scores_filt_kernel(const float* __restrict__ scores, int64_t lds, int B, int Vloc, int v_begin,
                                        const int32_t* __restrict__ gold_indptr,
                                        const int32_t* __restrict__ gold_indices, float* __restrict__ zg,
                                        const int32_t* __restrict__ ids) {
  gold_scores_body<true>(scores, lds, B, Vloc, v_begin, gold_indptr, gold_indices, zg, ids);
}
constexpr int RC_THREADS = 256, RC_G = 8, RC_CHUNK = 16384;
template <bool FILT>
__device__ __forceinline__ void rank_count_body(const float* __restrict__ scores, int64_t lds, int Vloc, int v_begin,
                                                const int32_t* __restrict__ gold_indptr,
                                                const int32_t* __restrict__ gold_indices,
                                                const float* __restrict__ zg, int32_t* __restrict__ cnt,
                                                const int32_t* __restrict__ ids, unsigned tid) {
  __shared__ int red[RC_THREADS / 32 + (FILT ? 1 : 0)][RC_G];    // FILT: the last row holds the gold tie positions
  int* lb_s = red[RC_THREADS / 32];
  const int row = blockIdx.y;
  const int c0 = blockIdx.x * RC_CHUNK, c1 = min(Vloc, c0 + RC_CHUNK);
  const int p0 = gold_indptr[row], p1 = gold_indptr[row + 1];
  const float* r = scores + (size_t)row * lds;
  const int lane = tid & 31, warp = tid >> 5;
  for (int g0 = p0; g0 < p1; g0 += RC_G) {
    if (FILT && ids) {          // tie position of each gold of the group, once per CTA (ids is uniform: no divergence)
      if (tid < RC_G && g0 + tid < p1) {
        const int g = gold_indices[g0 + tid];
        int lo = 0, hi = Vloc;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (__ldg(ids + mid) < g) lo = mid + 1; else hi = mid;
        }
        lb_s[tid] = lo;
      }
      __syncthreads();
    }
    float z[RC_G];
    int id[RC_G], c[RC_G];
#pragma unroll
    for (int j = 0; j < RC_G; ++j) {
      const bool ok = g0 + j < p1;
      z[j] = ok ? zg[g0 + j] : __int_as_float(0x7fc00000);      // NaN compares false: counts stay 0
      id[j] = ok ? ((FILT && ids) ? lb_s[j] : gold_indices[g0 + j] - v_begin) : -1;
      c[j] = 0;
    }
    for (int v = c0 + tid; v < c1; v += RC_THREADS) {
      const float x = r[v];
#pragma unroll
      for (int j = 0; j < RC_G; ++j) c[j] += (x > z[j] || (x == z[j] && v < id[j])) ? 1 : 0;
    }
#pragma unroll
    for (int j = 0; j < RC_G; ++j) {
      int t = c[j];
      for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
      if (lane == 0) red[warp][j] = t;
    }
    __syncthreads();
    if (tid < RC_G && g0 + tid < p1) {
      int t = 0;
      for (int w = 0; w < RC_THREADS / 32; ++w) t += red[w][tid];
      if (t) atomicAdd(cnt + g0 + tid, t);
    }
    __syncthreads();
  }
}
__global__ void __launch_bounds__(RC_THREADS) rank_count_kernel(const float* __restrict__ scores, int64_t lds, int Vloc,
                                                                int v_begin,
                                                                const int32_t* __restrict__ gold_indptr,
                                                                const int32_t* __restrict__ gold_indices,
                                                                const float* __restrict__ zg,
                                                                int32_t* __restrict__ cnt) {
  rank_count_body<false>(scores, lds, Vloc, v_begin, gold_indptr, gold_indices, zg, cnt, nullptr, threadIdx.x);
}
__global__ void __launch_bounds__(RC_THREADS) rank_count_filt_kernel(const float* __restrict__ scores, int64_t lds,
                                                                     int Vloc, int v_begin,
                                                                     const int32_t* __restrict__ gold_indptr,
                                                                     const int32_t* __restrict__ gold_indices,
                                                                     const float* __restrict__ zg,
                                                                     int32_t* __restrict__ cnt,
                                                                     const int32_t* __restrict__ ids) {
  rank_count_body<true>(scores, lds, Vloc, v_begin, gold_indptr, gold_indices, zg, cnt, ids, threadIdx.x);
}

}  // namespace aae

using namespace aae;

template <bool FILT = false>
static int launch_row_topk(const float* scores, int64_t lds, int B, int n, int k, int idx_offset,
                           const int32_t* idx_map, int32_t* idx_out, float* val_out, cudaStream_t s,
                           const int32_t* n_valid = nullptr, int skip_upto = -1, const int32_t* ids = nullptr) {
  size_t smem = sizeof(unsigned long long) * (TK_CAP + TK_SAMPLE);
  cudaError_t e = cudaFuncSetAttribute(row_topk_kernel<FILT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) {
    set_error("row_topk: %s", cudaGetErrorString(e));
    return AAE_E_CUDA;
  }
  row_topk_kernel<FILT><<<B, TK_THREADS, smem, s>>>(scores, lds, n, k, idx_offset, idx_map, n_valid, skip_upto, idx_out,
                                                    val_out, ids);
  return check_launch("row_topk");
}

static bool filter_active(const aae_rank_filter* f) { return f && (f->item_ids || f->excl_indptr); }

// Arguments every *_filtered entry point checks: the exclusion CSR comes whole, and a column table implies v_begin 0
// (the ranked matrix is the compact copy of aae_gather_item_rows).
static int check_filter(const aae_rank_filter* f, int v_begin, const char* fn) {
  if ((f->excl_indptr == nullptr) != (f->excl_indices == nullptr)) {
    set_error("%s: excl_indptr and excl_indices go together", fn);
    return AAE_E_ARG;
  }
  if (f->item_ids && v_begin != 0) {
    set_error("%s: a column table (item_ids) ranks a compact matrix: v_begin must be 0", fn);
    return AAE_E_ARG;
  }
  return AAE_OK;
}

extern "C" {

int aae_masked_topk(float* scores, int64_t lds, int B, int Vloc, int v_begin, const int32_t* indptr,
                    const int32_t* indices, int k, int32_t* idx_out, float* val_out, void* work, void* stream) {
  AAE_REQUIRE(scores && idx_out, "null pointer");
  AAE_REQUIRE(k > 0 && k <= TK_CAP / 2, "k outside the supported envelope (1..4096)");
  AAE_REQUIRE(B > 0 && Vloc > 0, "bad size");
  if (indptr && indices) {
    mask_known_kernel<<<std::min(4 * sm_count(), std::max(1, cdiv((int64_t)B * 32, 256))), 256, 0, as_stream(stream)>>>(
        scores, lds, B, Vloc, v_begin, indptr, indices);
    int rc = check_launch("mask_known");
    if (rc) return rc;
  }
  return launch_row_topk(scores, lds, B, Vloc, k, v_begin, nullptr, idx_out, val_out, as_stream(stream));
}

int aae_masked_topk_filtered(float* scores, int64_t lds, int B, int Vloc, int v_begin, const int32_t* indptr,
                             const int32_t* indices, int k, int32_t* idx_out, float* val_out, void* work, void* stream,
                             const aae_rank_filter* filt) {
  if (!filter_active(filt))
    return aae_masked_topk(scores, lds, B, Vloc, v_begin, indptr, indices, k, idx_out, val_out, work, stream);
  AAE_REQUIRE(scores && idx_out, "null pointer");
  AAE_REQUIRE(k > 0 && k <= TK_CAP / 2, "k outside the supported envelope (1..4096)");
  AAE_REQUIRE(B > 0 && Vloc > 0, "bad size");
  int rc = check_filter(filt, v_begin, __func__);
  if (rc) return rc;
  cudaStream_t s = as_stream(stream);
  const int grid = std::min(4 * sm_count(), std::max(1, cdiv((int64_t)B * 32, 256)));
  if (indptr && indices) {
    mask_cols_kernel<<<grid, 256, 0, s>>>(scores, lds, B, Vloc, v_begin, filt->item_ids, indptr, indices, -FLT_MAX);
    rc = check_launch("mask_cols(known)");
    if (rc) return rc;
  }
  if (filt->excl_indptr) {
    mask_cols_kernel<<<grid, 256, 0, s>>>(scores, lds, B, Vloc, v_begin, filt->item_ids, filt->excl_indptr,
                                          filt->excl_indices, -INFINITY);
    rc = check_launch("mask_cols(exclude)");
    if (rc) return rc;
  }
  return launch_row_topk<true>(scores, lds, B, Vloc, k, v_begin, nullptr, idx_out, val_out, s, nullptr, -1,
                               filt->item_ids);
}

int aae_gather_item_rows(const float* Wd3, const float* bd3, int H, int Vloc, int v_begin, const int32_t* item_ids,
                         int A, float* Wd3c, float* bd3c, int32_t* n_bad, void* stream) {
  AAE_REQUIRE(Wd3 && bd3 && item_ids && Wd3c && bd3c && n_bad, "null pointer");
  AAE_REQUIRE(H > 0 && Vloc > 0 && A > 0, "bad size");
  AAE_REQUIRE((H & 3) != 0 || ((reinterpret_cast<uintptr_t>(Wd3) | reinterpret_cast<uintptr_t>(Wd3c)) & 15) == 0,
              "Wd3 and Wd3c must be 16-byte aligned");
  cudaStream_t s = as_stream(stream);
  cudaMemsetAsync(n_bad, 0, sizeof(int32_t), s);
  gather_item_rows_kernel<<<std::min(8 * sm_count(), std::max(1, cdiv((int64_t)A * 32, 256))), 256, 0, s>>>(
      Wd3, bd3, H, Vloc, v_begin, item_ids, A, Wd3c, bd3c, n_bad);
  return check_launch("gather_item_rows");
}

int aae_rank_counts(float* scores, int64_t lds, int B, int Vloc, int v_begin, const int32_t* indptr,
                    const int32_t* indices, const int32_t* gold_indptr, const int32_t* gold_indices, int n_gold,
                    float* gold_scores, int gold_scores_given, int32_t* counts, void* stream) {
  AAE_REQUIRE(scores && gold_indptr && gold_indices && gold_scores && counts, "null pointer");
  AAE_REQUIRE(B > 0 && Vloc > 0 && n_gold >= 0 && lds >= Vloc, "bad size");
  cudaStream_t s = as_stream(stream);
  if (indptr && indices) {
    mask_known_kernel<<<std::min(4 * sm_count(), std::max(1, cdiv((int64_t)B * 32, 256))), 256, 0, s>>>(
        scores, lds, B, Vloc, v_begin, indptr, indices);
    int rc = check_launch("mask_known");
    if (rc) return rc;
  }
  if (n_gold == 0) return AAE_OK;
  cudaMemsetAsync(counts, 0, sizeof(int32_t) * (size_t)n_gold, s);
  if (!gold_scores_given)
    gold_scores_kernel<<<std::min(4 * sm_count(), std::max(1, cdiv(n_gold, 256))), 256, 0, s>>>(
        scores, lds, B, Vloc, v_begin, gold_indptr, gold_indices, gold_scores);
  dim3 grid((unsigned)cdiv(Vloc, RC_CHUNK), (unsigned)B);
  rank_count_kernel<<<grid, RC_THREADS, 0, s>>>(scores, lds, Vloc, v_begin, gold_indptr, gold_indices, gold_scores,
                                                counts);
  return check_launch("rank_count");
}

int aae_rank_counts_filtered(float* scores, int64_t lds, int B, int Vloc, int v_begin, const int32_t* indptr,
                             const int32_t* indices, const int32_t* gold_indptr, const int32_t* gold_indices,
                             int n_gold, float* gold_scores, int gold_scores_given, int32_t* counts, void* stream,
                             const aae_rank_filter* filt) {
  if (!filter_active(filt))
    return aae_rank_counts(scores, lds, B, Vloc, v_begin, indptr, indices, gold_indptr, gold_indices, n_gold,
                           gold_scores, gold_scores_given, counts, stream);
  AAE_REQUIRE(scores && gold_indptr && gold_indices && gold_scores && counts, "null pointer");
  AAE_REQUIRE(B > 0 && Vloc > 0 && n_gold >= 0 && lds >= Vloc, "bad size");
  int rc = check_filter(filt, v_begin, __func__);
  if (rc) return rc;
  cudaStream_t s = as_stream(stream);
  const int grid = std::min(4 * sm_count(), std::max(1, cdiv((int64_t)B * 32, 256)));
  if (indptr && indices) {
    mask_cols_kernel<<<grid, 256, 0, s>>>(scores, lds, B, Vloc, v_begin, filt->item_ids, indptr, indices, -FLT_MAX);
    rc = check_launch("mask_cols(known)");
    if (rc) return rc;
  }
  // excluded entries at -inf never rank before a returnable gold, whose score is finite (-FLT_MAX when known)
  if (filt->excl_indptr) {
    mask_cols_kernel<<<grid, 256, 0, s>>>(scores, lds, B, Vloc, v_begin, filt->item_ids, filt->excl_indptr,
                                          filt->excl_indices, -INFINITY);
    rc = check_launch("mask_cols(exclude)");
    if (rc) return rc;
  }
  if (n_gold == 0) return AAE_OK;
  cudaMemsetAsync(counts, 0, sizeof(int32_t) * (size_t)n_gold, s);
  if (!gold_scores_given)
    gold_scores_filt_kernel<<<std::min(4 * sm_count(), std::max(1, cdiv(n_gold, 256))), 256, 0, s>>>(
        scores, lds, B, Vloc, v_begin, gold_indptr, gold_indices, gold_scores, filt->item_ids);
  dim3 rgrid((unsigned)cdiv(Vloc, RC_CHUNK), (unsigned)B);
  rank_count_filt_kernel<<<rgrid, RC_THREADS, 0, s>>>(scores, lds, Vloc, v_begin, gold_indptr, gold_indices,
                                                      gold_scores, counts, filt->item_ids);
  return check_launch("rank_count");
}

int64_t aae_predict_topk_work_bytes(int B, int Vloc, int k) {
  if (B <= 0 || Vloc <= 0 || k <= 0) return 0;
  TopkPlan p = make_plan(B, Vloc, k);
  if (!p.ok) return 0;
  return (int64_t)(al256((size_t)B * p.S * 4) + 2 * al256((size_t)B * p.J * 4) + al256((size_t)B * p.nsub * 4) +
                   al256((size_t)B * 4) + 2 * al256((size_t)B * p.nsub * p.cap_sub * 4) +
                   2 * al256((size_t)B * p.cap * 4));
}

static int predict_topk_impl(const float* h2, int B, int H, const float* Wd3, const float* bd3, int Vloc, int v_begin,
                             const int32_t* indptr, const int32_t* indices, int k, int impl, void* work,
                             int64_t work_bytes, int32_t* idx_out, float* val_out, int32_t* n_bad, void* stream,
                             const aae_rank_filter* filt) {
  AAE_REQUIRE(h2 && Wd3 && bd3 && idx_out && n_bad && work, "null pointer");
  AAE_REQUIRE(B > 0 && H > 0 && Vloc > 0 && k > 0, "bad size");
  AAE_REQUIRE((indptr == nullptr) == (indices == nullptr), "indptr and indices go together");
  if (impl != 1 && impl != 2) {
    set_error("aae_predict_topk: the fused path runs on the tensor-core kernel (impl 1 or 2), got %d", impl);
    return AAE_E_UNSUPPORTED;
  }
  const TopkPlan p = make_plan(B, Vloc, k);
  if (!p.ok) {
    set_error("aae_predict_topk: shard of %d items / k = %d is outside the fused envelope (use the dense path)", Vloc, k);
    return AAE_E_UNSUPPORTED;
  }
  AAE_REQUIRE(work_bytes >= aae_predict_topk_work_bytes(B, Vloc, k), "workspace too small");
  cudaStream_t s = as_stream(stream);
  unsigned char* w = reinterpret_cast<unsigned char*>(work);
  float* samp = reinterpret_cast<float*>(w);        w += al256((size_t)B * p.S * 4);
  float* thr_val = reinterpret_cast<float*>(w);     w += al256((size_t)B * p.J * 4);
  int32_t* thr_idx = reinterpret_cast<int32_t*>(w); w += al256((size_t)B * p.J * 4);
  int32_t* cnt = reinterpret_cast<int32_t*>(w);     w += al256((size_t)B * p.nsub * 4);
  int32_t* tot = reinterpret_cast<int32_t*>(w);     w += al256((size_t)B * 4);
  float* sub_val = reinterpret_cast<float*>(w);     w += al256((size_t)B * p.nsub * p.cap_sub * 4);
  int32_t* sub_idx = reinterpret_cast<int32_t*>(w); w += al256((size_t)B * p.nsub * p.cap_sub * 4);
  float* cand_val = reinterpret_cast<float*>(w);    w += al256((size_t)B * p.cap * 4);
  int32_t* cand_idx = reinterpret_cast<int32_t*>(w);
  const int split = impl == 1 ? 3 : 1;
  // (1) scores of a strided sample of the tiles -> (2) per-row threshold = J-th largest sample score, chosen so that
  // about T of the shard's items pass it -> (3) full pass, candidates appended from the GEMM epilogue -> (4) known
  // items masked, candidates sorted, first k emitted
  int rc = dec_out_select_tc(h2, B, H, Wd3, bd3, Vloc, v_begin, p.stride, p.n_samp, 0, samp, p.S, 1, 0, nullptr, 0,
                             nullptr, nullptr, nullptr, 0, split, s);
  if (rc) return rc;
  const bool kth_fast = p.J <= 256;      // else: exact top-J of the sample (large k on a small shard)
  if (kth_fast) {
    row_kth_approx_kernel<<<B, KTH_THREADS, 0, s>>>(samp, p.S, p.S, p.J, thr_val);
    rc = check_launch("row_kth_approx");
  } else {
    rc = launch_row_topk(samp, p.S, B, p.S, p.J, 0, nullptr, thr_idx, thr_val, s);
  }
  if (rc) return rc;
  cudaMemsetAsync(n_bad, 0, 4, s);
  rc = dec_out_select_tc(h2, B, H, Wd3, bd3, Vloc, v_begin, 1, p.n_tiles, 1, nullptr, 0, 0, 0,
                         kth_fast ? thr_val : thr_val + (p.J - 1), kth_fast ? 1 : p.J, cnt, sub_val, sub_idx, p.cap_sub,
                         split, s);
  if (rc) return rc;
  const int fin_grid = std::min(B, 8 * sm_count());
  const size_t fin_smem = (p.nsub + 1) * sizeof(int);
  const RescoreArgs ra{nullptr, nullptr, nullptr, 0, 0};
  if (filt) {
    const RankFilt rf{filt->item_ids, filt->excl_indptr, filt->excl_indices};
    cand_finish_kernel<false, true><<<fin_grid, FIN_THREADS, fin_smem, s>>>(
        sub_val, sub_idx, cnt, p.nsub, p.cap_sub, cand_val, cand_idx, p.cap, tot, B, std::min(k, Vloc), indptr, indices,
        n_bad, ra, rf);
  } else {
    cand_finish_kernel<false, false><<<fin_grid, FIN_THREADS, fin_smem, s>>>(
        sub_val, sub_idx, cnt, p.nsub, p.cap_sub, cand_val, cand_idx, p.cap, tot, B, std::min(k, Vloc), indptr, indices,
        n_bad, ra, RankFilt{nullptr, nullptr, nullptr});
  }
  rc = check_launch("cand_finish");
  if (rc) return rc;
  if (filt) cand_sort_small_kernel<true><<<B, CS_THREADS, 0, s>>>(cand_val, cand_idx, p.cap, tot, k, idx_out, val_out,
                                                                  filt->item_ids);
  else cand_sort_small_kernel<false><<<B, CS_THREADS, 0, s>>>(cand_val, cand_idx, p.cap, tot, k, idx_out, val_out,
                                                              nullptr);
  rc = check_launch("cand_sort_small");
  if (rc) return rc;
  if (filt)
    return launch_row_topk<true>(cand_val, p.cap, B, p.cap, k, 0, cand_idx, idx_out, val_out, s, tot, CS_CAP,
                                 filt->item_ids);
  return launch_row_topk(cand_val, p.cap, B, p.cap, k, 0, cand_idx, idx_out, val_out, s, tot, CS_CAP);
}

int aae_predict_topk(const float* h2, int B, int H, const float* Wd3, const float* bd3, int Vloc, int v_begin,
                     const int32_t* indptr, const int32_t* indices, int k, int impl, void* work, int64_t work_bytes,
                     int32_t* idx_out, float* val_out, int32_t* n_bad, void* stream) {
  return predict_topk_impl(h2, B, H, Wd3, bd3, Vloc, v_begin, indptr, indices, k, impl, work, work_bytes, idx_out,
                           val_out, n_bad, stream, nullptr);
}

int aae_predict_topk_filtered(const float* h2, int B, int H, const float* Wd3, const float* bd3, int Vloc, int v_begin,
                              const int32_t* indptr, const int32_t* indices, int k, int impl, void* work,
                              int64_t work_bytes, int32_t* idx_out, float* val_out, int32_t* n_bad, void* stream,
                              const aae_rank_filter* filt) {
  if (filter_active(filt)) {
    const int rc = check_filter(filt, v_begin, __func__);
    if (rc) return rc;
  }
  return predict_topk_impl(h2, B, H, Wd3, bd3, Vloc, v_begin, indptr, indices, k, impl, work, work_bytes, idx_out,
                           val_out, n_bad, stream, filter_active(filt) ? filt : nullptr);
}

int64_t aae_predict_topk2_work_bytes(int B, int Vloc, int k, int H) {
  if (B <= 0 || Vloc <= 0 || k <= 0 || !select2_supported(H)) return 0;
  TopkPlan p = make_plan(B, Vloc, k, true);
  if (!p.ok) return 0;
  return (int64_t)(al256((size_t)B * p.S * 4) + 2 * al256((size_t)B * p.J * 4) + al256((size_t)B * p.nsub * 4) +
                   2 * al256((size_t)B * 4) + al256((size_t)B * p.nsub * p.cap_sub * 4) +
                   2 * al256((size_t)B * p.cap * 4) + al256((size_t)B * k * 4));
}

static int predict_topk2_impl(const float* h2, int B, int H, const float* Wd3, const float* bd3, const float* Wp,
                              const float* wmax, int Vloc, int v_begin, const int32_t* indptr, const int32_t* indices,
                              int k, void* work, int64_t work_bytes, int32_t* idx_out, float* val_out, int32_t* n_bad,
                              void* stream, const aae_rank_filter* filt) {
  AAE_REQUIRE(h2 && Wd3 && bd3 && Wp && wmax && idx_out && n_bad && work, "null pointer");
  AAE_REQUIRE(B > 0 && H > 0 && Vloc > 0 && k > 0, "bad size");
  AAE_REQUIRE((indptr == nullptr) == (indices == nullptr), "indptr and indices go together");
  AAE_REQUIRE(select2_supported(H), "n_hidden outside the TMA-fed filter's envelope");
  const TopkPlan p = make_plan(B, Vloc, k, true);
  if (!p.ok) {
    set_error("aae_predict_topk2: shard of %d items / k = %d is outside the fused envelope (use the dense path)", Vloc, k);
    return AAE_E_UNSUPPORTED;
  }
  AAE_REQUIRE(work_bytes >= aae_predict_topk2_work_bytes(B, Vloc, k, H), "workspace too small");
  cudaStream_t s = as_stream(stream);
  unsigned char* w = reinterpret_cast<unsigned char*>(work);
  float* samp = reinterpret_cast<float*>(w);        w += al256((size_t)B * p.S * 4);
  float* thr_val = reinterpret_cast<float*>(w);     w += al256((size_t)B * p.J * 4);
  int32_t* thr_idx = reinterpret_cast<int32_t*>(w); w += al256((size_t)B * p.J * 4);
  int32_t* cnt = reinterpret_cast<int32_t*>(w);     w += al256((size_t)B * p.nsub * 4);
  int32_t* tot = reinterpret_cast<int32_t*>(w);     w += al256((size_t)B * 4);
  float* tau_f = reinterpret_cast<float*>(w);       w += al256((size_t)B * 4);
  int32_t* sub_idx = reinterpret_cast<int32_t*>(w); w += al256((size_t)B * p.nsub * p.cap_sub * 4);
  float* cand_val = reinterpret_cast<float*>(w);    w += al256((size_t)B * p.cap * 4);
  int32_t* cand_idx = reinterpret_cast<int32_t*>(w); w += al256((size_t)B * p.cap * 4);
  float* val_tmp = reinterpret_cast<float*>(w);
  float* vout = val_out ? val_out : val_tmp;
  const int kk = std::min(k, Vloc);
  // (1) approximate (single-pass TF32) scores of a strided sample of the tiles -> (2) per-row threshold tau = J-th
  // largest sample score -> filter threshold tau - margin (rigorous TF32 error bound of the row) -> (3) full
  // TMA-multicast pass, item ids of the logits above the filter threshold appended from the GEMM epilogue -> (4) known
  // items masked, survivors re-scored EXACTLY in fp32, sorted, first k emitted -> (5) rows whose k-th exact score does
  // not clear tau are reported in n_bad
  int rc = dec_out_select2(h2, B, H, Wp, Vloc, v_begin, p.stride, p.n_samp, 0, samp, p.S, 1, nullptr, nullptr, nullptr, 0, s);
  if (rc) return rc;
  const bool kth_fast = p.J <= 256;
  if (kth_fast) {
    row_kth_approx_kernel<<<B, KTH_THREADS, 0, s>>>(samp, p.S, p.S, p.J, thr_val);
    rc = check_launch("row_kth_approx");
  } else {
    rc = launch_row_topk(samp, p.S, B, p.S, p.J, 0, nullptr, thr_idx, thr_val, s);
  }
  if (rc) return rc;
  const float* thr = kth_fast ? thr_val : thr_val + (p.J - 1);
  const int thr_stride = kth_fast ? 1 : p.J;
  tau_margin_kernel<<<cdiv((int64_t)B * 32, 256), 256, 0, s>>>(thr, thr_stride, h2, B, H, wmax, tau_f);
  rc = check_launch("tau_margin");
  if (rc) return rc;
  cudaMemsetAsync(n_bad, 0, 4, s);
  rc = dec_out_select2(h2, B, H, Wp, Vloc, v_begin, 1, p.n_tiles, 1, nullptr, 0, 0, tau_f, cnt, sub_idx, p.cap_sub, s);
  if (rc) return rc;
  const int fin_grid = std::min(B, 8 * sm_count());
  const size_t fin_smem = ((p.nsub + 4) & ~3) * sizeof(int) + H * sizeof(float) + 16;
  const RescoreArgs ra{h2, Wd3, bd3, H, v_begin};
  if (filt) {
    const RankFilt rf{filt->item_ids, filt->excl_indptr, filt->excl_indices};
    cand_finish_kernel<true, true><<<fin_grid, FIN_THREADS, fin_smem, s>>>(
        nullptr, sub_idx, cnt, p.nsub, p.cap_sub, cand_val, cand_idx, p.cap, tot, B, kk, indptr, indices, n_bad, ra, rf);
  } else {
    cand_finish_kernel<true, false><<<fin_grid, FIN_THREADS, fin_smem, s>>>(
        nullptr, sub_idx, cnt, p.nsub, p.cap_sub, cand_val, cand_idx, p.cap, tot, B, kk, indptr, indices, n_bad, ra,
        RankFilt{nullptr, nullptr, nullptr});
  }
  rc = check_launch("cand_finish(rescore)");
  if (rc) return rc;
  if (filt) cand_sort_small_kernel<true><<<B, CS_THREADS, 0, s>>>(cand_val, cand_idx, p.cap, tot, k, idx_out, vout,
                                                                  filt->item_ids);
  else cand_sort_small_kernel<false><<<B, CS_THREADS, 0, s>>>(cand_val, cand_idx, p.cap, tot, k, idx_out, vout, nullptr);
  rc = check_launch("cand_sort_small");
  if (rc) return rc;
  rc = filt ? launch_row_topk<true>(cand_val, p.cap, B, p.cap, k, 0, cand_idx, idx_out, vout, s, tot, CS_CAP,
                                    filt->item_ids)
            : launch_row_topk(cand_val, p.cap, B, p.cap, k, 0, cand_idx, idx_out, vout, s, tot, CS_CAP);
  if (rc) return rc;
  check_kth_kernel<<<cdiv(B, 256), 256, 0, s>>>(vout, k, thr, thr_stride, tot, B, n_bad);
  return check_launch("check_kth");
}

int aae_predict_topk2(const float* h2, int B, int H, const float* Wd3, const float* bd3, const float* Wp,
                      const float* wmax, int Vloc, int v_begin, const int32_t* indptr, const int32_t* indices, int k,
                      void* work, int64_t work_bytes, int32_t* idx_out, float* val_out, int32_t* n_bad, void* stream) {
  return predict_topk2_impl(h2, B, H, Wd3, bd3, Wp, wmax, Vloc, v_begin, indptr, indices, k, work, work_bytes, idx_out,
                            val_out, n_bad, stream, nullptr);
}

int aae_predict_topk2_filtered(const float* h2, int B, int H, const float* Wd3, const float* bd3, const float* Wp,
                               const float* wmax, int Vloc, int v_begin, const int32_t* indptr, const int32_t* indices,
                               int k, void* work, int64_t work_bytes, int32_t* idx_out, float* val_out, int32_t* n_bad,
                               void* stream, const aae_rank_filter* filt) {
  if (filter_active(filt)) {
    const int rc = check_filter(filt, v_begin, __func__);
    if (rc) return rc;
  }
  return predict_topk2_impl(h2, B, H, Wd3, bd3, Wp, wmax, Vloc, v_begin, indptr, indices, k, work, work_bytes, idx_out,
                            val_out, n_bad, stream, filter_active(filt) ? filt : nullptr);
}

int aae_topk_merge_seg(const float* cand_val, const int32_t* cand_idx, int world, int B, int kpad, int k,
                       int32_t* idx_out, float* val_out, void* stream) {
  AAE_REQUIRE(cand_val && cand_idx && idx_out, "null pointer");
  AAE_REQUIRE(world >= 1 && B > 0 && kpad > 0 && k > 0 && k <= world * kpad, "bad size");
  AAE_REQUIRE(world * kpad <= CS_CAP, "more than 2048 candidates per row: use aae_topk_merge");
  seg_merge_small_kernel<<<B, CS_THREADS, 0, as_stream(stream)>>>(cand_val, cand_idx, world, B, kpad, k, idx_out,
                                                                  val_out);
  return check_launch("seg_merge_small");
}

int aae_topk_merge(const float* cand_val, const int32_t* cand_idx, int B, int n_cand, int k, int32_t* idx_out,
                   float* val_out, void* stream) {
  AAE_REQUIRE(cand_val && cand_idx && idx_out, "null pointer");
  AAE_REQUIRE(k > 0 && k <= TK_CAP / 2 && n_cand > 0, "bad size");
  return launch_row_topk(cand_val, n_cand, B, n_cand, k, 0, cand_idx, idx_out, val_out, as_stream(stream));
}

}  // extern "C"
