// Host launchers of the decoder output layer, shared between translation units.  Included by the files that define
// them and by the files that call them, so that a signature change fails to compile instead of failing to load.
#pragma once
#include "common.cuh"

namespace aae {

// dec_out_simt.cu: fp32 CUDA-core kernels
int dec_out_train_simt(const float* h2, int B, int H, float* Wd3, float* bd3, float* mW, float* vW, float* mb,
                       float* vb, int v_begin, int Vloc, const int32_t* indptr, const int32_t* indices, double n_total,
                       const aae_step_state* st, float* dh2, double* loss_sum, cudaStream_t s);
int dec_out_scores_simt(const float* h2, int B, int H, const float* Wd3, const float* bd3, int Vloc, int apply_sigmoid,
                        float* out, int64_t ldo, cudaStream_t s);

// dec_out_tc.cu: K3, training on tcgen05 (split 3 = 3xTF32, 1 = single-pass TF32)
int dec_out_train_tc(const float* h2, int B, int H, float* Wd3, float* bd3, float* mW, float* vW, float* mb, float* vb,
                     int v_begin, int Vloc, const int32_t* indptr, const int32_t* indices, double n_total,
                     const aae_step_state* st, float* dh2, double* loss_sum, int split, bool pipelined, float* gwork,
                     cudaStream_t s);
// largest row chunk the pipelined kernel takes for this n_hidden (multiple of 8; 0: shape outside its envelope)
int tc2_max_rows(int H);

// dec_out_select.cu: K5 v1, dense scores and the threshold filter on tcgen05
int dec_out_scores_tc(const float* h2, int B, int H, const float* Wd3, const float* bd3, int Vloc, int apply_sigmoid,
                      float* out, int64_t ldo, int split, cudaStream_t s);
int dec_out_select_tc(const float* h2, int B, int H, const float* Wd3, const float* bd3, int Vloc, int v_begin,
                      int tile_stride, int n_sel, int filter, float* out, int64_t ldo, int out_by_visit,
                      int apply_sigmoid, const float* tau, int tau_stride, int32_t* cnt, float* cand_val,
                      int32_t* cand_idx, int cap, int split, cudaStream_t s);
void dec_out_select_grid(int B, int n_sel, int* gx, int* gy);

// dec_out_select2.cu: K5 v2, the TMA-fed single-pass TF32 filter
int dec_out_select2(const float* h2, int B, int H, const float* Wp, int Vloc, int v_begin, int tile_stride, int n_sel,
                    int filter, float* out, int64_t ldo, int out_by_visit, const float* tau, int32_t* cnt,
                    int32_t* cand_idx, int cap_sub, cudaStream_t s);
void dec_out_select2_grid(int B, int n_sel, int* gx, int* gy);
bool select2_supported(int H);

}  // namespace aae
