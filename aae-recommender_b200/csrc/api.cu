// C-ABI glue: error reporting, device check and the dispatchers of the decoder output layer.
#include <stdarg.h>
#include <string.h>
#include "dec_out.cuh"

namespace aae {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return AAE_E_CUDA;
  }
  return AAE_OK;
}

int sm_count() {
  // cached per device: a process may drive several GPUs (one engine each)
  static int cache[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  int n = cache[dev];
  if (n == 0) {
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
    cache[dev] = n;
  }
  return n;
}

}  // namespace aae

using namespace aae;

extern "C" {

int aae_version(void) { return 100; }
const char* aae_last_error(void) { return g_err; }

int aae_device_check(int dev) {
  int major = 0, minor = 0;
  cudaError_t e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
  if (e != cudaSuccess) {
    set_error("device_check: %s", cudaGetErrorString(e));
    return AAE_E_CUDA;
  }
  if (major != 10) {
    set_error("device %d is sm_%d%d; libaae_b200 is built for sm_100a only", dev, major, minor);
    return AAE_E_ARCH;
  }
  return AAE_OK;
}

int aae_trace_set(uint64_t* buf) {
  trace_set_bag(reinterpret_cast<unsigned long long*>(buf));
  trace_set_mlp(reinterpret_cast<unsigned long long*>(buf));
  trace_set_tc(reinterpret_cast<unsigned long long*>(buf));
  trace_set_w1b(reinterpret_cast<unsigned long long*>(buf));
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    set_error("trace_set: %s", cudaGetErrorString(e));
    return AAE_E_CUDA;
  }
  return AAE_OK;
}
int aae_trace_slots(void) { return 2 * (int)TR_N; }

int64_t aae_dec_out_train_work_floats(int B, int H, int Vloc, int impl) {
  if (impl != 1 || B <= 0 || H <= 0 || Vloc <= 0) return 0;
  const int rows = tc2_max_rows(H);
  if (rows <= 0 || B <= rows) return 0;
  return (int64_t)Vloc * H + Vloc;
}

int aae_dec_out_train_ws(const float* h2, int B, int H, float* Wd3, float* bd3, float* mW, float* vW, float* mb,
                         float* vb, int v_begin, int Vloc, const int32_t* indptr, const int32_t* indices,
                         double n_total, const aae_step_state* st, float* dh2, double* loss_sum, int impl, float* work,
                         int64_t work_floats, void* stream) {
  AAE_REQUIRE(h2 && Wd3 && bd3 && mW && vW && mb && vb && indptr && indices && st && dh2 && loss_sum, "null pointer");
  AAE_REQUIRE(B > 0 && H > 0 && Vloc > 0 && n_total > 0, "bad size");
  if (impl == 0)
    return dec_out_train_simt(h2, B, H, Wd3, bd3, mW, vW, mb, vb, v_begin, Vloc, indptr, indices, n_total, st, dh2,
                              loss_sum, as_stream(stream));
  if (impl >= 1 && impl <= 4) {   // 1/2: pipelined when the shape allows it; 3/4: the non-pipelined kernel
    if (work && work_floats < aae_dec_out_train_work_floats(B, H, Vloc, impl)) {
      set_error("dec_out_train: gradient scratch of %lld floats is too small", (long long)work_floats);
      return AAE_E_ARG;
    }
    return dec_out_train_tc(h2, B, H, Wd3, bd3, mW, vW, mb, vb, v_begin, Vloc, indptr, indices, n_total, st, dh2,
                            loss_sum, (impl & 1) ? 3 : 1, impl <= 2, work, as_stream(stream));
  }
  set_error("dec_out_train: unknown impl %d", impl);
  return AAE_E_ARG;
}

int aae_dec_out_train(const float* h2, int B, int H, float* Wd3, float* bd3, float* mW, float* vW, float* mb,
                      float* vb, int v_begin, int Vloc, const int32_t* indptr, const int32_t* indices, double n_total,
                      const aae_step_state* st, float* dh2, double* loss_sum, int impl, void* stream) {
  return aae_dec_out_train_ws(h2, B, H, Wd3, bd3, mW, vW, mb, vb, v_begin, Vloc, indptr, indices, n_total, st, dh2,
                              loss_sum, impl, nullptr, 0, stream);
}

int aae_dec_out_scores(const float* h2, int B, int H, const float* Wd3, const float* bd3, int Vloc, int apply_sigmoid,
                       float* out, int64_t ldo, int impl, void* stream) {
  AAE_REQUIRE(h2 && Wd3 && bd3 && out, "null pointer");
  AAE_REQUIRE(B > 0 && H > 0 && Vloc > 0 && ldo >= Vloc, "bad size");
  if (impl == 0) return dec_out_scores_simt(h2, B, H, Wd3, bd3, Vloc, apply_sigmoid, out, ldo, as_stream(stream));
  if (impl >= 1 && impl <= 4)   // 3/4 score as 1/2: the training-only choice of kernel has no counterpart here
    return dec_out_scores_tc(h2, B, H, Wd3, bd3, Vloc, apply_sigmoid, out, ldo, (impl & 1) ? 3 : 1, as_stream(stream));
  set_error("dec_out_scores: unknown impl %d", impl);
  return AAE_E_ARG;
}

}  // extern "C"
