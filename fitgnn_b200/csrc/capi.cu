// C-ABI plumbing: error state, version/device queries and the dense-transform dispatcher.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "common.cuh"

namespace fitgnn {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int sm_count() {
  static int cached[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (!cached[dev]) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

static int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return (e && e[0]) ? atoi(e) : dflt;
}
static Tuning& tuning_mut() {
  static Tuning t{env_int("FITGNN_GEMM_WS", 1),   getenv("FITGNN_HEAD_BULK") ? 0 : 1, env_int("FITGNN_AGG_WIDE", 0),
                  env_int("FITGNN_GEMM_WIDE", 0), env_int("FITGNN_GEMM_PAIR", 1), env_int("FITGNN_SM_RESERVE", 0),
                  env_int("FITGNN_GEMM_PAIR_WS", 1), 0, env_int("FITGNN_GEMM_PREFETCH", 0)};
  return t;
}
const Tuning& tuning() { return tuning_mut(); }
static int* tuning_field(const char* name) {
  Tuning& t = tuning_mut();
  if (!name) return nullptr;
  if (!strcmp(name, "gemm_ws")) return &t.gemm_ws;
  if (!strcmp(name, "head_bulk")) return &t.head_bulk;
  if (!strcmp(name, "agg_wide")) return &t.agg_wide;
  if (!strcmp(name, "gemm_wide")) return &t.gemm_wide;
  if (!strcmp(name, "gemm_pair")) return &t.gemm_pair;
  if (!strcmp(name, "sm_reserve")) return &t.sm_reserve;
  if (!strcmp(name, "gemm_pair_ws")) return &t.gemm_pair_ws;
  if (!strcmp(name, "gemm_prefetch")) return &t.gemm_prefetch;
  if (!strcmp(name, "gemm_debug")) return &t.gemm_debug;
  return nullptr;
}

int gemm_fp32(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias, int64_t M, int K, int N,
              int act, float* Y, int64_t ldy, cudaStream_t st);
int row_softmax(float* Y, int64_t ldy, int64_t M, int N, int head, cudaStream_t st);
int gemm_bf16x3(const void* A_hi, const void* A_lo, int64_t lda, const void* W_hi, const void* W_lo, int64_t ldw,
                const float* bias, int64_t M, int K, int N, int act, int head, float* Y, void* Y_lo, int64_t ldy,
                const uint64_t* agg_desc, const float* agg_dinv, const int32_t* row_map, float* const* peers, int n_peers,
                const float* row_scale, int agg_defer_scale, cudaStream_t st, int64_t m_batch_rows = 0, int w_batch_rows = 0,
                int64_t w_rows_total = 0, int in_f16 = 0, int out_f16 = 0, int agg_pre = 0,
                int a_seg_k0 = 0, int a0_cols = 0, const void* A1 = nullptr, int64_t lda1 = 0);

int gcn_layer_fused(const int32_t* rowptr, const int32_t* col, const float* dinv, const float* X, int64_t ldx, int width,
                    const int32_t* src_index, const int32_t* out_rows, int64_t M, const void* W_hi, const void* W_lo,
                    int64_t ldw, const float* bias, int N, int act, float* Y, void* Y_lo, int64_t ldy, cudaStream_t st);

}  // namespace fitgnn

using namespace fitgnn;

extern "C" int fitgnn_abi_version(void) { return FITGNN_ABI_VERSION; }

extern "C" int fitgnn_last_error(char* buf, size_t n) {
  const size_t len = strlen(g_err);
  if (buf && n > 0) {
    const size_t c = len < n - 1 ? len : n - 1;
    memcpy(buf, g_err, c);
    buf[c] = 0;
  }
  return (int)len;
}

extern "C" int fitgnn_tuning_set(const char* name, int value) {
  int* f = tuning_field(name);
  FG_REQUIRE(f, FITGNN_EINVAL, "tuning_set: unknown switch '%s'", name ? name : "(null)");
  *f = value;
  return FITGNN_OK;
}
extern "C" int fitgnn_tuning_get(const char* name, int* value) {
  int* f = tuning_field(name);
  FG_REQUIRE(f && value, FITGNN_EINVAL, "tuning_get: unknown switch '%s'", name ? name : "(null)");
  *value = *f;
  return FITGNN_OK;
}

extern "C" int fitgnn_device_info(int* sm_count, int* cc) {
  int dev = 0;
  FG_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp p;
  FG_CUDA(cudaGetDeviceProperties(&p, dev));
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (cc) *cc = p.major * 10 + p.minor;
  return FITGNN_OK;
}

extern "C" int fitgnn_gemm_rowscale_bias_act_split(int precision, const void* A, const void* A_lo, int64_t lda,
                                                   const void* W, const void* W_lo, int64_t ldw, const float* row_scale,
                                                   const float* bias, int64_t M, int K, int N, int act, int head, void* Yv,
                                                   void* Y_lo, int64_t ldy, void* stream) {
  float* Y = static_cast<float*>(Yv);
  FG_REQUIRE(!row_scale || precision == FITGNN_GEMM_BF16X3, FITGNN_EUNSUP, "gemm: row_scale needs FITGNN_GEMM_BF16X3");
  FG_REQUIRE(A && W && Y && M >= 0 && K > 0 && N > 0, FITGNN_EINVAL, "gemm: bad arguments (M=%lld K=%d N=%d)",
             (long long)M, K, N);
  FG_REQUIRE(lda >= K && ldw >= K && ldy >= N, FITGNN_EINVAL, "gemm: leading dimension smaller than the extent");
  FG_REQUIRE(act == FITGNN_ACT_NONE || act == FITGNN_ACT_ELU, FITGNN_EINVAL, "gemm: unknown act %d", act);
  FG_REQUIRE(head >= FITGNN_HEAD_IDENTITY && head <= FITGNN_HEAD_SOFTMAX, FITGNN_EINVAL, "gemm: unknown head %d", head);
  if (M == 0) return FITGNN_OK;
  cudaStream_t st = as_stream(stream);
  if (precision == FITGNN_GEMM_FP32) {
    FG_REQUIRE(!Y_lo, FITGNN_EUNSUP, "gemm: bf16 hi/lo output planes need FITGNN_GEMM_BF16X3");
    FG_TRY(gemm_fp32(static_cast<const float*>(A), lda, static_cast<const float*>(W), ldw, bias, M, K, N, act, Y, ldy,
                     st));
    return row_softmax(Y, ldy, M, N, head, st);
  }
  if (precision == FITGNN_GEMM_BF16X3) {
    FG_REQUIRE(A_lo && W_lo, FITGNN_EINVAL, "gemm: BF16X3 needs the lo planes");
    return gemm_bf16x3(A, A_lo, lda, W, W_lo, ldw, bias, M, K, N, act, head, Y, Y_lo, ldy, nullptr, nullptr, nullptr, nullptr, 0,
                       row_scale, 0, st);
  }
  set_error("gemm: unknown precision %d", precision);
  return FITGNN_EINVAL;
}

extern "C" int fitgnn_gemm_bias_act_split(int precision, const void* A, const void* A_lo, int64_t lda, const void* W,
                                          const void* W_lo, int64_t ldw, const float* bias, int64_t M, int K, int N,
                                          int act, int head, void* Yv, void* Y_lo, int64_t ldy, void* stream) {
  return fitgnn_gemm_rowscale_bias_act_split(precision, A, A_lo, lda, W, W_lo, ldw, nullptr, bias, M, K, N, act, head, Yv, Y_lo,
                                             ldy, stream);
}

extern "C" int fitgnn_gcn_transform_aggregate(const void* A_hi, const void* A_lo, int64_t lda, const void* W_hi,
                                              const void* W_lo, int64_t ldw, const float* bias, int64_t M, int K, int N,
                                              int act, const uint64_t* agg_desc, const float* dinv, int defer_row_scale,
                                              void* Y, void* Y_lo, int64_t ldy, void* stream) {
  FG_REQUIRE(A_hi && A_lo && W_hi && W_lo && Y && agg_desc && dinv && M >= 0 && K > 0 && N > 0, FITGNN_EINVAL,
             "gcn_transform_aggregate: bad arguments (M=%lld K=%d N=%d)", (long long)M, K, N);
  FG_REQUIRE(lda >= K && ldw >= K && ldy >= N, FITGNN_EINVAL, "gcn_transform_aggregate: leading dimension too small");
  FG_REQUIRE(act == FITGNN_ACT_NONE || act == FITGNN_ACT_ELU, FITGNN_EINVAL, "gcn_transform_aggregate: unknown act %d", act);
  if (M == 0) return FITGNN_OK;
  return gemm_bf16x3(A_hi, A_lo, lda, W_hi, W_lo, ldw, bias, M, K, N, act, FITGNN_HEAD_IDENTITY, static_cast<float*>(Y),
                     Y_lo, ldy, agg_desc, dinv, nullptr, nullptr, 0, nullptr, defer_row_scale, as_stream(stream));
}

extern "C" int fitgnn_gemm_head_rows(const void* A_hi, const void* A_lo, int64_t lda, const void* W_hi, const void* W_lo,
                                     int64_t ldw, const float* bias, int64_t M, int K, int N, int act, int head,
                                     const int32_t* row_map, float* Y, int64_t ldy, void* stream) {
  FG_REQUIRE(A_hi && A_lo && W_hi && W_lo && Y && row_map && M >= 0 && K > 0 && N > 0, FITGNN_EINVAL,
             "gemm_head_rows: bad arguments (M=%lld K=%d N=%d)", (long long)M, K, N);
  FG_REQUIRE(lda >= K && ldw >= K && ldy >= N, FITGNN_EINVAL, "gemm_head_rows: leading dimension too small");
  FG_REQUIRE(act == FITGNN_ACT_NONE || act == FITGNN_ACT_ELU, FITGNN_EINVAL, "gemm_head_rows: unknown act %d", act);
  FG_REQUIRE(head >= FITGNN_HEAD_IDENTITY && head <= FITGNN_HEAD_SOFTMAX, FITGNN_EINVAL, "gemm_head_rows: unknown head %d",
             head);
  if (M == 0) return FITGNN_OK;
  return gemm_bf16x3(A_hi, A_lo, lda, W_hi, W_lo, ldw, bias, M, K, N, act, head, Y, nullptr, ldy, nullptr, nullptr,
                     row_map, nullptr, 0, nullptr, 0, as_stream(stream));
}

extern "C" int fitgnn_gemm_head_rows_peers(const void* A_hi, const void* A_lo, int64_t lda, const void* W_hi,
                                           const void* W_lo, int64_t ldw, const float* bias, int64_t M, int K, int N,
                                           int act, int head, const int32_t* row_map, float* const* host_peer_bases,
                                           int n_peers, int64_t ldy, void* stream) {
  FG_REQUIRE(A_hi && A_lo && W_hi && W_lo && row_map && host_peer_bases && M >= 0 && K > 0 && N > 0, FITGNN_EINVAL,
             "gemm_head_rows_peers: bad arguments (M=%lld K=%d N=%d)", (long long)M, K, N);
  FG_REQUIRE(n_peers >= 1 && n_peers <= 8, FITGNN_EINVAL, "gemm_head_rows_peers: 1..8 peers (got %d)", n_peers);
  for (int p = 0; p < n_peers; ++p)
    FG_REQUIRE(host_peer_bases[p], FITGNN_EINVAL, "gemm_head_rows_peers: peer base %d is null", p);
  FG_REQUIRE(lda >= K && ldw >= K && ldy >= N, FITGNN_EINVAL, "gemm_head_rows_peers: leading dimension too small");
  FG_REQUIRE(act == FITGNN_ACT_NONE || act == FITGNN_ACT_ELU, FITGNN_EINVAL, "gemm_head_rows_peers: unknown act %d", act);
  FG_REQUIRE(head >= FITGNN_HEAD_IDENTITY && head <= FITGNN_HEAD_SOFTMAX, FITGNN_EINVAL,
             "gemm_head_rows_peers: unknown head %d", head);
  if (M == 0) return FITGNN_OK;
  return gemm_bf16x3(A_hi, A_lo, lda, W_hi, W_lo, ldw, bias, M, K, N, act, head, nullptr, nullptr, ldy, nullptr, nullptr,
                     row_map, host_peer_bases, n_peers, nullptr, 0, as_stream(stream));
}

extern "C" int fitgnn_gemm_bias_act(int precision, const void* A, const void* A_lo, int64_t lda, const void* W,
                                    const void* W_lo, int64_t ldw, const float* bias, int64_t M, int K, int N, int act,
                                    int head, float* Y, int64_t ldy, void* stream) {
  return fitgnn_gemm_bias_act_split(precision, A, A_lo, lda, W, W_lo, ldw, bias, M, K, N, act, head, Y, nullptr, ldy,
                                    stream);
}

extern "C" int fitgnn_gcn_layer_fused(const int32_t* rowptr, const int32_t* col, const float* dinv, const float* X,
                                      int64_t ldx, int width, const int32_t* src_index, const int32_t* out_rows,
                                      int64_t n_out, const void* W_hi, const void* W_lo, int64_t ldw, const float* bias,
                                      int N, int act, void* Y, void* Y_lo, int64_t ldy, void* stream) {
  FG_REQUIRE(rowptr && col && dinv && X && W_hi && W_lo && Y && n_out >= 0 && N > 0 && width > 0, FITGNN_EINVAL,
             "gcn_layer_fused: bad arguments");
  FG_REQUIRE(act == FITGNN_ACT_NONE || act == FITGNN_ACT_ELU, FITGNN_EINVAL, "gcn_layer_fused: unknown act %d", act);
  if (n_out == 0) return FITGNN_OK;
  return gcn_layer_fused(rowptr, col, dinv, X, ldx, width, src_index, out_rows, n_out, W_hi, W_lo, ldw, bias, N, act,
                         static_cast<float*>(Y), Y_lo, ldy, as_stream(stream));
}

// ---- FITGNN_GEMM_FP16X2: the A operand is ONE fp16 plane, W an fp16 hi/lo pair (see include/fitgnn.h) ------------------
extern "C" int fitgnn_gemm_f16(const void* A, int64_t lda, const void* W_hi, const void* W_lo, int64_t ldw,
                               const float* row_scale, const float* bias, int64_t M, int K, int N, int act, int head, void* Y,
                               int64_t ldy, int out_f16, const int32_t* row_map, void* stream) {
  FG_REQUIRE(A && W_hi && Y && M >= 0 && K > 0 && N > 0, FITGNN_EINVAL, "gemm_f16: bad arguments (M=%lld K=%d N=%d)",
             (long long)M, K, N);
  FG_REQUIRE(lda >= K && ldw >= K && ldy >= N, FITGNN_EINVAL, "gemm_f16: leading dimension smaller than the extent");
  FG_REQUIRE(act == FITGNN_ACT_NONE || act == FITGNN_ACT_ELU, FITGNN_EINVAL, "gemm_f16: unknown act %d", act);
  FG_REQUIRE(head >= FITGNN_HEAD_IDENTITY && head <= FITGNN_HEAD_SOFTMAX, FITGNN_EINVAL, "gemm_f16: unknown head %d", head);
  if (M == 0) return FITGNN_OK;
  return gemm_bf16x3(A, nullptr, lda, W_hi, W_lo, ldw, bias, M, K, N, act, head, static_cast<float*>(Y), nullptr, ldy, nullptr,
                     nullptr, row_map, nullptr, 0, row_scale, 0, as_stream(stream), 0, 0, 0, 1, out_f16 ? 1 : 0);
}

extern "C" int fitgnn_gemm_f16_2seg(const void* A0, int64_t lda0, int a0_cols, int K0, const void* A1, int64_t lda1,
                                    const void* W_hi, const void* W_lo, int64_t ldw, const float* bias, int64_t M, int K, int N,
                                    int act, void* Y, int64_t ldy, int out_f16, void* stream) {
  FG_REQUIRE(A0 && A1 && W_hi && Y && M >= 0 && K > 0 && N > 0, FITGNN_EINVAL,
             "gemm_f16_2seg: bad arguments (M=%lld K=%d N=%d)", (long long)M, K, N);
  FG_REQUIRE(K0 > 0 && K0 % 64 == 0 && K > K0, FITGNN_EUNSUP,
             "gemm_f16_2seg: K0 (%d) must be a positive multiple of 64 (the k-block) and below K (%d)", K0, K);
  FG_REQUIRE(a0_cols > 0 && a0_cols <= K0, FITGNN_EINVAL, "gemm_f16_2seg: A0 has %d columns, segment 0 is %d wide", a0_cols, K0);
  FG_REQUIRE(lda0 >= a0_cols && lda1 >= K - K0 && ldw >= K && ldy >= N, FITGNN_EINVAL,
             "gemm_f16_2seg: leading dimension smaller than the extent");
  FG_REQUIRE(act == FITGNN_ACT_NONE || act == FITGNN_ACT_ELU, FITGNN_EINVAL, "gemm_f16_2seg: unknown act %d", act);
  if (M == 0) return FITGNN_OK;
  return gemm_bf16x3(A0, nullptr, lda0, W_hi, W_lo, ldw, bias, M, K, N, act, FITGNN_HEAD_IDENTITY, static_cast<float*>(Y), nullptr,
                     ldy, nullptr, nullptr, nullptr, nullptr, 0, nullptr, 0, as_stream(stream), 0, 0, 0, 1, out_f16 ? 1 : 0, 0,
                     K0, a0_cols, A1, lda1);
}

extern "C" int fitgnn_gcn_transform_aggregate_f16(int in_f16, const void* A_hi, const void* A_lo, int64_t lda, const void* W_hi,
                                                  const void* W_lo, int64_t ldw, const float* bias, int64_t M, int K, int N,
                                                  int act, const uint64_t* agg_desc, const float* dinv, int defer_row_scale,
                                                  void* Y, int64_t ldy, void* stream) {
  FG_REQUIRE(A_hi && W_hi && (W_lo || in_f16) && Y && (!agg_desc || dinv) && M >= 0 && K > 0 && N > 0, FITGNN_EINVAL,
             "gcn_transform_aggregate_f16: bad arguments (M=%lld K=%d N=%d)", (long long)M, K, N);
  FG_REQUIRE(in_f16 ? !A_lo : A_lo != nullptr, FITGNN_EINVAL, "gcn_transform_aggregate_f16: A_lo must match in_f16");
  FG_REQUIRE(lda >= K && ldw >= K && ldy >= N, FITGNN_EINVAL, "gcn_transform_aggregate_f16: leading dimension too small");
  FG_REQUIRE(act == FITGNN_ACT_NONE || act == FITGNN_ACT_ELU, FITGNN_EINVAL, "gcn_transform_aggregate_f16: unknown act %d", act);
  if (M == 0) return FITGNN_OK;
  return gemm_bf16x3(A_hi, A_lo, lda, W_hi, W_lo, ldw, bias, M, K, N, act, FITGNN_HEAD_IDENTITY, static_cast<float*>(Y), nullptr,
                     ldy, agg_desc, agg_desc ? dinv : nullptr, nullptr, nullptr, 0, nullptr, agg_desc ? defer_row_scale : 0,
                     as_stream(stream), 0, 0, 0, in_f16 ? 1 : 0, 1);
}

extern "C" int fitgnn_gcn_conv_aligned_f16(const void* A, int64_t lda, const void* W_hi, const void* W_lo, int64_t ldw,
                                           const float* bias, int64_t M, int K, int N, int act, const uint64_t* agg_desc,
                                           const float* dinv, void* Y, int64_t ldy, void* stream) {
  FG_REQUIRE(A && W_hi && Y && agg_desc && dinv && M >= 0 && K > 0 && N > 0, FITGNN_EINVAL,
             "gcn_conv_aligned_f16: bad arguments (M=%lld K=%d N=%d)", (long long)M, K, N);
  FG_REQUIRE(lda >= K && ldw >= K && ldy >= N, FITGNN_EINVAL, "gcn_conv_aligned_f16: leading dimension too small");
  FG_REQUIRE(act == FITGNN_ACT_NONE || act == FITGNN_ACT_ELU, FITGNN_EINVAL, "gcn_conv_aligned_f16: unknown act %d", act);
  if (M == 0) return FITGNN_OK;
  // the trailing dinv[r] of the aggregation rides on the bias add (row_scale = dinv, agg_defer_scale = 1)
  return gemm_bf16x3(A, nullptr, lda, W_hi, W_lo, ldw, bias, M, K, N, act, FITGNN_HEAD_IDENTITY, static_cast<float*>(Y), nullptr,
                     ldy, agg_desc, dinv, nullptr, nullptr, 0, dinv, 1, as_stream(stream), 0, 0, 0, 1, 1, 1);
}

extern "C" int fitgnn_gemm_f16_head_rows_peers(const void* A, int64_t lda, const void* W_hi, const void* W_lo, int64_t ldw,
                                               const float* bias, int64_t M, int K, int N, int act, int head,
                                               const int32_t* row_map, float* const* host_peer_bases, int n_peers, int64_t ldy,
                                               void* stream) {
  FG_REQUIRE(A && W_hi && W_lo && row_map && host_peer_bases && M >= 0 && K > 0 && N > 0, FITGNN_EINVAL,
             "gemm_f16_head_rows_peers: bad arguments (M=%lld K=%d N=%d)", (long long)M, K, N);
  FG_REQUIRE(n_peers >= 1 && n_peers <= 8, FITGNN_EINVAL, "gemm_f16_head_rows_peers: 1..8 peers (got %d)", n_peers);
  for (int p = 0; p < n_peers; ++p)
    FG_REQUIRE(host_peer_bases[p], FITGNN_EINVAL, "gemm_f16_head_rows_peers: peer base %d is null", p);
  FG_REQUIRE(lda >= K && ldw >= K && ldy >= N, FITGNN_EINVAL, "gemm_f16_head_rows_peers: leading dimension too small");
  FG_REQUIRE(act == FITGNN_ACT_NONE || act == FITGNN_ACT_ELU, FITGNN_EINVAL, "gemm_f16_head_rows_peers: unknown act %d", act);
  FG_REQUIRE(head >= FITGNN_HEAD_IDENTITY && head <= FITGNN_HEAD_SOFTMAX, FITGNN_EINVAL,
             "gemm_f16_head_rows_peers: unknown head %d", head);
  if (M == 0) return FITGNN_OK;
  return gemm_bf16x3(A, nullptr, lda, W_hi, W_lo, ldw, bias, M, K, N, act, head, nullptr, nullptr, ldy, nullptr, nullptr, row_map,
                     host_peer_bases, n_peers, nullptr, 0, as_stream(stream), 0, 0, 0, 1, 0);
}
