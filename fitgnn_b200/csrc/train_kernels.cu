// Training-path kernels (SURVEY §8f rank 1: node_train_Gs_GD /root/reference/run.py:177-215, node_train_Gc :26-37; the model
// body network.py:29-35 with F.dropout(p = 0.5) active in train mode, network.py:33):
//   fitgnn_gemm_tn            dW[out, in] = G[R, out]^T · A[R, in]  — the weight gradient of GCNConv.lin / lt1 — on the
//                             tensor cores: a transposing bf16 hi/lo split of both operands (the contraction runs over the
//                             ROWS, so they become the K-major dimension), a batched split-K tcgen05 GEMM, a deterministic
//                             reduction of the per-split partial sums (no atomics)
//   fitgnn_elu_dropout_backward   gz = g ⊙ mask/(1-p) ⊙ ELU'(h)   (the backward of x = dropout(elu(conv(x))))
//   fitgnn_dropout            y = x ⊙ mask/(1-p) with a counter-based Philox4x32-10 mask (same (seed, offset) -> same mask
//                             in forward and backward; nothing is stored)
//   fitgnn_adam_step          one fused Adam step over a flat parameter buffer (torch.optim.Adam semantics, main.py:193-194:
//                             lr 0.01, weight_decay 5e-4 as L2 added to the gradient)
#include <cuda_bf16.h>
#include "common.cuh"

namespace fitgnn {

int gemm_bf16x3(const void* A_hi, const void* A_lo, int64_t lda, const void* W_hi, const void* W_lo, int64_t ldw,
                const float* bias, int64_t M, int K, int N, int act, int head, float* Y, void* Y_lo, int64_t ldy,
                const uint64_t* agg_desc, const float* agg_dinv, const int32_t* row_map, float* const* peers, int n_peers,
                const float* row_scale, int agg_defer_scale, cudaStream_t st, int64_t m_batch_rows, int w_batch_rows,
                int64_t w_rows_total, int in_f16 = 0, int out_f16 = 0, int agg_pre = 0, int a_seg_k0 = 0,
                int a0_cols = 0, const void* A1 = nullptr, int64_t lda1 = 0);

namespace {

// ---------------------------------------------------------------------------------------------- Philox4x32-10
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}
// keep-mask of the 4 consecutive elements [4*quad, 4*quad + 4): element kept with probability 1 - p
__device__ __forceinline__ void dropout_keep4(uint64_t seed, uint64_t offset, int64_t quad, uint32_t thresh, bool (&keep)[4]) {
  const uint64_t c = (uint64_t)quad + offset;
  const uint4 r = philox4x32_10(make_uint4((uint32_t)c, (uint32_t)(c >> 32), 0u, 0u), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  keep[0] = r.x >= thresh; keep[1] = r.y >= thresh; keep[2] = r.z >= thresh; keep[3] = r.w >= thresh;
}
__host__ inline uint32_t drop_threshold(float p) {  // P(u32 < thresh) = p
  const double t = (double)p * 4294967296.0;
  return t >= 4294967295.0 ? 0xffffffffu : (uint32_t)t;
}

// x viewed as rows x cols with pitch ld; element index for the mask = r * cols + c (independent of the pitch)
__global__ void dropout_kernel(const float* __restrict__ x, float* __restrict__ y, int64_t rows, int cols, int64_t ldx, int64_t ldy,
                               uint32_t thresh, float scale, uint64_t seed, uint64_t offset) {
  const int64_t quads = (rows * cols + 3) / 4;
  for (int64_t qd = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; qd < quads; qd += (int64_t)gridDim.x * blockDim.x) {
    bool keep[4];
    dropout_keep4(seed, offset, qd, thresh, keep);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t e = 4 * qd + j;
      if (e < rows * cols) {
        const int64_t r = e / cols;
        const int c = (int)(e - r * cols);
        y[r * ldy + c] = keep[j] ? x[r * ldx + c] * scale : 0.f;
      }
    }
  }
}

// gz = g * (mask / (1 - p)) * (h > 0 ? 1 : h + 1);  h = ELU output before the dropout; p = 0 disables the mask
__global__ void elu_dropout_backward_kernel(const float* __restrict__ g, const float* __restrict__ h, float* __restrict__ gz,
                                            int64_t rows, int cols, int64_t ldg, int64_t ldh, int64_t ldo, int act,
                                            uint32_t thresh, float scale, uint64_t seed, uint64_t offset) {
  const int64_t quads = (rows * cols + 3) / 4;
  for (int64_t qd = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; qd < quads; qd += (int64_t)gridDim.x * blockDim.x) {
    bool keep[4] = {true, true, true, true};
    if (thresh) dropout_keep4(seed, offset, qd, thresh, keep);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t e = 4 * qd + j;
      if (e < rows * cols) {
        const int64_t r = e / cols;
        const int c = (int)(e - r * cols);
        const float hv = h[r * ldh + c];
        const float d = (act == FITGNN_ACT_ELU) ? (hv > 0.f ? 1.f : hv + 1.f) : 1.f;
        gz[r * ldo + c] = keep[j] ? g[r * ldg + c] * scale * d : 0.f;
      }
    }
  }
}

// torch.optim.Adam (amsgrad = False, maximize = False): L2 weight decay folded into the gradient, bias-corrected moments
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                            int64_t n, float lr, float beta1, float beta2, float eps, float wd, float bc1, float bc2_sqrt) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float gi = g[i];
    const float pi = p[i];
    if (wd != 0.f) gi = fmaf(wd, pi, gi);
    const float mi = fmaf(beta1, m[i], (1.f - beta1) * gi);
    const float vi = fmaf(beta2, v[i], (1.f - beta2) * gi * gi);
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = pi - (lr / bc1) * (mi / denom);
  }
}

// ---------------------------------------------------------------------------------------------- dW = G^T · A
// Transposing split: src [R, cols] fp32 (pitch ld) -> bf16 hi/lo planes laid out [S][rows_pad][Ks]:
//   plane[(s * rows_pad + c) * Ks + k] = split(src[s * Ks + k][c])   (zero for source rows >= R and for c >= cols)
// 32 x 32 tiles through shared memory: coalesced 128-byte reads along c, coalesced 64-byte bf16 writes along k.
__global__ void __launch_bounds__(256)
split_transpose_kernel(const float* __restrict__ src, int64_t ld, int64_t R, int cols, int rows_pad, int64_t Ks, int S,
                       __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  __shared__ float tile[32][33];
  const int64_t k_tiles = Ks / 32;  // Ks is a multiple of 64
  const int c_tiles = rows_pad / 32;
  const int64_t tiles = (int64_t)S * k_tiles * c_tiles;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
    const int ct = (int)(t % c_tiles);
    const int64_t kt = (t / c_tiles) % k_tiles;
    const int s = (int)(t / (c_tiles * k_tiles));
    const int64_t r0 = (int64_t)s * Ks + kt * 32;  // first source row of the tile
    const int c0 = ct * 32;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t r = r0 + ty + 8 * j;
      const int c = c0 + tx;
      tile[ty + 8 * j][tx] = (r < R && c < cols) ? __ldg(src + r * ld + c) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = c0 + ty + 8 * j;  // plane row
      const float x = tile[tx][ty + 8 * j];
      const __nv_bfloat16 h = __float2bfloat16_rn(x);
      const int64_t o = ((int64_t)s * rows_pad + c) * Ks + kt * 32 + tx;
      hi[o] = h;
      lo[o] = __float2bfloat16_rn(x - __bfloat162float(h));
    }
    __syncthreads();
  }
}

// dW[o, i] = sum_s part[(s * m_pad + o) * ldp + i]   (fixed summation order: deterministic)
__global__ void reduce_splits_kernel(const float* __restrict__ part, int S, int m_pad, int64_t ldp, int out, int in,
                                     float* __restrict__ dW, int64_t lddw) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)out * in) return;
  const int o = (int)(e / in), i = (int)(e % in);
  float acc = 0.f;
  for (int s = 0; s < S; ++s) acc += part[((int64_t)s * m_pad + o) * ldp + i];
  dW[(int64_t)o * lddw + i] = acc;
}

struct TnPlan {
  int S, m_pad, w_pad, ldp;
  int64_t Ks;
  size_t o_ghi, o_glo, o_ahi, o_alo, o_part, total;
};

TnPlan tn_plan(int64_t R, int out, int in) {
  TnPlan p{};
  p.m_pad = (out + 255) / 256 * 256;
  const int bn = in <= 16 ? 16 : in <= 32 ? 32 : in <= 48 ? 48 : in <= 64 ? 64 : in <= 128 ? 128 : 256;
  p.w_pad = (in + bn - 1) / bn * bn;
  if (p.w_pad % 32) p.w_pad = (p.w_pad + 31) / 32 * 32;
  const int tiles_per_batch = (p.m_pad / (in > 128 ? 256 : 128)) * (p.w_pad / bn);
  const int units = in > 128 ? sm_count() / 2 : sm_count();  // CTA pairs for wide outputs
  int S = (units + tiles_per_batch - 1) / tiles_per_batch;
  const int64_t max_s = (R + 4095) / 4096;  // at least 4096 rows per split
  if (S > max_s) S = (int)max_s;
  if (S < 1) S = 1;
  p.S = S;
  p.Ks = ((R + S - 1) / S + 63) / 64 * 64;
  p.ldp = (in + 3) / 4 * 4;
  Bump b(nullptr, (size_t)1 << 62);
  auto take = [&](size_t bytes) { size_t o = b.off; b.take<char>(bytes); return o; };
  p.o_ghi = take((size_t)S * p.m_pad * p.Ks * 2);
  p.o_glo = take((size_t)S * p.m_pad * p.Ks * 2);
  p.o_ahi = take((size_t)S * p.w_pad * p.Ks * 2);
  p.o_alo = take((size_t)S * p.w_pad * p.Ks * 2);
  p.o_part = take((size_t)S * p.m_pad * p.ldp * 4);
  p.total = b.off + 256;
  return p;
}

}  // namespace
}  // namespace fitgnn

using namespace fitgnn;

extern "C" size_t fitgnn_gemm_tn_workspace_bytes(int64_t R, int out, int in) {
  if (R <= 0 || out <= 0 || in <= 0) return 0;
  return tn_plan(R, out, in).total;
}

extern "C" int fitgnn_gemm_tn(const float* G, int64_t ldg, const float* A, int64_t lda, int64_t R, int out, int in, float* dW,
                              int64_t lddw, void* ws, size_t ws_bytes, void* stream) {
  FG_REQUIRE(G && A && dW && ws && R > 0 && out > 0 && in > 0, FITGNN_EINVAL, "gemm_tn: bad arguments");
  FG_REQUIRE(ldg >= out && lda >= in && lddw >= in, FITGNN_EINVAL, "gemm_tn: leading dimension smaller than the extent");
  FG_REQUIRE(((uintptr_t)ws & 255) == 0, FITGNN_EINVAL, "gemm_tn: workspace must be 256-byte aligned");
  const TnPlan p = tn_plan(R, out, in);
  FG_REQUIRE(ws_bytes >= p.total, FITGNN_EWS, "gemm_tn: workspace needs %zu bytes (got %zu)", p.total, ws_bytes);
  FG_REQUIRE(p.Ks < (1ll << 31) - 64 && (int64_t)p.S * p.m_pad < (1ll << 31) - 256, FITGNN_ERANGE, "gemm_tn: split too large");
  cudaStream_t st = as_stream(stream);
  char* base = static_cast<char*>(ws);
  __nv_bfloat16* ghi = reinterpret_cast<__nv_bfloat16*>(base + p.o_ghi);
  __nv_bfloat16* glo = reinterpret_cast<__nv_bfloat16*>(base + p.o_glo);
  __nv_bfloat16* ahi = reinterpret_cast<__nv_bfloat16*>(base + p.o_ahi);
  __nv_bfloat16* alo = reinterpret_cast<__nv_bfloat16*>(base + p.o_alo);
  float* part = reinterpret_cast<float*>(base + p.o_part);
  const unsigned grid = (unsigned)(sm_count() * 8);
  split_transpose_kernel<<<grid, 256, 0, st>>>(G, ldg, R, out, p.m_pad, p.Ks, p.S, ghi, glo);
  FG_LAUNCH_CHECK();
  split_transpose_kernel<<<grid, 256, 0, st>>>(A, lda, R, in, p.w_pad, p.Ks, p.S, ahi, alo);
  FG_LAUNCH_CHECK();
  FG_TRY(gemm_bf16x3(ghi, glo, p.Ks, ahi, alo, p.Ks, nullptr, (int64_t)p.S * p.m_pad, (int)p.Ks, in, FITGNN_ACT_NONE,
                     FITGNN_HEAD_IDENTITY, part, nullptr, p.ldp, nullptr, nullptr, nullptr, nullptr, 0, nullptr, 0, st, p.m_pad,
                     p.w_pad, (int64_t)p.S * p.w_pad));
  const int64_t n = (int64_t)out * in;
  reduce_splits_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(part, p.S, p.m_pad, p.ldp, out, in, dW, lddw);
  FG_LAUNCH_CHECK();
  return FITGNN_OK;
}

extern "C" int fitgnn_dropout(const float* X, int64_t ldx, int64_t rows, int cols, float p, uint64_t seed, uint64_t offset,
                              float* Y, int64_t ldy, void* stream) {
  FG_REQUIRE(X && Y && rows >= 0 && cols > 0 && ldx >= cols && ldy >= cols, FITGNN_EINVAL, "dropout: bad arguments");
  FG_REQUIRE(p >= 0.f && p < 1.f, FITGNN_EINVAL, "dropout: p must be in [0, 1) (got %f)", (double)p);
  if (rows == 0) return FITGNN_OK;
  const int64_t quads = (rows * cols + 3) / 4;
  const int64_t want = ceil_div(quads, 256);
  const unsigned grid = (unsigned)(want < (int64_t)sm_count() * 16 ? want : (int64_t)sm_count() * 16);
  dropout_kernel<<<grid, 256, 0, as_stream(stream)>>>(X, Y, rows, cols, ldx, ldy, drop_threshold(p), 1.f / (1.f - p), seed, offset);
  FG_LAUNCH_CHECK();
  return FITGNN_OK;
}

extern "C" int fitgnn_elu_dropout_backward(const float* G, int64_t ldg, const float* H, int64_t ldh, int64_t rows, int cols,
                                           int act, float p, uint64_t seed, uint64_t offset, float* GZ, int64_t ldo,
                                           void* stream) {
  FG_REQUIRE(G && H && GZ && rows >= 0 && cols > 0 && ldg >= cols && ldh >= cols && ldo >= cols, FITGNN_EINVAL,
             "elu_dropout_backward: bad arguments");
  FG_REQUIRE(p >= 0.f && p < 1.f, FITGNN_EINVAL, "elu_dropout_backward: p must be in [0, 1)");
  FG_REQUIRE(act == FITGNN_ACT_NONE || act == FITGNN_ACT_ELU, FITGNN_EINVAL, "elu_dropout_backward: unknown act %d", act);
  if (rows == 0) return FITGNN_OK;
  const int64_t quads = (rows * cols + 3) / 4;
  const int64_t want = ceil_div(quads, 256);
  const unsigned grid = (unsigned)(want < (int64_t)sm_count() * 16 ? want : (int64_t)sm_count() * 16);
  elu_dropout_backward_kernel<<<grid, 256, 0, as_stream(stream)>>>(G, H, GZ, rows, cols, ldg, ldh, ldo, act,
                                                                   p > 0.f ? drop_threshold(p) : 0u, 1.f / (1.f - p), seed, offset);
  FG_LAUNCH_CHECK();
  return FITGNN_OK;
}

extern "C" int fitgnn_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                                float beta1, float beta2, float eps, float weight_decay, int64_t step, void* stream) {
  FG_REQUIRE(param && grad && exp_avg && exp_avg_sq && n >= 0 && step >= 1, FITGNN_EINVAL, "adam_step: bad arguments");
  if (n == 0) return FITGNN_OK;
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  const int64_t want = ceil_div(n, 256);
  const unsigned grid = (unsigned)(want < (int64_t)sm_count() * 8 ? want : (int64_t)sm_count() * 8);
  adam_kernel<<<grid, 256, 0, as_stream(stream)>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay,
                                                   (float)bc1, (float)sqrt(bc2));
  FG_LAUNCH_CHECK();
  return FITGNN_OK;
}
