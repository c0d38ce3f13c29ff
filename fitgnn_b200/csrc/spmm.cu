// Segmented symmetric-normalised SpMM over the packed block-diagonal CSR:
//   Y[i,:] = act( dinv[r] * sum_{e in row r} dinv[col_e] * X[src(col_e), :] + bias ),  r = out_rows[i]
// Replaces gcn_norm + MessagePassing.propagate + bias (+F.elu) inside PyG GCNConv, as called at
// /root/reference/network.py:31-32 (and :60,:90,:126,:161,:197).
//
// HBM-bound gather kernel.  A group of LPR lanes (8, 16 or 32, chosen from the row width) owns one output row
// and every lane keeps NV float4 accumulators, so a 512-wide row is 4 fully coalesced 512-byte LDG.128 requests
// per source row while a 100-wide row uses 8 lanes and a warp works on 4 rows at once.  The packed subgraphs
// have 2-6 entries per row, so the kernel is latency- not bandwidth-limited unless the dependent chain
// rowptr -> col -> dinv/gid -> X rows is hidden: each warp walks a run of consecutive rows and software-pipelines
// it (row info 3 rows ahead, column indices 2 ahead, dinv/gid 1 ahead of the row being gathered), which keeps
// the 16-byte feature gathers of the current row in flight back to back.  Rows of one subgraph are adjacent in
// the pack, so neighbouring warps re-hit each other's source rows in L1/L2 and every source row comes from HBM
// once.  High-degree rows (deg >= hub_deg) are split across the 8 warps of a CTA and reduced through shared
// memory by the hub kernel so one warp never serialises thousands of gathers.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "common.cuh"

namespace fitgnn {

#ifndef FG_SPMM_MINB
#define FG_SPMM_MINB 3  // resident CTAs per SM the pipelined kernel is compiled for (register budget)
#endif
#ifndef FG_SPMM_UNROLL
#define FG_SPMM_UNROLL 2  // edges gathered per inner step (independent 16-byte loads in flight = UNROLL * NV)
#endif
#ifndef FG_SPMM_RPW
#define FG_SPMM_RPW 16  // row steps per warp (length of the software pipeline)
#endif
constexpr int SPMM_WARPS = 8;
constexpr int SPMM_THREADS = SPMM_WARPS * 32;

// branchless ELU (MUFU.EX2 path), absolute error <= ~2e-7
__device__ __forceinline__ float elu1(float x) { return elu_fast(x); }

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
// I/O modes of the gather kernels: 0 = fp32 rows in, fp32 out; 1 = fp32 in, bf16 hi/lo planes out; 2 = ONE fp16 plane in and
// out (the hidden state of FITGNN_GEMM_FP16X2: half the gathered bytes; accumulation stays fp32).  ldx / ldy count elements.
constexpr int IO_F32 = 0, IO_SPLIT = 1, IO_F16 = 2;
// four consecutive elements at element offset `off` of a row-major fp32 (or, XH, fp16) matrix
template <bool XH>
__device__ __forceinline__ float4 ldx4(const float* X, int64_t off) {
  if (!XH) return ldg4(X + off);
  const uint2 r = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __half*>(X) + off));
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&r.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
  return make_float4(a.x, a.y, b.x, b.y);
}

__device__ __forceinline__ void fma4(float4& a, float w, const float4& x) {
  a.x = fmaf(w, x.x, a.x);
  a.y = fmaf(w, x.y, a.y);
  a.z = fmaf(w, x.z, a.z);
  a.w = fmaf(w, x.w, a.w);
}

// bf16 hi/lo split of one fp32: hi = rn_bf16(x), lo = rn_bf16(x - hi)
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

template <int SPLIT>
__device__ __forceinline__ void store_row4(void* Y, void* Ylo, int64_t off, float4 v) {
  if (SPLIT == IO_F32) {
    *reinterpret_cast<float4*>(static_cast<float*>(Y) + off) = v;
  } else if (SPLIT == IO_F16) {
    uint2 h;
    h.x = pack_f16x2_rn(v.x, v.y);
    h.y = pack_f16x2_rn(v.z, v.w);
    *reinterpret_cast<uint2*>(static_cast<__half*>(Y) + off) = h;
  } else {
    uint2 h, l;
    split_bf16x2(v.x, v.y, h.x, l.x);
    split_bf16x2(v.z, v.w, h.y, l.y);
    *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(Y) + off) = h;
    *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(Ylo) + off) = l;
  }
}

// One warp accumulates edges [beg, end) of row r for the column block starting at float4 index q0.
template <int NV, bool XH = false>
__device__ __forceinline__ void gather_edges(float4 (&acc)[NV], int beg, int end, const int32_t* __restrict__ col,
                                             const float* __restrict__ dinv, const int32_t* __restrict__ src_index,
                                             const float* __restrict__ X, int64_t ldx, int q0, int nq, int lane) {
  for (int e0 = beg; e0 < end; e0 += 32) {
    const int cnt = min(32, end - e0);
    int c = 0;
    float w = 0.f;
    int64_t s = 0;
    if (lane < cnt) {
      c = __ldg(col + e0 + lane);
      w = __ldg(dinv + c);
      s = src_index ? (int64_t)__ldg(src_index + c) : (int64_t)c;
    }
    const int64_t soff = s * ldx;
    int j = 0;
    for (; j + 4 <= cnt; j += 4) {
      float wj[4];
      int64_t pj[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        wj[u] = __shfl_sync(0xffffffffu, w, j + u);
        pj[u] = __shfl_sync(0xffffffffu, soff, j + u);
      }
      float4 x[4][NV];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          const int q = q0 + lane + 32 * v;
          x[u][v] = (q < nq) ? ldx4<XH>(X, pj[u] + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < NV; ++v) fma4(acc[v], wj[u], x[u][v]);
    }
    for (; j < cnt; ++j) {
      const float wj = __shfl_sync(0xffffffffu, w, j);
      const int64_t pj = __shfl_sync(0xffffffffu, soff, j);
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const int q = q0 + lane + 32 * v;
        if (q < nq) fma4(acc[v], wj, ldx4<XH>(X, pj + 4 * q));
      }
    }
  }
}

template <int NV, int SPLIT>
__device__ __forceinline__ void epilogue(const float4 (&acc)[NV], float dr, const float* __restrict__ bias, int act,
                                         void* Y, void* Ylo, int64_t yoff, int q0, int nq, int lane) {
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int q = q0 + lane + 32 * v;
    if (q < nq) {
      float4 o = make_float4(acc[v].x * dr, acc[v].y * dr, acc[v].z * dr, acc[v].w * dr);
      if (bias) {
        const float4 b = ldg4(bias + 4 * q);
        o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
      }
      if (act == FITGNN_ACT_ELU) {
        o.x = elu1(o.x); o.y = elu1(o.y); o.z = elu1(o.z); o.w = elu1(o.w);
      }
      store_row4<SPLIT>(Y, Ylo, yoff + 4 * q, o);
    }
  }
}

// warp-per-row kernel; rows with degree >= hub_deg are skipped when hub_list != nullptr (hub pass owns them)
template <int NV, bool SPLIT>
__global__ void __launch_bounds__(SPMM_THREADS)
spmm_warp_row_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                     const float* __restrict__ dinv, const float* __restrict__ X, int64_t ldx, int nq,
                     const int32_t* __restrict__ src_index, const float* __restrict__ bias, int act,
                     const int32_t* __restrict__ out_rows, int64_t n_out, void* Y, void* Ylo, int64_t ldy,
                     int hub_deg) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * SPMM_WARPS + (threadIdx.x >> 5);
  if (i >= n_out) return;
  const int r = out_rows ? __ldg(out_rows + i) : (int)i;
  const int beg = __ldg(rowptr + r), end = __ldg(rowptr + r + 1);
  if (end - beg >= hub_deg) return;
  const float dr = __ldg(dinv + r);
  for (int q0 = 0; q0 < nq; q0 += 32 * NV) {
    float4 acc[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    gather_edges<NV>(acc, beg, end, col, dinv, src_index, X, ldx, q0, nq, lane);
    epilogue<NV, SPLIT>(acc, dr, bias, act, Y, Ylo, i * ldy, q0, nq, lane);
  }
}


// ---------------------------------------------------------------------------------------------------------
// software-pipelined kernel: LPR lanes per row, G = 32 / LPR rows per warp per step, rows_per_warp steps
// ---------------------------------------------------------------------------------------------------------
struct RowInfo {
  int beg, end;  // CSR range (end = beg for rows this warp must not gather)
  float dr;
  bool live;     // this warp writes the row (false: out of range, or a hub row the hub kernel owns)
};

// A lane's unit of work is one GROUP of a row: 4 fp32 (one 16-byte load, one float4 accumulator) or, on the fp16 plane, 8
// halfs (one 16-byte load, two float4 accumulators) — the same number of load instructions moves half the bytes, and a
// 512-wide row takes 2 loads per lane instead of 4.  nq counts groups; NV = groups per lane and column block.
template <bool F16>
struct Grp {
  float4 v[F16 ? 2 : 1];
};
template <bool F16>
__device__ __forceinline__ Grp<F16> grp_zero() {
  Grp<F16> g;
#pragma unroll
  for (int i = 0; i < (F16 ? 2 : 1); ++i) g.v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  return g;
}
template <bool F16>
__device__ __forceinline__ Grp<F16> grp_load(const float* X, int64_t off) {  // off: element offset of the group
  Grp<F16> g;
  if (!F16) {
    g.v[0] = ldg4(X + off);
  } else {
    const uint4 r = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(X) + off));
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&r.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
    const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&r.z));
    const float2 d = __half22float2(*reinterpret_cast<const __half2*>(&r.w));
    g.v[0] = make_float4(a.x, a.y, b.x, b.y);
    g.v[F16 ? 1 : 0] = make_float4(c.x, c.y, d.x, d.y);
  }
  return g;
}

template <int NV, int LPR, int SPLIT>
__global__ void __launch_bounds__(SPMM_THREADS, FG_SPMM_MINB)
spmm_pipe_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ dinv,
                 const float* __restrict__ X, int64_t ldx, int nq, const int32_t* __restrict__ src_index,
                 const float* __restrict__ bias, int act, const int32_t* __restrict__ out_rows, int64_t n_out, void* Y,
                 void* Ylo, int64_t ldy, int hub_deg, int rows_per_warp) {
  constexpr int G = 32 / LPR;
  constexpr unsigned FULL = 0xffffffffu;
  constexpr bool F16 = SPLIT == IO_F16;
  constexpr int EPG = F16 ? 8 : 4;  // elements per group
  constexpr int W4 = F16 ? 2 : 1;   // float4 accumulators per group
  const int lane = threadIdx.x & 31;
  const int sub = lane & (LPR - 1);
  const int grp = lane / LPR;
  const int64_t warp_global = (int64_t)blockIdx.x * SPMM_WARPS + (threadIdx.x >> 5);
  const int64_t i_base = warp_global * rows_per_warp * G + grp;
  if (warp_global * rows_per_warp * G >= n_out) return;

  auto load_info = [&](int step) {
    RowInfo ri{0, 0, 0.f, false};
    const int64_t i = i_base + (int64_t)step * G;
    if (step < rows_per_warp && i < n_out) {
      const int r = out_rows ? __ldg(out_rows + i) : (int)i;
      ri.beg = __ldg(rowptr + r);
      ri.end = __ldg(rowptr + r + 1);
      ri.dr = __ldg(dinv + r);
      ri.live = true;
      if (ri.end - ri.beg >= hub_deg) {  // the hub kernel owns this row
        ri.end = ri.beg;
        ri.live = false;
      }
    }
    return ri;
  };
  auto load_col = [&](const RowInfo& ri, int e0) { return (e0 + sub < ri.end) ? __ldg(col + e0 + sub) : -1; };
  auto load_w = [&](int c) { return c >= 0 ? __ldg(dinv + c) : 0.f; };
  auto load_s = [&](int c) { return c >= 0 ? (src_index ? __ldg(src_index + c) : c) : 0; };

  // gather up to LPR edges (one per sub-lane: weight w, source row s) into acc for the column block at q0
  auto gather_chunk = [&](Grp<F16> (&acc)[NV], int cnt, float w, int s, int q0) {
    const int maxcnt = __reduce_max_sync(FULL, cnt);
    constexpr int U = FG_SPMM_UNROLL;
    for (int j = 0; j < maxcnt; j += U) {
      float wj[U];
      int64_t pj[U];
      bool on[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        wj[u] = __shfl_sync(FULL, w, j + u, LPR);
        const int sj = __shfl_sync(FULL, s, j + u, LPR);
        pj[u] = (int64_t)sj * ldx;
        on[u] = j + u < cnt;
      }
      Grp<F16> x[U][NV];
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          const int q = q0 + sub + LPR * v;
          x[u][v] = (on[u] && q < nq) ? grp_load<F16>(X, pj[u] + EPG * q) : grp_zero<F16>();
        }
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int v = 0; v < NV; ++v)
#pragma unroll
          for (int h = 0; h < W4; ++h) fma4(acc[v].v[h], wj[u], x[u][v].v[h]);
    }
  };

  RowInfo ia = load_info(0), ib = load_info(1), ic = load_info(2);
  int ca = load_col(ia, ia.beg), cb = load_col(ib, ib.beg);
  float wa = load_w(ca);
  int sa = load_s(ca);
  for (int step = 0; step < rows_per_warp; ++step) {
    // prefetch: row info 3 steps ahead, column indices 2 ahead, weights / source rows 1 ahead
    const RowInfo id = load_info(step + 3);
    const int cc = load_col(ic, ic.beg);
    const float wb = load_w(cb);
    const int sb = load_s(cb);

    const int64_t i = i_base + (int64_t)step * G;
    const int deg = ia.end - ia.beg;
    const bool long_row = deg > LPR;
    for (int q0 = 0; q0 < nq; q0 += LPR * NV) {
      Grp<F16> acc[NV];
#pragma unroll
      for (int v = 0; v < NV; ++v) acc[v] = grp_zero<F16>();
      gather_chunk(acc, min(deg, LPR), wa, sa, q0);
      for (int e0 = ia.beg + LPR; __any_sync(FULL, long_row && e0 < ia.end); e0 += LPR) {
        const int c = (long_row) ? load_col(ia, e0) : -1;
        gather_chunk(acc, long_row ? max(0, min(ia.end - e0, LPR)) : 0, load_w(c), load_s(c), q0);
      }
      if (ia.live) {  // empty rows (the padding rows of a group-aligned pack) are written too: act(bias), i.e. zeros
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          const int q = q0 + sub + LPR * v;
          if (q < nq) {
            float4 o[W4];
#pragma unroll
            for (int h = 0; h < W4; ++h) {
              const float4 a = acc[v].v[h];
              o[h] = make_float4(a.x * ia.dr, a.y * ia.dr, a.z * ia.dr, a.w * ia.dr);
              if (bias) {
                const float4 b = ldg4(bias + EPG * q + 4 * h);
                o[h].x += b.x; o[h].y += b.y; o[h].z += b.z; o[h].w += b.w;
              }
              if (act == FITGNN_ACT_ELU) {
                o[h].x = elu1(o[h].x); o[h].y = elu1(o[h].y); o[h].z = elu1(o[h].z); o[h].w = elu1(o[h].w);
              }
            }
            if (F16) {
              uint4 pk;
              pk.x = pack_f16x2_rn(o[0].x, o[0].y);
              pk.y = pack_f16x2_rn(o[0].z, o[0].w);
              pk.z = pack_f16x2_rn(o[W4 - 1].x, o[W4 - 1].y);
              pk.w = pack_f16x2_rn(o[W4 - 1].z, o[W4 - 1].w);
              *reinterpret_cast<uint4*>(static_cast<__half*>(Y) + i * ldy + EPG * q) = pk;
            } else {
              store_row4<SPLIT>(Y, Ylo, i * ldy + 4 * q, o[0]);
            }
          }
        }
      }
    }
    ia = ib; ib = ic; ic = id;
    ca = cb; cb = cc;
    wa = wb; sa = sb;
  }
}

// hub rows: one CTA per row, the 8 warps take interleaved 32-edge chunks, partial sums are
// reduced through shared memory (NV*128 floats per warp) by warp 0.
template <int NV, int SPLIT>
__global__ void __launch_bounds__(SPMM_THREADS)
spmm_hub_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ dinv,
                const float* __restrict__ X, int64_t ldx, int nq, const int32_t* __restrict__ src_index,
                const float* __restrict__ bias, int act, const int32_t* __restrict__ out_rows,
                const int32_t* __restrict__ hub_list, int n_hub, const int32_t* __restrict__ hub_count_dev, void* Y,
                void* Ylo, int64_t ldy) {
  __shared__ float4 part[SPMM_WARPS][NV][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  // the number of hub rows is either known on the host (n_hub) or lives on the device (hub_count_dev, capped at n_hub:
  // fitgnn_gcn_forward finds the hubs and launches this kernel without a host round trip)
  const int n_list = hub_count_dev ? min(__ldg(hub_count_dev), n_hub) : n_hub;
  for (int hb = blockIdx.x; hb < n_list; hb += gridDim.x) {
  const int64_t i = __ldg(hub_list + hb);
  const int r = out_rows ? __ldg(out_rows + i) : (int)i;
  const int beg = __ldg(rowptr + r), end = __ldg(rowptr + r + 1);
  const float dr = __ldg(dinv + r);
  for (int q0 = 0; q0 < nq; q0 += 32 * NV) {
    float4 acc[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int e0 = beg + 32 * w; e0 < end; e0 += 32 * SPMM_WARPS)
      gather_edges<NV, SPLIT == IO_F16>(acc, e0, min(e0 + 32, end), col, dinv, src_index, X, ldx, q0, nq, lane);
#pragma unroll
    for (int v = 0; v < NV; ++v) part[w][v][lane] = acc[v];
    __syncthreads();
    if (w == 0) {
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        float4 s = part[0][v][lane];
#pragma unroll
        for (int k = 1; k < SPMM_WARPS; ++k) {
          const float4 t = part[k][v][lane];
          s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w;
        }
        acc[v] = s;
      }
      epilogue<NV, SPLIT>(acc, dr, bias, act, Y, Ylo, i * ldy, q0, nq, lane);
    }
    __syncthreads();
  }
  }
}

// ---------------------------------------------------------------------------------------------------------
// group-local aggregation on a GROUP-ALIGNED pack (align.cu): every CSR entry of a row lies inside the row's own
// group of 32 rows.  One warp per group:
//   1. stage the group's 32 source rows in shared memory ONCE (cp.async, 16-byte pieces: a contiguous 12.8 KB
//      stream when the features come pack-ordered, 32 row gathers through gid otherwise) -> HBM sees each byte once
//      (the generic pipelined kernel re-fetches a source row once per referencing row through L1/L2);
//   2. LANE = ROW: each lane keeps the smem offsets and weights dinv[col] of its row's first SG_SLOTS entries in
//      registers and walks the float4 columns; per column one LDS.128 + 4 FFMA per entry, all 32 lanes busy
//      (warp-per-row used 25 of 32 lanes for 100-wide rows and spent ~150 instructions per row on index handling:
//      ncu r1t, 377 M instructions, issue-bound at 20 % occupancy);
//   3. a column's results go back IN PLACE (the 16 bytes of xs[row][q] become the row's bf16 hi/lo quad or fp32
//      float4: column q is dead once every lane has read it), so no second tile is needed;
//   4. copy-out row by row: coalesced 8/16-byte stores.
// Same accumulation order as spmm_pipe_kernel (CSR order, fmaf chain, then dinv[r]) -> bit-identical results.
// ---------------------------------------------------------------------------------------------------------
constexpr int SG_SLOTS = 8;  // CSR entries per row cached in registers; longer rows read the rest from global memory

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}

__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}

// SPLIT: 0 = fp32 rows out, 1 = bf16 hi/lo planes, 2 = ONE fp16 plane (the layer-1 operand of precision 'fp16')
template <int SPLIT>
__global__ void __launch_bounds__(32)
spmm_group_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ dinv,
                  const float* __restrict__ X, int64_t ldx, int nq, const int32_t* __restrict__ src_index,
                  int64_t n_rows, void* Y, void* Ylo, int64_t ldy, int64_t n_groups, int fill_pad, uint32_t pad_hi_bits) {
  extern __shared__ __align__(16) unsigned char sg_smem[];
  float4* xs = reinterpret_cast<float4*>(sg_smem);  // [32][nq]
  const uint32_t xs_u32 = (uint32_t)__cvta_generic_to_shared(xs);
  constexpr unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x;
  const bool contiguous = src_index == nullptr && ldx == 4 * (int64_t)nq;
  for (int64_t g = blockIdx.x; g < n_groups; g += gridDim.x) {
    const int64_t R0 = g * 32;
    const int64_t r = R0 + lane;
    const bool live = r < n_rows;
    const int rows_here = (int)(n_rows - R0 < 32 ? n_rows - R0 : 32);
    const int rp = __ldg(rowptr + (live ? r : n_rows));
    const int deg = live ? __ldg(rowptr + r + 1) - rp : 0;
    const float dr = live ? __ldg(dinv + r) : 0.f;
    // 1. stage the source rows
    if (contiguous) {
      const float* Xg = X + R0 * ldx;
      for (int t = lane; t < rows_here * nq; t += 32) cp_async16(xs + t, Xg + 4 * t);
    } else {
      const int64_t srow = live ? (src_index ? (int64_t)__ldg(src_index + r) : r) : 0;
      for (int i = 0; i < rows_here; ++i) {
        const int64_t s = __shfl_sync(FULL, srow, i);
        if (lane < nq) cp_async16(xs + i * nq + lane, X + s * ldx + 4 * lane);
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    // 2. this lane's row: smem byte addresses + weights of its first entries.  Unused slots point at the lane's own row
    //    with weight 0 (finite * 0 adds nothing; the row's own x is part of its sum anyway), so the slot loop below has
    //    no lane-dependent branch: the first version predicated the LDS + FFMAs on (slot < deg) and the compiler
    //    emitted BSSY/BSYNC/BRA around every slot (ncu r1u: 3,330 instructions per group, 2/3 of them overhead).
    uint32_t addr[SG_SLOTS];
    float w[SG_SLOTS];
#pragma unroll
    for (int s_ = 0; s_ < SG_SLOTS; ++s_) {
      const bool on = s_ < deg;
      const int c = on ? ((__ldg(col + rp + s_) - (int)R0) & 31) : lane;  // precondition: group-aligned pack
      const float wc = __shfl_sync(FULL, dr, c);
      addr[s_] = xs_u32 + (uint32_t)(c * nq) * 16u;
      w[s_] = on ? wc : 0.f;
    }
    const uint32_t mine = xs_u32 + (uint32_t)(lane * nq) * 16u;
    const int maxdeg = __reduce_max_sync(FULL, deg);
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    for (int q = 0; q < nq; ++q) {
      const uint32_t qo = (uint32_t)q * 16u;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int s_ = 0; s_ < SG_SLOTS; ++s_) {
        if (s_ >= maxdeg) break;  // warp-uniform
        fma4(acc, w[s_], lds128(addr[s_] + qo));
      }
      for (int s_ = SG_SLOTS; s_ < maxdeg; ++s_) {  // rows longer than the register cache (rare)
        const bool on = s_ < deg;
        const int c = on ? ((__ldg(col + rp + s_) - (int)R0) & 31) : lane;
        const float wc = __shfl_sync(FULL, dr, c);
        fma4(acc, on ? wc : 0.f, lds128(xs_u32 + (uint32_t)(c * nq) * 16u + qo));
      }
      const float4 o = make_float4(acc.x * dr, acc.y * dr, acc.z * dr, acc.w * dr);
      __syncwarp();  // every lane has read column q
      if (SPLIT == 2) {
        const uint32_t h0 = pack_f16x2_rn(o.x, o.y), h1 = pack_f16x2_rn(o.z, o.w);  // the row's fp16 quad
        asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(mine + qo), "r"(h0), "r"(h1) : "memory");
      } else if (SPLIT == 1) {
        uint4 pk;  // (hi quad, lo quad)
        split_bf16x2(o.x, o.y, pk.x, pk.z);
        split_bf16x2(o.z, o.w, pk.y, pk.w);
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(mine + qo), "r"(pk.x), "r"(pk.y), "r"(pk.z), "r"(pk.w)
                     : "memory");
      } else {
        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(mine + qo), "f"(o.x), "f"(o.y), "f"(o.z), "f"(o.w)
                     : "memory");
      }
    }
    __syncwarp();
    // 4. copy-out
    if (lane < nq) {
      for (int i = 0; i < rows_here; ++i) {
        const float4 v = xs[i * nq + lane];
        const int64_t yo = (R0 + i) * ldy + 4 * lane;
        if (SPLIT == 2) {
          *reinterpret_cast<uint2*>(static_cast<__half*>(Y) + yo) = make_uint2(__float_as_uint(v.x), __float_as_uint(v.y));
        } else if (SPLIT == 1) {
          *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(Y) + yo) =
              make_uint2(__float_as_uint(v.x), __float_as_uint(v.y));
          *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(Ylo) + yo) =
              make_uint2(__float_as_uint(v.z), __float_as_uint(v.w));
        } else {
          *reinterpret_cast<float4*>(static_cast<float*>(Y) + yo) = v;
        }
      }
    } else if (SPLIT == 2 && fill_pad && lane == nq) {
      for (int i = 0; i < rows_here; ++i)
        *reinterpret_cast<uint2*>(static_cast<__half*>(Y) + (R0 + i) * ldy + 4 * lane) = make_uint2(pad_hi_bits, 0u);
    } else if (SPLIT == 1 && fill_pad && lane == nq) {
      // the planes' 4 pad columns [width, ldy): written too, so that every 32-byte sector of the planes is fully written
      // (leaving them out costs a DRAM read-modify-write per row and plane: ncu r1u, +157 MB of reads)
      for (int i = 0; i < rows_here; ++i) {
        const int64_t yo = (R0 + i) * ldy + 4 * lane;
        *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(Y) + yo) = make_uint2(pad_hi_bits, 0u);
        *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(Ylo) + yo) = make_uint2(0u, 0u);
      }
    }
    __syncwarp();  // the next group's staging overwrites xs
  }
}

static size_t spmm_group_smem(int nq) { return (size_t)32 * nq * 16; }

// ---------------------------------------------------------------------------------------------------------
// block-staged aggregation (the "shared-memory staging" of the pack's dense neighbourhoods).
// The pack is block-diagonal: every CSR entry of a row points into the row's own subgraph.  When rows have many
// entries (cluster_node subgraphs: ~25 per row; heavy-tailed subgraphs: 3-4 per row) the pipelined kernel above fetches
// every source row once per ENTRY through L1/L2 — 10^12 bytes of L2 traffic per layer-0 aggregation of the
// ogbn-products-shaped cluster_node pack, which made that kernel the slowest of the forward (ncu/bench r2b: 155 ms at
// 0.58 TB/s algorithmic).  Here a CTA takes a BLOCK of consecutive pack rows that is closed under adjacency (whole
// subgraphs, blk_ptr from the host side), stages the block's source rows — one column slice of them — in shared memory
// ONCE (cp.async, through src_index when the features are de-duplicated), and every row of the block then aggregates
// from shared memory: HBM and L2 see each source row once per slice, the per-entry traffic is LDS.128.
// LPR lanes own a row (16 for 64-column slices of wide rows, 32 for rows up to 128 floats); arithmetic order = CSR
// order, fmaf chain, then dinv[r]: bit-identical to spmm_pipe_kernel.  Blocks larger than the staging capacity take the
// same loop with loads from global memory (correct for any block, just not staged).
// ---------------------------------------------------------------------------------------------------------
constexpr int SB_THREADS = 256;
constexpr int SB_LPR = 8;  // lanes per row: a warp works on 4 rows at once (4 independent accumulation chains)
#ifndef FG_SB_CTAS
#define FG_SB_CTAS 4       // resident CTAs per SM the kernel is compiled for (register cap) and sized for (shared memory)
#endif
constexpr size_t SB_SMEM = (FG_SB_CTAS == 4 ? 56 : 72) * 1024;

// shared memory a staged pass needs: features [rows][wq float4], dinv [rows], row ranges [rows + 1], column indices (u16)
__host__ __device__ inline size_t sb_bytes(int rows, int wq, int n_ent) {
  return (size_t)rows * wq * 16 + 128 /* slack: lanes past wq read (and drop) up to 7 float4 beyond the last row */ +
         (size_t)rows * 4 + (size_t)(rows + 1) * 4 + 16 + (((size_t)n_ent * 2 + 15) & ~(size_t)15);
}

// One staged pass over float4 columns [qa, qa + wq) of the rows [base, base + rows_b): stage features, dinv, row ranges and
// the block-local column indices in shared memory, aggregate every row from there, store.  PV = float4 per lane (wq <= 8 * PV).
template <int PV, bool SPLIT>
__device__ __forceinline__ void sb_staged_pass(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                               const float* __restrict__ dinv, const float* __restrict__ X, int64_t ldx,
                                               const int32_t* __restrict__ src_index, const int32_t* __restrict__ row_order,
                                               int base, int rows_b, int ebase, int n_ent, int qa, int wq,
                                               const float* __restrict__ bias, int act, void* Y, void* Ylo, int64_t ldy,
                                               unsigned char* smem) {
  constexpr int LPR = SB_LPR;
  constexpr unsigned FULL = 0xffffffffu;
  constexpr int GROUPS = SB_THREADS / LPR;
  constexpr int GPW = 32 / LPR;
  float4* xs = reinterpret_cast<float4*>(smem);  // [rows_b][wq]
  float* ds = reinterpret_cast<float*>(smem + (size_t)rows_b * wq * 16 + 128);
  int32_t* rp = reinterpret_cast<int32_t*>(ds + rows_b);  // [rows_b + 1] row ranges relative to ebase
  uint16_t* cs = reinterpret_cast<uint16_t*>(rp + rows_b + 1);
  cs = reinterpret_cast<uint16_t*>(((uintptr_t)cs + 15) & ~(uintptr_t)15);
  const uint32_t xs_u32 = (uint32_t)__cvta_generic_to_shared(xs);
  const uint32_t cs_u32 = (uint32_t)__cvta_generic_to_shared(cs);
  const uint32_t ds_u32 = (uint32_t)__cvta_generic_to_shared(ds);
  const int sub = threadIdx.x & (LPR - 1);
  const int grp = threadIdx.x / LPR;
  const int gw = grp % GPW;
  for (int i = grp; i < rows_b; i += GROUPS) {
    const int64_t srow = src_index ? (int64_t)__ldg(src_index + base + i) : (int64_t)(base + i);
    const float* xr = X + srow * ldx + 4 * qa;
#pragma unroll
    for (int v = 0; v < PV; ++v) {
      const int q = sub + LPR * v;
      if (q < wq) cp_async16(xs + (size_t)i * wq + q, xr + 4 * q);
    }
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  for (int i = threadIdx.x; i < rows_b; i += SB_THREADS) ds[i] = __ldg(dinv + base + i);
  for (int i = threadIdx.x; i <= rows_b; i += SB_THREADS) rp[i] = __ldg(rowptr + base + i) - ebase;
  for (int e = threadIdx.x; e < n_ent; e += SB_THREADS) cs[e] = (uint16_t)(__ldg(col + ebase + e) - base);  // closed block
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  // warp-uniform loop over the block's rows in `row_order` (degree-sorted inside the block, so the 4 rows a warp works on
  // have similar lengths); a group past the last row idles
  for (int k0 = grp - gw; k0 < rows_b; k0 += GROUPS) {
    const int k = k0 + gw;
    const bool live = k < rows_b;
    const int i = live ? (row_order ? __ldg(row_order + base + k) - base : k) : 0;
    const int beg = live ? rp[i] : 0, end = live ? rp[i + 1] : 0;
    const float dr = ds[i];
    const int len = end - beg;
    const int maxlen = __reduce_max_sync(FULL, len);
    float4 acc[PV];
#pragma unroll
    for (int v = 0; v < PV; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    // every lane of a group reads the same (index, weight) from shared memory (broadcast); past the row's end the entry is
    // (row 0, weight 0): a valid, finite row times zero
    for (int j = 0; j < maxlen; j += 2) {
      const bool on0 = j < len, on1 = j + 1 < len;
      uint32_t c0 = 0, c1 = 0;
      float w0 = 0.f, w1 = 0.f;
      if (on0) {
        asm volatile("ld.shared.u16 %0, [%1];" : "=r"(c0) : "r"(cs_u32 + 2u * (uint32_t)(beg + j)));
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(w0) : "r"(ds_u32 + 4u * c0));
      }
      if (on1) {
        asm volatile("ld.shared.u16 %0, [%1];" : "=r"(c1) : "r"(cs_u32 + 2u * (uint32_t)(beg + j + 1)));
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(w1) : "r"(ds_u32 + 4u * c1));
      }
      const uint32_t a0 = xs_u32 + (c0 * (uint32_t)wq + (uint32_t)sub) * 16u;
      const uint32_t a1 = xs_u32 + (c1 * (uint32_t)wq + (uint32_t)sub) * 16u;
      float4 x0[PV], x1[PV];
#pragma unroll
      for (int v = 0; v < PV; ++v) {
        x0[v] = lds128(a0 + (uint32_t)(LPR * v) * 16u);
        x1[v] = lds128(a1 + (uint32_t)(LPR * v) * 16u);
      }
#pragma unroll
      for (int v = 0; v < PV; ++v) fma4(acc[v], w0, x0[v]);
#pragma unroll
      for (int v = 0; v < PV; ++v) fma4(acc[v], w1, x1[v]);
    }
    if (live) {
      const int r = base + i;
#pragma unroll
      for (int v = 0; v < PV; ++v) {
        const int qs = sub + LPR * v;
        if (qs < wq) {
          const int q = qa + qs;
          float4 o = make_float4(acc[v].x * dr, acc[v].y * dr, acc[v].z * dr, acc[v].w * dr);
          if (bias) {
            const float4 bq = ldg4(bias + 4 * q);
            o.x += bq.x; o.y += bq.y; o.z += bq.z; o.w += bq.w;
          }
          if (act == FITGNN_ACT_ELU) {
            o.x = elu1(o.x); o.y = elu1(o.y); o.z = elu1(o.z); o.w = elu1(o.w);
          }
          store_row4<SPLIT>(Y, Ylo, (int64_t)r * ldy + 4 * q, o);
        }
      }
    }
  }
  __syncthreads();  // the next pass / item overwrites the staging area
}

template <bool SPLIT>
__global__ void __launch_bounds__(SB_THREADS, FG_SB_CTAS)
spmm_block_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ dinv,
                  const float* __restrict__ X, int64_t ldx, int nq, const int32_t* __restrict__ src_index,
                  const int32_t* __restrict__ blk_ptr, int64_t n_blk, const int32_t* __restrict__ row_order, int n_slices,
                  const float* __restrict__ bias, int act, void* Y, void* Ylo, int64_t ldy) {
  constexpr int LPR = SB_LPR;
  constexpr int NQS = 32;  // float4 columns per static slice (128 floats)
  extern __shared__ __align__(16) unsigned char sb_smem[];
  constexpr unsigned FULL = 0xffffffffu;
  constexpr int GROUPS = SB_THREADS / LPR;
  constexpr int GPW = 32 / LPR;
  const int sub = threadIdx.x & (LPR - 1);
  const int grp = threadIdx.x / LPR;
  const int gw = grp % GPW;
  const int64_t items = n_blk * n_slices;
  for (int64_t it = blockIdx.x; it < items; it += gridDim.x) {
    const int64_t b = it / n_slices;
    const int sl = (int)(it % n_slices);
    const int base = __ldg(blk_ptr + b);
    const int rows_b = __ldg(blk_ptr + b + 1) - base;
    if (rows_b <= 0) continue;  // CTA-uniform
    const int q0 = sl * NQS;            // first float4 column of this slice
    const int nqs = min(NQS, nq - q0);  // float4 columns in this slice
    const int ebase = __ldg(rowptr + base);
    const int n_ent = __ldg(rowptr + base + rows_b) - ebase;
    // Passes: the fewest column ranges of equal width whose staging fits the shared memory (the CSR part is re-staged per
    // pass: 2 bytes per entry against 16 * width bytes of features per row).  All CTA-uniform.
    int n_pass = 0;
    if (rows_b <= 65535) {
      for (int t = 1; t <= nqs; ++t) {
        const int w = (nqs + t - 1) / t;
        if (sb_bytes(rows_b, w, n_ent) <= SB_SMEM) { n_pass = t; break; }
      }
    }
    if (n_pass != 0) {
      const int w = (nqs + n_pass - 1) / n_pass;
      for (int qa = 0; qa < nqs; qa += w) {
        const int wq = min(w, nqs - qa);
        if (wq > 24) sb_staged_pass<4, SPLIT>(rowptr, col, dinv, X, ldx, src_index, row_order, base, rows_b, ebase, n_ent, q0 + qa, wq, bias, act, Y, Ylo, ldy, sb_smem);
        else if (wq > 16) sb_staged_pass<3, SPLIT>(rowptr, col, dinv, X, ldx, src_index, row_order, base, rows_b, ebase, n_ent, q0 + qa, wq, bias, act, Y, Ylo, ldy, sb_smem);
        else if (wq > 8) sb_staged_pass<2, SPLIT>(rowptr, col, dinv, X, ldx, src_index, row_order, base, rows_b, ebase, n_ent, q0 + qa, wq, bias, act, Y, Ylo, ldy, sb_smem);
        else sb_staged_pass<1, SPLIT>(rowptr, col, dinv, X, ldx, src_index, row_order, base, rows_b, ebase, n_ent, q0 + qa, wq, bias, act, Y, Ylo, ldy, sb_smem);
      }
      continue;
    }
    // block beyond any staging capacity: the same aggregation straight from global memory
    for (int i0 = grp - gw; i0 < rows_b; i0 += GROUPS) {
      const int i = i0 + gw;
      const bool live = i < rows_b;
      const int r = base + (live ? i : 0);
      const int beg = live ? __ldg(rowptr + r) : 0, end = live ? __ldg(rowptr + r + 1) : 0;
      const float dr = __ldg(dinv + r);
      float4 acc[4];
#pragma unroll
      for (int v = 0; v < 4; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int e0 = beg; __any_sync(FULL, e0 < end); e0 += LPR) {
        const bool has = e0 + sub < end;
        const int c = has ? __ldg(col + e0 + sub) : 0;
        const float w = has ? __ldg(dinv + c) : 0.f;
        const int64_t goff = (src_index ? (int64_t)__ldg(src_index + c) : (int64_t)c) * ldx;
        const int cnt = max(0, min(LPR, end - e0));
        const int maxcnt = __reduce_max_sync(FULL, cnt);
        for (int j = 0; j < maxcnt; ++j) {
          const float wj = __shfl_sync(FULL, w, j, LPR);
          const int64_t oj = __shfl_sync(FULL, goff, j, LPR);
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            const int q = sub + LPR * v;
            if (q < nqs) fma4(acc[v], wj, ldg4(X + oj + 4 * (q0 + q)));
          }
        }
      }
      if (live) {
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const int qs = sub + LPR * v;
          if (qs < nqs) {
            const int q = q0 + qs;
            float4 o = make_float4(acc[v].x * dr, acc[v].y * dr, acc[v].z * dr, acc[v].w * dr);
            if (bias) {
              const float4 bq = ldg4(bias + 4 * q);
              o.x += bq.x; o.y += bq.y; o.z += bq.z; o.w += bq.w;
            }
            if (act == FITGNN_ACT_ELU) {
              o.x = elu1(o.x); o.y = elu1(o.y); o.z = elu1(o.z); o.w = elu1(o.w);
            }
            store_row4<SPLIT>(Y, Ylo, (int64_t)r * ldy + 4 * q, o);
          }
        }
      }
    }
  }
}

// hub detection: hub_list[atomic slot] = i for output rows with degree >= hub_deg
__global__ void spmm_find_hubs_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ out_rows,
                                      int64_t n_out, int hub_deg, int32_t* hub_list, int32_t* hub_count,
                                      int hub_cap) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_out) return;
  const int r = out_rows ? out_rows[i] : (int)i;
  if (rowptr[r + 1] - rowptr[r] >= hub_deg) {
    const int slot = atomicAdd(hub_count, 1);
    if (slot < hub_cap) hub_list[slot] = (int32_t)i;
  }
}

template <int NV, int LPR, int SPLIT>
static int launch_spmm(const int32_t* rowptr, const int32_t* col, const float* dinv, const float* X, int64_t ldx,
                       int nq, const int32_t* src_index, const float* bias, int act, const int32_t* out_rows,
                       int64_t n_out, void* Y, void* Ylo, int64_t ldy, const int32_t* hub_list, int n_hub,
                       int hub_deg, cudaStream_t st, const int32_t* hub_count_dev = nullptr) {
  constexpr int G = 32 / LPR;
  // long enough runs per warp for the prefetch pipeline to pay, but keep >= ~4 CTAs per SM on small inputs
  int rpw = FG_SPMM_RPW;
  while (rpw > 1 && ceil_div(n_out, (int64_t)G * rpw * SPMM_WARPS) < (int64_t)sm_count() * 4) rpw >>= 1;
  const int64_t blocks = ceil_div(n_out, (int64_t)G * rpw * SPMM_WARPS);
  // nq counts float4 quads; the fp16 variant of the pipelined kernel works on groups of 8 halfs (the hub kernel on quads)
  spmm_pipe_kernel<NV, LPR, SPLIT><<<(unsigned)blocks, SPMM_THREADS, 0, st>>>(
      rowptr, col, dinv, X, ldx, SPLIT == IO_F16 ? nq / 2 : nq, src_index, bias, act, out_rows, n_out, Y, Ylo, ldy, hub_deg, rpw);
  FG_LAUNCH_CHECK();
  if (n_hub > 0) {
    const unsigned hub_blocks = hub_count_dev ? (unsigned)min((int64_t)n_hub, (int64_t)sm_count() * 4) : (unsigned)n_hub;
    spmm_hub_kernel<4, SPLIT><<<hub_blocks, SPMM_THREADS, 0, st>>>(rowptr, col, dinv, X, ldx, nq, src_index, bias, act, out_rows,
                                                                   hub_list, n_hub, hub_count_dev, Y, Ylo, ldy);
    FG_LAUNCH_CHECK();
  }
  return FITGNN_OK;
}

}  // namespace fitgnn

using namespace fitgnn;

extern "C" int fitgnn_spmm_hubs(const int32_t* rowptr, const int32_t* out_rows, int64_t n_out, int hub_deg,
                                int32_t* hub_list, int32_t* hub_count, int hub_cap, void* stream) {
  FG_REQUIRE(rowptr && hub_list && hub_count && n_out >= 0 && hub_deg > 0, FITGNN_EINVAL, "spmm_hubs: bad arguments");
  cudaStream_t st = as_stream(stream);
  FG_CUDA(cudaMemsetAsync(hub_count, 0, sizeof(int32_t), st));
  if (n_out == 0) return FITGNN_OK;
  spmm_find_hubs_kernel<<<(unsigned)ceil_div(n_out, 256), 256, 0, st>>>(rowptr, out_rows, n_out, hub_deg, hub_list,
                                                                        hub_count, hub_cap);
  FG_LAUNCH_CHECK();
  return FITGNN_OK;
}

static int spmm_dispatch(const int32_t* rowptr, const int32_t* col, const float* dinv, const float* X, int64_t ldx, int width,
                         const int32_t* src_index, const float* bias, int act, const int32_t* out_rows, int64_t n_out, void* Y,
                         void* Y_lo, int64_t ldy, const int32_t* hub_list, int n_hub, int hub_deg,
                         const int32_t* hub_count_dev, void* stream, int f16 = 0);

extern "C" int fitgnn_spmm_symnorm_hub(const int32_t* rowptr, const int32_t* col, const float* dinv, const float* X,
                                       int64_t ldx, int width, const int32_t* src_index, const float* bias, int act,
                                       const int32_t* out_rows, int64_t n_out, void* Y, void* Y_lo, int64_t ldy,
                                       const int32_t* hub_list, int n_hub, int hub_deg, void* stream) {
  return spmm_dispatch(rowptr, col, dinv, X, ldx, width, src_index, bias, act, out_rows, n_out, Y, Y_lo, ldy, hub_list, n_hub,
                       hub_deg, nullptr, stream);
}

// hub list whose length lives on the device (fitgnn_spmm_hubs wrote hub_count): at most hub_cap entries are used; no host sync
extern "C" int fitgnn_spmm_symnorm_devhub(const int32_t* rowptr, const int32_t* col, const float* dinv, const float* X,
                                          int64_t ldx, int width, const int32_t* src_index, const float* bias, int act,
                                          const int32_t* out_rows, int64_t n_out, void* Y, void* Y_lo, int64_t ldy,
                                          const int32_t* hub_list, const int32_t* hub_count, int hub_cap, int hub_deg,
                                          void* stream) {
  FG_REQUIRE(hub_list && hub_count && hub_cap > 0 && hub_deg > 0, FITGNN_EINVAL, "spmm_devhub: bad hub arguments");
  return spmm_dispatch(rowptr, col, dinv, X, ldx, width, src_index, bias, act, out_rows, n_out, Y, Y_lo, ldy, hub_list, hub_cap,
                       hub_deg, hub_count, stream);
}

static int spmm_dispatch(const int32_t* rowptr, const int32_t* col, const float* dinv, const float* X, int64_t ldx, int width,
                         const int32_t* src_index, const float* bias, int act, const int32_t* out_rows, int64_t n_out, void* Y,
                         void* Y_lo, int64_t ldy, const int32_t* hub_list, int n_hub, int hub_deg,
                         const int32_t* hub_count_dev, void* stream, int f16) {
  FG_REQUIRE(rowptr && col && dinv && X && Y, FITGNN_EINVAL, "spmm: null pointer");
  FG_REQUIRE(!f16 || !Y_lo, FITGNN_EINVAL, "spmm: the fp16 variant writes ONE plane (Y_lo must be NULL)");
  FG_REQUIRE(n_out >= 0 && width > 0, FITGNN_EINVAL, "spmm: n_out=%lld width=%d", (long long)n_out, width);
  FG_REQUIRE(width % 4 == 0 && ldx % 4 == 0 && ldy % 4 == 0, FITGNN_EUNSUP,
             "spmm: width (%d), ldx (%lld), ldy (%lld) must be multiples of 4", width, (long long)ldx, (long long)ldy);
  FG_REQUIRE(((uintptr_t)X % 16) == 0 && ((uintptr_t)Y % 8) == 0 && (!bias || ((uintptr_t)bias % 16) == 0),
             FITGNN_EUNSUP, "spmm: X/bias must be 16-byte aligned");
  FG_REQUIRE(act == FITGNN_ACT_NONE || act == FITGNN_ACT_ELU, FITGNN_EINVAL, "spmm: unknown act %d", act);
  FG_REQUIRE(n_hub == 0 || hub_list, FITGNN_EINVAL, "spmm: n_hub without hub_list");
  if (n_out == 0) return FITGNN_OK;
  FG_REQUIRE(ceil_div(n_out, SPMM_WARPS) < (1ll << 31), FITGNN_ERANGE, "spmm: too many rows");
  cudaStream_t st = as_stream(stream);
  const int nq = width / 4;
  const bool split = Y_lo != nullptr;
  if (n_hub == 0) hub_deg = 0x7fffffff;
#define FG_SPMM_IO(NV, LPR, IO)                                                                                            \
  launch_spmm<NV, LPR, IO>(rowptr, col, dinv, X, ldx, nq, src_index, bias, act, out_rows, n_out, Y, Y_lo, ldy, hub_list, \
                           n_hub, hub_deg, st, hub_count_dev)
  if (f16) {  // 16-byte loads of 8 halfs: width, pitches multiples of 8 and 16-byte aligned planes
    FG_REQUIRE(width % 8 == 0 && ldx % 8 == 0 && ldy % 8 == 0 && ((uintptr_t)Y % 16) == 0, FITGNN_EUNSUP,
               "spmm_f16: width (%d), ldx (%lld), ldy (%lld) must be multiples of 8, planes 16-byte aligned", width,
               (long long)ldx, (long long)ldy);
    // (groups per lane NV, lanes per row): 64 halfs -> 8 lanes x 1, 128 -> 8 x 2, 256 -> 16 x 2, 512+ -> 32 x 2 per column block
    if (nq <= 16) return FG_SPMM_IO(1, 8, IO_F16);
    if (nq <= 32) return FG_SPMM_IO(2, 8, IO_F16);
    if (nq <= 64) return FG_SPMM_IO(2, 16, IO_F16);
    return FG_SPMM_IO(2, 32, IO_F16);
  }
#define FG_SPMM(NV, LPR) return split ? FG_SPMM_IO(NV, LPR, IO_SPLIT) : FG_SPMM_IO(NV, LPR, IO_F32)
  if (nq <= 8) { FG_SPMM(1, 8); }
  if (nq <= 16) { FG_SPMM(2, 8); }
  if (nq <= 32) { FG_SPMM(4, 8); }
  if (nq <= 64) { FG_SPMM(4, 16); }
  FG_SPMM(4, 32);  // nq > 128 loops over 512-column blocks
#undef FG_SPMM
#undef FG_SPMM_IO
}

// The same aggregation on the fp16 hidden state of FITGNN_GEMM_FP16X2: X and Y are ONE fp16 plane each (ldx / ldy in
// elements), sums in fp32.  hub_count (device) may be NULL: hub_cap is then the host-known number of hub rows.
extern "C" int fitgnn_spmm_symnorm_f16(const int32_t* rowptr, const int32_t* col, const float* dinv, const void* X,
                                       int64_t ldx, int width, const int32_t* src_index, const float* bias, int act,
                                       const int32_t* out_rows, int64_t n_out, void* Y, int64_t ldy,
                                       const int32_t* hub_list, const int32_t* hub_count, int hub_cap, int hub_deg,
                                       void* stream) {
  return spmm_dispatch(rowptr, col, dinv, static_cast<const float*>(X), ldx, width, src_index, bias, act, out_rows, n_out, Y,
                       nullptr, ldy, hub_list, hub_list ? hub_cap : 0, hub_deg, hub_count, stream, 1);
}

extern "C" int fitgnn_spmm_symnorm(const int32_t* rowptr, const int32_t* col, const float* dinv, const float* X,
                                   int64_t ldx, int width, const int32_t* src_index, const float* bias, int act,
                                   const int32_t* out_rows, int64_t n_out, void* Y, void* Y_lo, int64_t ldy,
                                   void* stream) {
  return fitgnn_spmm_symnorm_hub(rowptr, col, dinv, X, ldx, width, src_index, bias, act, out_rows, n_out, Y, Y_lo,
                                 ldy, nullptr, 0, 0, stream);
}

extern "C" int fitgnn_spmm_symnorm_blocked(const int32_t* rowptr, const int32_t* col, const float* dinv, const float* X,
                                           int64_t ldx, int width, const int32_t* src_index, const int32_t* blk_ptr,
                                           int64_t n_blk, const int32_t* row_order, const float* bias, int act, void* Y,
                                           void* Y_lo, int64_t ldy, void* stream) {
  FG_REQUIRE(rowptr && col && dinv && X && Y && blk_ptr, FITGNN_EINVAL, "spmm_blocked: null pointer");
  FG_REQUIRE(n_blk >= 0 && width > 0, FITGNN_EINVAL, "spmm_blocked: n_blk=%lld width=%d", (long long)n_blk, width);
  FG_REQUIRE(width % 4 == 0 && ldx % 4 == 0 && ldy % 4 == 0, FITGNN_EUNSUP,
             "spmm_blocked: width (%d), ldx (%lld), ldy (%lld) must be multiples of 4", width, (long long)ldx, (long long)ldy);
  FG_REQUIRE(((uintptr_t)X % 16) == 0 && ((uintptr_t)Y % 8) == 0 && (!bias || ((uintptr_t)bias % 16) == 0), FITGNN_EUNSUP,
             "spmm_blocked: X/bias must be 16-byte aligned");
  FG_REQUIRE(act == FITGNN_ACT_NONE || act == FITGNN_ACT_ELU, FITGNN_EINVAL, "spmm_blocked: unknown act %d", act);
  if (n_blk == 0) return FITGNN_OK;
  cudaStream_t st = as_stream(stream);
  const int nq = width / 4;
  // static slices of 128 floats (32 float4); inside a slice the kernel picks the staging pitch per block
  const int n_slices = (int)ceil_div(nq, 32);
  const int64_t items = n_blk * n_slices;
  const int64_t max_blocks = (int64_t)sm_count() * FG_SB_CTAS;
  const unsigned blocks = (unsigned)(items < max_blocks ? items : max_blocks);
  if (Y_lo) {
    FG_CUDA(cudaFuncSetAttribute(spmm_block_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SB_SMEM));
    spmm_block_kernel<true><<<blocks, SB_THREADS, SB_SMEM, st>>>(rowptr, col, dinv, X, ldx, nq, src_index, blk_ptr, n_blk,
                                                                 row_order, n_slices, bias, act, Y, Y_lo, ldy);
  } else {
    FG_CUDA(cudaFuncSetAttribute(spmm_block_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SB_SMEM));
    spmm_block_kernel<false><<<blocks, SB_THREADS, SB_SMEM, st>>>(rowptr, col, dinv, X, ldx, nq, src_index, blk_ptr, n_blk,
                                                                  row_order, n_slices, bias, act, Y, Y_lo, ldy);
  }
  FG_LAUNCH_CHECK();
  return FITGNN_OK;
}

extern "C" int fitgnn_spmm_symnorm_grouped(const int32_t* rowptr, const int32_t* col, const float* dinv, const float* X,
                                           int64_t ldx, int width, const int32_t* src_index, int64_t n_rows, int group,
                                           void* Y, void* Y_lo, int64_t ldy, int fill_pad, float pad_value, void* stream) {
  FG_REQUIRE(rowptr && col && dinv && X && Y, FITGNN_EINVAL, "spmm_grouped: null pointer");
  FG_REQUIRE(n_rows >= 0 && width > 0, FITGNN_EINVAL, "spmm_grouped: n_rows=%lld width=%d", (long long)n_rows, width);
  FG_REQUIRE(group == 32, FITGNN_EUNSUP, "spmm_grouped: group must be 32 (got %d)", group);
  FG_REQUIRE(width % 4 == 0 && width <= 128 && ldx % 4 == 0 && ldy % 4 == 0, FITGNN_EUNSUP,
             "spmm_grouped: width (%d) must be a multiple of 4 and <= 128, ldx (%lld) / ldy (%lld) multiples of 4", width,
             (long long)ldx, (long long)ldy);
  FG_REQUIRE(((uintptr_t)X % 16) == 0 && ((uintptr_t)Y % 8) == 0 && ((uintptr_t)Y_lo % 8) == 0, FITGNN_EUNSUP,
             "spmm_grouped: X must be 16-byte, Y 8-byte aligned");
  if (n_rows == 0) return FITGNN_OK;
  cudaStream_t st = as_stream(stream);
  const int nq = width / 4;
  const int64_t n_groups = ceil_div(n_rows, 32);
  const size_t smem = spmm_group_smem(nq);
  const int64_t max_blocks = (int64_t)sm_count() * 64;
  const unsigned blocks = (unsigned)(n_groups < max_blocks ? n_groups : max_blocks);
  // pad fill: bf16 planes whose pitch leaves exactly one quad of pad columns; column `width` of the hi plane gets
  // pad_value (rounded to bf16), every other pad element zero
  const int do_pad = (fill_pad && Y_lo && ldy == width + 4 && width < 128) ? 1 : 0;
  const uint32_t pad_bits = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(pad_value));
  if (Y_lo) {
    FG_CUDA(cudaFuncSetAttribute(spmm_group_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    spmm_group_kernel<1><<<blocks, 32, smem, st>>>(rowptr, col, dinv, X, ldx, nq, src_index, n_rows, Y, Y_lo, ldy,
                                                   n_groups, do_pad, pad_bits);
  } else {
    FG_CUDA(cudaFuncSetAttribute(spmm_group_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    spmm_group_kernel<0><<<blocks, 32, smem, st>>>(rowptr, col, dinv, X, ldx, nq, src_index, n_rows, Y, Y_lo, ldy,
                                                   n_groups, 0, 0u);
  }
  FG_LAUNCH_CHECK();
  return FITGNN_OK;
}

// the same aggregation written as ONE fp16 plane [n_rows, ldy] (ldy in elements): the A operand of the first transform when
// the whole forward runs on fp16 planes (PackedForward(precision="fp16")); fp32 sums, one rounding (saturating) at the end
extern "C" int fitgnn_spmm_symnorm_grouped_f16(const int32_t* rowptr, const int32_t* col, const float* dinv, const float* X,
                                               int64_t ldx, int width, const int32_t* src_index, int64_t n_rows, int group,
                                               void* Y, int64_t ldy, int fill_pad, float pad_value, void* stream) {
  FG_REQUIRE(rowptr && col && dinv && X && Y, FITGNN_EINVAL, "spmm_grouped_f16: null pointer");
  FG_REQUIRE(n_rows >= 0 && width > 0, FITGNN_EINVAL, "spmm_grouped_f16: n_rows=%lld width=%d", (long long)n_rows, width);
  FG_REQUIRE(group == 32, FITGNN_EUNSUP, "spmm_grouped_f16: group must be 32 (got %d)", group);
  FG_REQUIRE(width % 4 == 0 && width <= 128 && ldx % 4 == 0 && ldy % 4 == 0 && ldy >= width, FITGNN_EUNSUP,
             "spmm_grouped_f16: width (%d) must be a multiple of 4 and <= 128, ldx (%lld) / ldy (%lld) multiples of 4", width,
             (long long)ldx, (long long)ldy);
  FG_REQUIRE(((uintptr_t)X % 16) == 0 && ((uintptr_t)Y % 8) == 0, FITGNN_EUNSUP, "spmm_grouped_f16: X must be 16-byte, Y 8-byte aligned");
  if (n_rows == 0) return FITGNN_OK;
  cudaStream_t st = as_stream(stream);
  const int nq = width / 4;
  const int64_t n_groups = ceil_div(n_rows, 32);
  const size_t smem = spmm_group_smem(nq);
  const int64_t max_blocks = (int64_t)sm_count() * 64;
  const unsigned blocks = (unsigned)(n_groups < max_blocks ? n_groups : max_blocks);
  // pad fill (pitch = width + 4 only): Y[:, width] = pad_value, the other three pad elements 0 — whole 8-byte quads
  const int do_pad = (fill_pad && ldy == width + 4 && width < 128) ? 1 : 0;
  const uint32_t pad_bits = (uint32_t)__half_as_ushort(__float2half_rn(pad_value));
  FG_CUDA(cudaFuncSetAttribute(spmm_group_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  spmm_group_kernel<2><<<blocks, 32, smem, st>>>(rowptr, col, dinv, X, ldx, nq, src_index, n_rows, Y, nullptr, ldy, n_groups,
                                                 do_pad, pad_bits);
  FG_LAUNCH_CHECK();
  return FITGNN_OK;
}

// ---------------------------------------------------------------------------------------------------------
// SAGEConv mean aggregation (PyG SAGEConv with aggr='mean', root_weight=True):
//   concat form: Y[i] = [ mean_{e in row r} X[src(col_e)] | X[src(r)] ]   (each half `half` columns wide, pad columns 0)
//   root form:   Y[i] = act( mean_{e in row r} Z[src(col_e), 0:width] + Z[src(r), root_off : root_off + width] + bias )
// r = out_rows[i].  The concat row is the A operand of ONE transform against [W_l | W_r]; the root form finishes a
// transform-first layer whose GEMM produced Z = X·[W_l ; W_r]^T.  With skip_self the entry col == r (the single self entry
// a pack materialises per row) is neither summed nor counted.  With src_scale the sum is weighted by src_scale[col_e] and not
// divided (the transposed mean operator of the backward).
// Layout as spmm_pipe_kernel: LPR lanes own a row, every lane a float4 column slice; a group reads LPR column indices at
// once and then gathers their rows FG_SPMM_UNROLL at a time.  The sum runs in CSR order as one fmaf chain per element, then
// ONE correctly rounded division by the count, so results do not depend on out_rows / src_index / the launch shape.
// Rows of any length are walked in LPR-entry chunks by their own group (no hub split).
// ---------------------------------------------------------------------------------------------------------
namespace fitgnn {

template <int NV, int LPR, bool ROOT, bool SPLIT>
__global__ void __launch_bounds__(SPMM_THREADS, FG_SPMM_MINB)
spmm_mean_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ X,
                 int64_t ldx, int nq, int nqh, int64_t root_off, const int32_t* __restrict__ src_index,
                 const float* __restrict__ src_scale, int skip_self, const float* __restrict__ bias, int act,
                 const int32_t* __restrict__ out_rows, int64_t n_out, void* Y, void* Ylo, int64_t ldy) {
  constexpr unsigned FULL = 0xffffffffu;
  constexpr int G = 32 / LPR;
  constexpr int U = FG_SPMM_UNROLL;
  constexpr unsigned GMASK = LPR == 32 ? FULL : ((1u << LPR) - 1u);
  const int lane = threadIdx.x & 31;
  const int sub = lane & (LPR - 1);
  const int gshift = lane & ~(LPR - 1);
  const int64_t i = ((int64_t)blockIdx.x * SPMM_WARPS + (threadIdx.x >> 5)) * G + lane / LPR;
  const bool live = i < n_out;
  int r = 0, beg = 0, end = 0;  // every lane stays for the shuffles; a dead group has an empty range
  if (live) {
    r = out_rows ? __ldg(out_rows + i) : (int)i;
    beg = __ldg(rowptr + r);
    end = __ldg(rowptr + r + 1);
  }
  const int64_t root = live ? (src_index ? (int64_t)__ldg(src_index + r) : (int64_t)r) * ldx + root_off : 0;
  for (int q0 = 0; q0 < nqh; q0 += LPR * NV) {
    float4 acc[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    int cnt = 0;
    for (int e0 = beg; __any_sync(FULL, e0 < end); e0 += LPR) {
      int c = -1;
      if (e0 + sub < end) {
        c = __ldg(col + e0 + sub);
        if (skip_self && c == r) c = -1;
      }
      const int64_t soff = c >= 0 ? (src_index ? (int64_t)__ldg(src_index + c) : (int64_t)c) * ldx : 0;
      const float w = (c >= 0 && src_scale) ? __ldg(src_scale + c) : 1.f;
      const unsigned gm = (__ballot_sync(FULL, c >= 0) >> gshift) & GMASK;  // this group's live entries
      cnt += __popc(gm);
      const int m = __reduce_max_sync(FULL, 32 - __clz(gm));
      for (int j = 0; j < m; j += U) {
        float wj[U];
        int64_t pj[U];
        bool on[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          wj[u] = __shfl_sync(FULL, w, j + u, LPR);
          pj[u] = __shfl_sync(FULL, soff, j + u, LPR);
          on[u] = j + u < LPR && ((gm >> (j + u)) & 1u);
        }
        float4 x[U][NV];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
          for (int v = 0; v < NV; ++v) {
            const int q = q0 + sub + LPR * v;
            x[u][v] = (on[u] && q < nq) ? ldg4(X + pj[u] + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (on[u]) {
#pragma unroll
            for (int v = 0; v < NV; ++v) fma4(acc[v], wj[u], x[u][v]);
          }
      }
    }
    if (!live) continue;
    const float fc = (float)cnt;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int q = q0 + sub + LPR * v;
      if (q >= nqh) continue;
      float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
      if (q < nq) {
        o = acc[v];
        if (!src_scale && cnt > 0) {
          o.x = __fdiv_rn(o.x, fc); o.y = __fdiv_rn(o.y, fc); o.z = __fdiv_rn(o.z, fc); o.w = __fdiv_rn(o.w, fc);
        }
      }
      if (ROOT) {
        const float4 z = ldg4(X + root + 4 * q);
        o.x += z.x; o.y += z.y; o.z += z.z; o.w += z.w;
        if (bias) {
          const float4 b = ldg4(bias + 4 * q);
          o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
        }
        if (act == FITGNN_ACT_ELU) {
          o.x = elu1(o.x); o.y = elu1(o.y); o.z = elu1(o.z); o.w = elu1(o.w);
        }
        store_row4<SPLIT ? IO_SPLIT : IO_F32>(Y, Ylo, i * ldy + 4 * q, o);
      } else {
        store_row4<SPLIT ? IO_SPLIT : IO_F32>(Y, Ylo, i * ldy + 4 * q, o);
        const float4 z = q < nq ? ldg4(X + root + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
        store_row4<SPLIT ? IO_SPLIT : IO_F32>(Y, Ylo, i * ldy + 4 * (int64_t)nqh + 4 * q, z);
      }
    }
  }
}

template <int NV, int LPR, bool ROOT>
static int launch_mean(const int32_t* rowptr, const int32_t* col, const float* X, int64_t ldx, int nq, int nqh,
                       int64_t root_off, const int32_t* src_index, const float* src_scale, int skip_self, const float* bias,
                       int act, const int32_t* out_rows, int64_t n_out, void* Y, void* Ylo, int64_t ldy, cudaStream_t st) {
  constexpr int G = 32 / LPR;
  const int64_t blocks = ceil_div(n_out, (int64_t)G * SPMM_WARPS);
  FG_REQUIRE(blocks < (1ll << 31), FITGNN_ERANGE, "spmm_mean: too many rows");
  if (Ylo)
    spmm_mean_kernel<NV, LPR, ROOT, true><<<(unsigned)blocks, SPMM_THREADS, 0, st>>>(
        rowptr, col, X, ldx, nq, nqh, root_off, src_index, src_scale, skip_self, bias, act, out_rows, n_out, Y, Ylo, ldy);
  else
    spmm_mean_kernel<NV, LPR, ROOT, false><<<(unsigned)blocks, SPMM_THREADS, 0, st>>>(
        rowptr, col, X, ldx, nq, nqh, root_off, src_index, src_scale, skip_self, bias, act, out_rows, n_out, Y, Ylo, ldy);
  FG_LAUNCH_CHECK();
  return FITGNN_OK;
}

template <bool ROOT>
static int mean_dispatch(const int32_t* rowptr, const int32_t* col, const float* X, int64_t ldx, int nq, int nqh,
                         int64_t root_off, const int32_t* src_index, const float* src_scale, int skip_self, const float* bias,
                         int act, const int32_t* out_rows, int64_t n_out, void* Y, void* Ylo, int64_t ldy, void* stream) {
  if (n_out == 0) return FITGNN_OK;
  cudaStream_t st = as_stream(stream);
#define FG_MEAN(NV, LPR)                                                                                                    \
  return launch_mean<NV, LPR, ROOT>(rowptr, col, X, ldx, nq, nqh, root_off, src_index, src_scale, skip_self, bias, act,   \
                                    out_rows, n_out, Y, Ylo, ldy, st)
  // (float4 per lane, lanes per row) from the output half's width, as spmm_dispatch; wider rows loop over 512-column blocks
  if (nqh <= 8) { FG_MEAN(1, 8); }
  if (nqh <= 16) { FG_MEAN(2, 8); }
  if (nqh <= 32) { FG_MEAN(4, 8); }
  if (nqh <= 64) { FG_MEAN(4, 16); }
  FG_MEAN(4, 32);
#undef FG_MEAN
}

}  // namespace fitgnn

extern "C" int fitgnn_spmm_mean_concat(const int32_t* rowptr, const int32_t* col, const float* X, int64_t ldx, int width,
                                       int half, const int32_t* src_index, const float* src_scale, int skip_self,
                                       const int32_t* out_rows, int64_t n_out, void* Y, void* Y_lo, int64_t ldy, void* stream) {
  FG_REQUIRE(rowptr && col && X && Y, FITGNN_EINVAL, "spmm_mean_concat: null pointer");
  FG_REQUIRE(n_out >= 0 && width > 0 && half >= width, FITGNN_EINVAL, "spmm_mean_concat: n_out=%lld width=%d half=%d",
             (long long)n_out, width, half);
  FG_REQUIRE(width % 4 == 0 && half % 4 == 0 && ldx % 4 == 0 && ldy % 4 == 0 && ldy >= 2 * (int64_t)half, FITGNN_EUNSUP,
             "spmm_mean_concat: width (%d), half (%d), ldx (%lld), ldy (%lld) must be multiples of 4, ldy >= 2 * half", width,
             half, (long long)ldx, (long long)ldy);
  FG_REQUIRE(((uintptr_t)X % 16) == 0 && ((uintptr_t)Y % (Y_lo ? 8 : 16)) == 0 && ((uintptr_t)Y_lo % 8) == 0, FITGNN_EUNSUP,
             "spmm_mean_concat: X must be 16-byte aligned, Y 16-byte (fp32) / 8-byte (planes)");
  return mean_dispatch<false>(rowptr, col, X, ldx, width / 4, half / 4, 0, src_index, src_scale, skip_self, nullptr,
                              FITGNN_ACT_NONE, out_rows, n_out, Y, Y_lo, ldy, stream);
}

extern "C" int fitgnn_spmm_mean_root(const int32_t* rowptr, const int32_t* col, const float* Z, int64_t ldz, int width,
                                     int64_t root_off, const int32_t* src_index, const float* src_scale, int skip_self,
                                     const float* bias, int act, const int32_t* out_rows, int64_t n_out, void* Y, void* Y_lo,
                                     int64_t ldy, void* stream) {
  FG_REQUIRE(rowptr && col && Z && Y, FITGNN_EINVAL, "spmm_mean_root: null pointer");
  FG_REQUIRE(n_out >= 0 && width > 0 && root_off >= 0, FITGNN_EINVAL, "spmm_mean_root: n_out=%lld width=%d root_off=%lld",
             (long long)n_out, width, (long long)root_off);
  FG_REQUIRE(width % 4 == 0 && root_off % 4 == 0 && ldz % 4 == 0 && ldy % 4 == 0 && ldy >= width && width <= ldz &&
                 root_off + width <= ldz,
             FITGNN_EUNSUP, "spmm_mean_root: width (%d), root_off (%lld), ldz (%lld), ldy (%lld): multiples of 4, "
             "root_off + width <= ldz", width, (long long)root_off, (long long)ldz, (long long)ldy);
  FG_REQUIRE(((uintptr_t)Z % 16) == 0 && ((uintptr_t)Y % (Y_lo ? 8 : 16)) == 0 && ((uintptr_t)Y_lo % 8) == 0 &&
                 (!bias || ((uintptr_t)bias % 16) == 0),
             FITGNN_EUNSUP, "spmm_mean_root: Z / bias must be 16-byte aligned, Y 16-byte (fp32) / 8-byte (planes)");
  FG_REQUIRE(act == FITGNN_ACT_NONE || act == FITGNN_ACT_ELU, FITGNN_EINVAL, "spmm_mean_root: unknown act %d", act);
  return mean_dispatch<true>(rowptr, col, Z, ldz, width / 4, width / 4, root_off, src_index, src_scale, skip_self, bias, act,
                             out_rows, n_out, Y, Y_lo, ldy, stream);
}
