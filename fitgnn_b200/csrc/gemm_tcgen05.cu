// Dense transform on the 5th-gen tensor cores (FITGNN_GEMM_BF16X3):
//     Y[M,N] = head(act(A[M,K] · W[N,K]^T + bias))      (GCNConv.lin / lt1, /root/reference/network.py:31,34)
// with fp32-grade accuracy from bf16 MMAs: both operands are hi/lo bf16 planes (x = hi + lo, |x - hi - lo| <= 2^-17|x|)
// and every k-block issues  A_hi·W_hi + A_lo·W_hi + A_hi·W_lo  into one fp32 TMEM accumulator (the lo·lo term is
// below fp32 rounding).  Measured against the 1e-3 bound in tests/test_gpu_gemm_tc.py.
//
// Structure (one persistent CTA per SM, 192 threads):
//   warp 0      TMA producer: 4 cp.async.bulk.tensor loads per stage (A_hi, A_lo, W_hi, W_lo; 128B-swizzled,
//               K-major, OOB rows/columns zero-filled by the TMA unit) completing on a full[] mbarrier
//   warp 1      TMEM allocator + single-thread tcgen05.mma issuer (cta_group::1, kind::f16, M=128, N=BLOCK_N, K=16);
//               tcgen05.commit releases the smem stage (empty[]) and publishes the accumulator (tmem_full[])
//   warps 2..5  epilogue: tcgen05.ld 32x32b (thread = one output row), + bias, ELU / row (log-)softmax, st.global;
//               two TMEM accumulator stages so the epilogue of tile i overlaps the MMAs of tile i+1
// Every mbarrier wait is bounded (clock64 budget) and traps instead of hanging the GPU.
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>
#include <cuda_bf16.h>
#include <type_traits>
#include "common.cuh"

namespace fitgnn {

namespace tc {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;                      // bf16 elements = 128 bytes = one SWIZZLE_128B row
constexpr int UMMA_K = 16;
constexpr int EPI_WARPS = 8;                      // default: two per TMEM lane quadrant, each taking half of the columns
constexpr int EPI_WARPS_WIDE = 16;                // epilogue-bound instantiations: four per quadrant (one 32-column box each)
constexpr int EPI_WARPS_12 = 12;                  // fused aggregation with an fp16-plane output: three per quadrant (3 + 3 + 2 boxes)
constexpr int THREADS = 64 + 32 * EPI_WARPS;
constexpr int GATHER_WARPS = 4;                   // fused layer: produce the A tile (Â·X) in-kernel, 32 rows per warp
constexpr int GATHER_WARP0 = 2 + EPI_WARPS;
constexpr int THREADS_GATHER = THREADS + 32 * GATHER_WARPS;

// Fused GCN layer (aggregate-first, K <= 128): the A operand of the transform is Â·X[src], gathered through the
// pack CSR by dedicated warps instead of being loaded by TMA (replaces a separate SpMM launch and its HBM round trip).
struct GatherArgs {
  const int32_t* rowptr;
  const int32_t* col;
  const float* dinv;
  const float* X;          // [n_src, ldx] fp32
  const int32_t* src_index;  // gid (may be null)
  const int32_t* out_rows;   // output row -> pack row (may be null)
  int64_t ldx;
  int nq;                  // float4 per feature row (width / 4)
};
// Epilogue extensions.
//  * agg_desc / agg_dinv (AGG instantiation): the rows form a group-aligned pack (align.cu) and the epilogue applies
//    the NEXT layer's normalised aggregation to the activated tile before storing it:
//        G[r,:] = dinv[r] * ( dinv[r]*h[r,:] + sum_{c in desc(r)} dinv[c]*h[c,:] ),   h = act(A·W^T + bias)
//    Thread = row and a warp's 32 rows are exactly one aligned group, so every neighbour c is another lane of the same
//    warp: the exchange is register-to-register (__shfl_sync), no shared memory, no HBM round trip for h.
//  * row_map: output row m is written to Y row row_map[m] (skipped when negative) with per-thread stores instead of
//    TMA boxes — used by the head to drop the padding rows / scatter straight into the caller's row order.
struct EpiArgs {
  const unsigned long long* agg_desc;  // [M] bits [0,4) = entry count (<= 12), then 5-bit lanes
  const float* agg_dinv;               // [M] deg^-1/2 (0 for padding rows)
  const int32_t* row_map;              // [M] or null
  // n_peers > 0 (needs row_map): every output row is stored to peers[0..n_peers) + row_map[m] * ldy instead of Y — the
  // same slot of every rank's gather buffer (peer-mapped pointers: the stores travel over NVLink), which replaces the
  // all-gather that would otherwise follow the head kernel
  float* peers[8];
  int n_peers;
  // row-mapped narrow heads: stage each quadrant's 32 rows linearly (pitch ldy) in shared memory and write every run of
  // consecutive destination rows with ONE bulk copy per destination — full-line writes, which is what makes the stores
  // to peer memory run at NVLink speed (16-byte per-thread stores reach ~120 GB/s).  Set by the launcher when
  // N <= 64, ldy == pad4(N) and all bases are 16-byte aligned.
  int bulk_rows;
  // row_scale: y = act(row_scale[m] * (A·W^T)[m,:] + bias) — a per-row factor folded into the bias add as one FFMA.
  // agg_defer_scale: the AGG epilogue stores dinv[r]*h[r] + sum dinv[c]*h[c] WITHOUT the leading dinv[r]; the consumer
  // (the next transform, through its row_scale) applies it — a row scaling commutes with the GEMM.
  const float* row_scale;
  int agg_defer_scale;
  // Batched product (split-K of the training path's dW = G^T·A, fitgnn_gemm_tn): the M rows are n_batches stacked blocks of
  // m_batch_rows rows (a multiple of the tile height), and the tiles of block s multiply W rows [s * w_batch_rows,
  // s * w_batch_rows + N): Y_s = A_s · W_s^T.  m_batch_rows = 0: plain GEMM.  w_rows_total = rows of the stacked W.
  int64_t m_batch_rows;
  int w_batch_rows;
  int64_t w_rows_total;
  // Operand / output formats.  a_planes = 2: A is a bf16 hi/lo pair (3 MMAs per k-step: hi*hi + lo*hi + hi*lo, the default).
  // a_planes = 1 with f16 = 1 (FITGNN_GEMM_FP16X2): A is ONE fp16 plane (11-bit significand), W an fp16 hi/lo pair; 2 MMAs per
  // k-step (A*W_hi + A*W_lo), no A_lo load.  out_f16 = 1: the result is stored as ONE fp16 plane (the next FP16X2 product's A).
  int a_planes;
  int f16;
  int out_f16;
  // w_planes = 1 (FITGNN_GEMM_FP16X2 with W_lo = NULL, i.e. "fp16x1"): W is ONE fp16 plane as well — one MMA per k-step, no
  // W_lo load.  Halves the B bytes an SM has to ingest per k-block, and a pair's half of a 256 x 512 weight block (128 KB)
  // then fits in shared memory: the W-stationary CTA-pair plan below.
  int w_planes;
  int l2_prefetch;  // producer: prefetch the next m-block's A rows into L2 (tuning switch gemm_prefetch, default off)
  int debug;        // measurement switches (tuning gemm_debug, default 0): bit 0 = the epilogue skips its TMA stores
};
constexpr int EPI_WARP0 = 2;
constexpr int ACC_STAGES = 2;
constexpr uint32_t A_PLANE_BYTES = BLOCK_M * BLOCK_K * 2;  // 16 KB
constexpr long long WAIT_BUDGET_CYCLES = 4000000000ll;     // ~2 s at 1.9 GHz

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// bounded wait: a protocol bug must fail loudly (trap -> sticky CUDA error) instead of hanging the device
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > WAIT_BUDGET_CYCLES) {
      printf("fitgnn gemm_bf16x3: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
}

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

// pull a tile into L2 only (no shared memory, no barrier): the producer runs these one m-block ahead of its loads
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* map, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(map), "r"(c0), "r"(c1) : "memory");
}

// smem -> global tile store (clipped at the tensor bounds by the TMA unit), tracked by bulk async-groups
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map), "r"(src),
               "r"(c0), "r"(c1)
               : "memory");
}
// contiguous smem -> global copy (16-byte aligned, size a multiple of 16); the destination may be peer memory
__device__ __forceinline__ void bulk_store_1d(void* dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// K-major, 128B-swizzled operand tile: rows of 128 bytes, 8-row swizzle atoms 1024 bytes apart
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);  // start address, bits [0,14)
  d |= (uint64_t)0 << 16;                        // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024u >> 4) << 32;             // stride byte offset between 8-row atoms, bits [32,46)
  d |= (uint64_t)1 << 46;                        // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                        // layout type: SWIZZLE_128B
  return d;
}

// kind::f16 instruction descriptor: D = f32, A = B = bf16, both K-major, M x N
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// same with fp16 operands (format code 0)
__host__ __device__ constexpr uint32_t umma_idesc_f16(int m, int n) {
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// ---- CTA pair (cta_group::2): two SMs of one TPC share one 256-row MMA; each holds its own 128 rows of A and HALF of
// the B tile, which is what cuts the per-SM operand traffic (the streaming GEMM is bound by the SM's TMA ingest)
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t mapa_rank(uint32_t local_addr, uint32_t rank) {  // shared::cluster address in CTA `rank`
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load into THIS CTA's shared memory whose bytes are counted on a barrier of the pair's leader CTA
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the barrier at this offset in BOTH CTAs of the pair once the MMAs issued so far have retired
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"(mask)
               : "memory");
}
// The only thing this arrive orders is the TMEM reads before it (complete after tcgen05.wait::ld, made visible by
// tcgen05.fence::before_thread_sync): default .release.cta semantics suffice.  `.release.cluster` compiled to
// MEMBAR.ALL.CTA + ERRBAR and cost 14 % of the peer CTA's epilogue samples (ncu r2s).
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// one lane of the (converged) warp; the same lane every time, so its commits track its own MMAs
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,"
      "%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
// the same load split into issue and wait, so that independent global loads (the bias) can be issued in between.  The wait
// takes the 32 registers as in/out operands: nothing that reads them can be scheduled above it.
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,"
      "%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld32_wait(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]),
                 "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
                 "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// branchless ELU: exp via MUFU.EX2, absolute error <= ~2e-7 (far below the fp32 re-association noise of the GEMM)
__device__ __forceinline__ float elu1(float x) { return elu_fast(x); }

__host__ __device__ constexpr int tmem_cols(int n) { return n <= 32 ? 32 : n <= 64 ? 64 : n <= 128 ? 128 : n <= 256 ? 256 : 512; }
__host__ __device__ constexpr uint32_t stage_bytes(int block_n) { return 2 * A_PLANE_BYTES + 2 * (uint32_t)block_n * BLOCK_K * 2; }
constexpr uint32_t EPI_BOX_BYTES = 32 * 32 * 4;             // one 32-row x 32-column fp32 store box (128B rows)
__host__ __device__ constexpr int num_stages(int block_n) {
  int s = (int)((192 * 1024) / stage_bytes(block_n));
  return s > 8 ? 8 : s;
}

template <int BLOCK_N, bool GATHER, int AGG, int EW, bool CTA2 = false>
__global__ void __launch_bounds__(64 + 32 * EW + (GATHER ? 32 * GATHER_WARPS : 0), 1)
gemm_bf16x3_kernel(const GatherArgs ga, const EpiArgs ea, const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                   const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                   const __grid_constant__ CUtensorMap map_y, const __grid_constant__ CUtensorMap map_y_lo,
                   int tma_store, const float* __restrict__ bias, int64_t M, int K, int N, int act, int head,
                   float* __restrict__ Y, int64_t ldy, int w_stationary, int n_stages) {
  constexpr int STAGES = num_stages(BLOCK_N);
  constexpr int MAX_STAGES = 8;
  // CTA2: launched as clusters of two CTAs; the pair computes a 256-row x BLOCK_N tile (this CTA: its own 128 rows),
  // every CTA stages its own A rows and HALF of the B tile (BLOCK_N / 2 weight rows), the leader (cluster rank 0) issues
  // cta_group::2 MMAs that read both halves.  Streaming plan only.
  constexpr int B_ROWS = CTA2 ? BLOCK_N / 2 : BLOCK_N;
  constexpr uint32_t B_PLANE_BYTES = (uint32_t)B_ROWS * BLOCK_K * 2;
  constexpr int TMEM_COLS = tmem_cols(ACC_STAGES * BLOCK_N);
  constexpr uint32_t IDESC_BF16 = umma_idesc_bf16(CTA2 ? 2 * BLOCK_M : BLOCK_M, BLOCK_N);
  constexpr uint32_t IDESC_F16 = umma_idesc_f16(CTA2 ? 2 * BLOCK_M : BLOCK_M, BLOCK_N);
  const uint32_t IDESC = ea.f16 ? IDESC_F16 : IDESC_BF16;
  const bool a_single = ea.a_planes == 1;
  const bool w_single = ea.w_planes == 1;
  static_assert(!CTA2 || (!GATHER && BLOCK_N % 32 == 0), "CTA pairs: streaming plan, UMMA N multiple of 32 for M=256");
  const uint32_t cta_rank = CTA2 ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;
  static_assert(BLOCK_N % 16 == 0 && BLOCK_N >= 16 && BLOCK_N <= 256, "UMMA N for M=128");
  static_assert(STAGES >= 2, "need at least two smem stages");
  static_assert(EW == EPI_WARPS || (EW == EPI_WARPS_WIDE && !GATHER) || (EW == EPI_WARPS_12 && !GATHER && BLOCK_N == 256),
                "2, 3 (256-column tile with an fp16-plane output) or 4 epilogue warps per TMEM lane quadrant");
  // one 32 x 32 box per epilogue warp: 4 KB (fp32, or bf16 hi + lo); the 12-warp variant only writes ONE fp16 plane (2 KB)
  constexpr bool HALF_STAGE = BLOCK_N == 256 && (EW == EPI_WARPS_12 || (AGG && EW == EPI_WARPS_WIDE));  // these require out_f16
  // (the CTA-pair instantiation decides at run time: an fp16-plane output leaves 16 KB for one more A stage)
  const uint32_t WARP_STAGE = (HALF_STAGE || (CTA2 && ea.out_f16)) ? EPI_BOX_BYTES / 2 : EPI_BOX_BYTES;
  const uint32_t STAGING_BYTES = EW * WARP_STAGE;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);  // SWIZZLE_128B atoms
  const int k_blocks = (K + BLOCK_K - 1) / BLOCK_K;
  // Two smem plans.  Streaming: n_stages x {A_hi, A_lo, W_hi, W_lo}.  W-stationary (small K): the CTA keeps its
  // N-block of the weights resident for the whole kernel (k_blocks x {W_hi, W_lo}) and only A streams, which removes
  // the per-tile weight re-load from L2 that otherwise dominates the SM<->L2 traffic of a small-K transform.
  // CTA pairs can be W-stationary too (each CTA keeps ITS half of the pair's N-block): the pair's n-block is fixed and it
  // strides over the m-blocks, so per k-block an SM ingests only its 16 KB of A.
  const uint32_t b_bytes = (w_single ? 1u : 2u) * B_PLANE_BYTES;  // W share of a k-block: hi (+ lo)
  const uint32_t w_region_bytes = w_stationary ? (uint32_t)k_blocks * b_bytes : 0u;
  // a single-plane A (fp16) has no lo slot: the stage shrinks by one plane, which buys pipeline depth (the N = 48 head:
  // 5 stages of 16 KB instead of 2 of 32 KB beside its resident weights)
  const uint32_t a_bytes = (a_single ? 1u : 2u) * A_PLANE_BYTES;
  const uint32_t stage_bytes_rt = w_stationary ? a_bytes : a_bytes + b_bytes;
  uint8_t* staging = smem + w_region_bytes + (size_t)n_stages * stage_bytes_rt;  // multiples of 1024 throughout
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + STAGING_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * MAX_STAGES + 2 * ACC_STAGES + 1);
  const uint32_t smem_base = smem_u32(smem) + w_region_bytes;  // first streaming stage
  const uint32_t w_base = smem_u32(smem);                       // resident weights (W-stationary)
  const uint32_t bar_base = smem_u32(bars);
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (MAX_STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * MAX_STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * MAX_STAGES + ACC_STAGES + s); };
  const uint32_t wfull_bar = bar_base + 8u * (2 * MAX_STAGES + 2 * ACC_STAGES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (N + BLOCK_N - 1) / BLOCK_N;
  constexpr int TILE_M = CTA2 ? 2 * BLOCK_M : BLOCK_M;  // rows per tile of the walk (a pair's tile has 256)
  const int64_t m_tiles = (M + TILE_M - 1) / TILE_M;
  const int64_t tiles = m_tiles * n_tiles;
  // Tile walk.  Every role (producer, MMA issuer, epilogue warps) steps through the same sequence of (m-block, n-block)
  // pairs with a few 32-bit adds per tile.  (The first version derived every tile from a running index with 64-bit
  // divisions — tile_at(i), t / n_tiles, t % n_tiles, twice per tile for the prefetch of the next tile's row data: ~370
  // dependent instructions per tile and epilogue warp, a third of the epilogue warps' samples in ncu r2af.)
  //   streaming, single CTA : tile t = blockIdx, + gridDim, ... with the n-block fastest (t = mb * n_tiles + nt)
  //   W-stationary          : the CTA's (pair's) n-block is fixed, it strides over the m-blocks
  //   streaming CTA pairs   : pair p takes m-blocks p, p + n_pairs, ... and ALL n-blocks of a block back to back: the block's
  //                           A rows are re-read from L2 by the same two SMs a few microseconds later.  (Round-robin over
  //                           (m, n) gave the two N-tiles of a block to two different pairs at about the same time; ncu r1x
  //                           counted 7.1 GB of DRAM reads for 5.0 GB of operands.)
  //   W-stationary pairs    : pair p keeps n-block p % n_tiles and walks the m-blocks p / n_tiles, + n_pairs / n_tiles, ...
  //                           (the launcher makes n_pairs a multiple of n_tiles); the n_tiles pairs that share an m-block run
  //                           side by side, so the block's second read is (mostly) an L2 hit.
  struct Walk { int mb, nt; };
  const int ctas_per_n = (int)gridDim.x / n_tiles;
  Walk w0;
  int walk_dm, walk_dn, walk_carry;
  if (CTA2) {
    const int p = (int)(blockIdx.x >> 1), np = (int)(gridDim.x >> 1);
    if (w_stationary) { w0 = Walk{p / n_tiles, p % n_tiles}; walk_dm = np / n_tiles; walk_dn = 0; walk_carry = 0; }
    else { w0 = Walk{p, 0}; walk_dm = 0; walk_dn = 1; walk_carry = np; }
  } else if (w_stationary) {
    w0 = Walk{(int)blockIdx.x / n_tiles, (int)blockIdx.x % n_tiles}; walk_dm = ctas_per_n; walk_dn = 0; walk_carry = 0;
  } else {
    w0 = Walk{(int)blockIdx.x / n_tiles, (int)blockIdx.x % n_tiles};
    walk_dm = (int)gridDim.x / n_tiles; walk_dn = (int)gridDim.x % n_tiles; walk_carry = 1;
  }
  auto advance = [&](Walk& w) {
    w.nt += walk_dn;
    w.mb += walk_dm;
    if (w.nt >= n_tiles) { w.nt -= n_tiles; w.mb += walk_carry; }
  };
  auto valid = [&](const Walk& w) { return (int64_t)w.mb < m_tiles; };
  // first row THIS CTA owns in the tile
  auto tile_row0 = [&](const Walk& w) { return (int64_t)w.mb * TILE_M + (int64_t)cta_rank * BLOCK_M; };
  // batched product: first W row of the batch the tile belongs to
  auto w_batch_off = [&](const Walk& w) -> int {
    return ea.m_batch_rows ? (int)(((int64_t)w.mb * TILE_M) / ea.m_batch_rows) * ea.w_batch_rows : 0;
  };
  // the gather warps (GATHER: single CTA, W-stationary) keep their own arithmetic walk over the running tile index
  const int64_t t_first = blockIdx.x;
  const int64_t t_step = (int64_t)ctas_per_n * n_tiles;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(full_bar(s), GATHER ? GATHER_WARPS : 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(wfull_bar, 1);
    for (int s = 0; s < ACC_STAGES; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), CTA2 ? 2 * EW : EW);  // one arrival per epilogue warp (of both CTAs of a pair)
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if (CTA2) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                   "r"((uint32_t)TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                   "r"((uint32_t)TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  fence_before();
  __syncthreads();
  if (CTA2) cluster_sync_all();  // the peer's barriers are initialised before anything arrives on them remotely
  fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    // warp-uniform loop, one elected lane issues (same reason as the MMA issuer below)
    {
      uint32_t stage = 0, phase = 0;
      if (w_stationary && valid(w0)) {
        const int n0 = w0.nt * BLOCK_N;
        if (elect_one()) {
          if (CTA2) {  // both CTAs' halves are counted on the LEADER's barrier (its MMA thread reads both)
            const uint32_t lbar = mapa_rank(wfull_bar, 0);
            if (leader) mbar_arrive_expect_tx(wfull_bar, 2 * w_region_bytes);
            for (int kb = 0; kb < k_blocks; ++kb) {
              tma_load_2d_pair(w_base + kb * b_bytes, &map_w_hi, lbar, kb * BLOCK_K, n0 + (int)cta_rank * B_ROWS);
              if (!w_single)
                tma_load_2d_pair(w_base + kb * b_bytes + B_PLANE_BYTES, &map_w_lo, lbar, kb * BLOCK_K, n0 + (int)cta_rank * B_ROWS);
            }
          } else {
            mbar_arrive_expect_tx(wfull_bar, w_region_bytes);
            for (int kb = 0; kb < k_blocks; ++kb) {
              tma_load_2d(w_base + kb * b_bytes, &map_w_hi, wfull_bar, kb * BLOCK_K, n0);
              if (!w_single) tma_load_2d(w_base + kb * b_bytes + B_PLANE_BYTES, &map_w_lo, wfull_bar, kb * BLOCK_K, n0);
            }
          }
        }
        __syncwarp();
      }
      int prev_mb = -1;
      for (Walk w = w0; valid(w) && !GATHER; advance(w)) {  // gather mode: A is produced by the gather warps
        const int m0 = (int)tile_row0(w);
        const int n0 = w.nt * BLOCK_N + w_batch_off(w);  // W row of this tile (epilogue columns: nt * BLOCK_N)
        // L2 prefetch, one m-block ahead (tuning switch gemm_prefetch, OFF by default): while the first tile of an m-block
        // streams, the A rows of the NEXT m-block of the walk are pulled into L2, k-block by k-block.  Built because ncu r2ai
        // showed the MMA warp of a W-stationary pair (4 A stages of 16 KB beside 128 KB of weights) waiting for operands a
        // third of the time; MEASURED SLOWER (r2aj: layer-2 transform 1.21 -> 1.31 ms, fused transform 1.14 -> 1.16 ms): the
        // prefetches queue in front of the loads in the SM's one TMA pipe.
        int pf_m0 = -1;
        if (w.mb != prev_mb) {
          Walk pf = w;
          for (int i = 0; i < n_tiles && valid(pf) && pf.mb == w.mb; ++i) advance(pf);
          if (valid(pf) && pf.mb != w.mb) pf_m0 = (int)tile_row0(pf);
        }
        prev_mb = w.mb;
        for (int kb = 0; kb < k_blocks; ++kb) {
          if (pf_m0 >= 0 && ea.l2_prefetch) {
            if (elect_one()) {
              tma_prefetch_2d(&map_a_hi, kb * BLOCK_K, pf_m0);
              if (!a_single) tma_prefetch_2d(&map_a_lo, kb * BLOCK_K, pf_m0);
            }
            __syncwarp();
          }
          mbar_wait(empty_bar(stage), phase ^ 1);
          const uint32_t dst = smem_base + stage * stage_bytes_rt;
          const uint32_t tx_bytes = stage_bytes_rt;
          __syncwarp();
          if (elect_one()) {
            if (CTA2) {
              // both CTAs' bytes are counted on the LEADER's full barrier (its MMA thread consumes both halves)
              const uint32_t lbar = mapa_rank(full_bar(stage), 0);
              if (leader) mbar_arrive_expect_tx(full_bar(stage), 2 * tx_bytes);
              tma_load_2d_pair(dst, &map_a_hi, lbar, kb * BLOCK_K, m0);
              if (!a_single) tma_load_2d_pair(dst + A_PLANE_BYTES, &map_a_lo, lbar, kb * BLOCK_K, m0);
              if (!w_stationary) {
                tma_load_2d_pair(dst + a_bytes, &map_w_hi, lbar, kb * BLOCK_K, n0 + (int)cta_rank * B_ROWS);
                if (!w_single)
                  tma_load_2d_pair(dst + a_bytes + B_PLANE_BYTES, &map_w_lo, lbar, kb * BLOCK_K, n0 + (int)cta_rank * B_ROWS);
              }
            } else {
              mbar_arrive_expect_tx(full_bar(stage), tx_bytes);
              tma_load_2d(dst, &map_a_hi, full_bar(stage), kb * BLOCK_K, m0);
              if (!a_single) tma_load_2d(dst + A_PLANE_BYTES, &map_a_lo, full_bar(stage), kb * BLOCK_K, m0);
              if (!w_stationary) {
                tma_load_2d(dst + a_bytes, &map_w_hi, full_bar(stage), kb * BLOCK_K, n0);
                if (!w_single) tma_load_2d(dst + a_bytes + B_PLANE_BYTES, &map_w_lo, full_bar(stage), kb * BLOCK_K, n0);
              }
            }
          }
          __syncwarp();
          if (++stage == (uint32_t)n_stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (the pair's leader CTA)
    // The WHOLE warp walks the loop (waits included) so that every address and descriptor is warp-uniform, and one
    // elected lane issues the MMAs + commits of a k-block.  With the loop under `lane == 0` instead, the compiler cannot
    // prove uniformity and wraps EVERY tcgen05.mma in an ELECT / R2UR.BROADCAST waterfall: ~260 SASS instructions and
    // ~1,100 cycles per k-block on one thread (ncu r2q) — the bound of the N = 48 head (8 small MMAs per k-block) and
    // level with the 8 MMAs of a pair's fp16 k-block.
    // The loop is instantiated per operand format (hi/lo or single planes): with the plane counts as run-time predicates the
    // k-block body carried the descriptor arithmetic of all 12 possible MMAs (~140 uniform-datapath instructions, ~560
    // cycles per k-block on the one issuing thread — level with the 512 cycles the 4 MMAs of a single-plane k-block execute;
    // ncu r2ai).
    auto mma_loop = [&](auto a1_t, auto w1_t) {
      constexpr bool A1 = decltype(a1_t)::value, W1 = decltype(w1_t)::value;
      uint32_t stage = 0, phase = 0;
      uint32_t it = 0;
      if (w_stationary && valid(w0)) mbar_wait(wfull_bar, 0);  // resident weights have landed
      for (Walk w = w0; valid(w); ++it, advance(w)) {
        const uint32_t acc = it % ACC_STAGES;
        const uint32_t acc_phase = (it / ACC_STAGES) & 1u;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1);  // epilogue has drained this accumulator
        fence_after();
        const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(full_bar(stage), phase);  // TMA bytes have landed
          fence_after();
          const uint32_t a_hi = smem_base + stage * stage_bytes_rt;
          const uint32_t w_hi = w_stationary ? w_base + kb * b_bytes : a_hi + a_bytes;
          const uint64_t d_a_hi = umma_desc_sw128(a_hi);
          const uint64_t d_a_lo = umma_desc_sw128(a_hi + A_PLANE_BYTES);
          const uint64_t d_w_hi = umma_desc_sw128(w_hi);
          const uint64_t d_w_lo = umma_desc_sw128(w_hi + B_PLANE_BYTES);
          __syncwarp();
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
              const uint64_t adv = (uint64_t)((k * UMMA_K * 2) >> 4);  // +32 bytes per K=16 step inside the swizzle row
              if (CTA2) {
                umma_bf16_pair(tmem_d, d_a_hi + adv, d_w_hi + adv, IDESC, (kb | k) != 0);
                if (!A1) umma_bf16_pair(tmem_d, d_a_lo + adv, d_w_hi + adv, IDESC, 1);
                if (!W1) umma_bf16_pair(tmem_d, d_a_hi + adv, d_w_lo + adv, IDESC, 1);
              } else {
                umma_bf16(tmem_d, d_a_hi + adv, d_w_hi + adv, IDESC, (kb | k) != 0);
                if (!A1) umma_bf16(tmem_d, d_a_lo + adv, d_w_hi + adv, IDESC, 1);
                if (!W1) umma_bf16(tmem_d, d_a_hi + adv, d_w_lo + adv, IDESC, 1);
              }
            }
            if (CTA2) {
              umma_commit_pair(empty_bar(stage));  // frees the stage in BOTH CTAs
              if (kb == k_blocks - 1) umma_commit_pair(tfull_bar(acc));
            } else {
              umma_commit(empty_bar(stage));  // smem stage is free once these MMAs retire
              if (kb == k_blocks - 1) umma_commit(tfull_bar(acc));
            }
          }
          __syncwarp();
          if (++stage == (uint32_t)n_stages) { stage = 0; phase ^= 1; }
        }
      }
    };
    if (leader) {
      if (a_single && w_single) mma_loop(std::true_type{}, std::true_type{});
      else if (a_single) mma_loop(std::true_type{}, std::false_type{});
      else mma_loop(std::false_type{}, std::false_type{});
    }
    __syncwarp();
  } else if (GATHER && warp >= GATHER_WARP0) {
    // ------------------------------------------------------------------ gather warps: A tile = Â·X[src] (bf16 hi/lo)
    // 8 lanes per row, 4 rows per warp step, 8 steps per tile; software-pipelined across steps AND tiles exactly like
    // spmm_pipe_kernel (row info 3 steps ahead, column indices 2, dinv/gid 1).  A row's 128 columns (4 float4 per
    // lane) cover both 64-column k-blocks; element (row r, col c) of k-block c/64 goes to the canonical K-major
    // SWIZZLE_128B position r*128 + (((c%64)/8) ^ (r&7))*16 + ((c%8)/4)*8 of the hi / lo plane.
    constexpr int LPR = 8, STEPS = BLOCK_M / (GATHER_WARPS * 4);
    constexpr unsigned FULL = 0xffffffffu;
    const int gw = warp - GATHER_WARP0, sub = lane & (LPR - 1), grp = lane / LPR;
    const int64_t my_tiles = (t_first < tiles) ? (tiles - 1 - t_first) / t_step + 1 : 0;
    const int64_t total_steps = my_tiles * STEPS;
    struct RI { int beg, end; float dr; };
    auto load_info = [&](int64_t step) {
      RI ri{0, 0, 0.f};
      if (step < total_steps) {
        const int64_t t = t_first + (step / STEPS) * t_step;
        const int64_t i = (t / n_tiles) * BLOCK_M + gw * 32 + (int)(step % STEPS) * 4 + grp;
        if (i < M) {
          const int r = ga.out_rows ? __ldg(ga.out_rows + i) : (int)i;
          ri.beg = __ldg(ga.rowptr + r);
          ri.end = __ldg(ga.rowptr + r + 1);
          ri.dr = __ldg(ga.dinv + r);
        }
      }
      return ri;
    };
    auto load_col = [&](const RI& ri, int e0) { return (e0 + sub < ri.end) ? __ldg(ga.col + e0 + sub) : -1; };
    auto load_w = [&](int c) { return c >= 0 ? __ldg(ga.dinv + c) : 0.f; };
    auto load_s = [&](int c) { return c >= 0 ? (ga.src_index ? __ldg(ga.src_index + c) : c) : 0; };
    auto gather_chunk = [&](float4 (&acc)[4], int cnt, float w, int sidx) {
      const int maxcnt = __reduce_max_sync(FULL, cnt);
      for (int j = 0; j < maxcnt; j += 2) {
        float wj[2];
        const float* pj[2];
        bool on[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          wj[u] = __shfl_sync(FULL, w, j + u, LPR);
          const int sj = __shfl_sync(FULL, sidx, j + u, LPR);
          pj[u] = ga.X + (int64_t)sj * ga.ldx;
          on[u] = j + u < cnt;
        }
        float4 x[2][4];
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            const int q = sub + LPR * v;
            x[u][v] = (on[u] && q < ga.nq) ? __ldg(reinterpret_cast<const float4*>(pj[u]) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            acc[v].x = fmaf(wj[u], x[u][v].x, acc[v].x); acc[v].y = fmaf(wj[u], x[u][v].y, acc[v].y);
            acc[v].z = fmaf(wj[u], x[u][v].z, acc[v].z); acc[v].w = fmaf(wj[u], x[u][v].w, acc[v].w);
          }
      }
    };
    RI ia = load_info(0), ib = load_info(1), ic = load_info(2);
    int ca = load_col(ia, ia.beg), cb = load_col(ib, ib.beg);
    float wa = load_w(ca);
    int sa = load_s(ca);
    uint32_t stage = 0, phase = 0;
    for (int64_t step = 0; step < total_steps; ++step) {
      const RI id = load_info(step + 3);
      const int cc = load_col(ic, ic.beg);
      const float wb = load_w(cb);
      const int sb = load_s(cb);
      const int s_in_tile = (int)(step % STEPS);
      if (s_in_tile == 0) {  // the k_blocks stages of this tile must have been released by the MMAs that read them
        if (lane == 0)
          for (int kb = 0; kb < k_blocks; ++kb) mbar_wait(empty_bar(stage + kb), phase ^ 1);
        __syncwarp();
      }
      const int deg = ia.end - ia.beg;
      float4 acc[4];
#pragma unroll
      for (int v = 0; v < 4; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
      gather_chunk(acc, min(deg, LPR), wa, sa);
      const bool long_row = deg > LPR;
      for (int e0 = ia.beg + LPR; __any_sync(FULL, long_row && e0 < ia.end); e0 += LPR) {
        const int c = long_row ? load_col(ia, e0) : -1;
        gather_chunk(acc, long_row ? max(0, min(ia.end - e0, LPR)) : 0, load_w(c), load_s(c));
      }
      const int lr = gw * 32 + s_in_tile * 4 + grp;  // row inside the tile
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int c = 4 * (sub + LPR * v);  // first of this lane's 4 columns
        const int kb = c >> 6;
        if (kb < k_blocks) {
          const float x[4] = {acc[v].x * ia.dr, acc[v].y * ia.dr, acc[v].z * ia.dr, acc[v].w * ia.dr};
          uint32_t hi[2], lo[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) split_bf16x2(x[2 * u], x[2 * u + 1], hi[u], lo[u]);
          const int cc64 = c & 63;
          const uint32_t a = smem_base + (stage + kb) * stage_bytes_rt + lr * 128 +
                             ((uint32_t)(cc64 >> 3) ^ (uint32_t)(lr & 7)) * 16 + ((cc64 & 7) >> 2) * 8;
          asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(a), "r"(hi[0]), "r"(hi[1]) : "memory");
          asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(a + A_PLANE_BYTES), "r"(lo[0]), "r"(lo[1]) : "memory");
        }
      }
      if (s_in_tile == STEPS - 1) {
        fence_proxy_async();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
        __syncwarp();
        if (lane == 0)
          for (int kb = 0; kb < k_blocks; ++kb) mbar_arrive(full_bar(stage + kb));
        stage += k_blocks;
        if (stage >= (uint32_t)n_stages) { stage = 0; phase ^= 1; }
      }
      ia = ib; ib = ic; ic = id;
      ca = cb; cb = cc;
      wa = wb; sa = sb;
    }
  } else {
    // ------------------------------------------------------------------ epilogue (thread = output row)
    const int quad = warp & 3;  // TMEM lane quadrant this warp may access
    const int row_in_tile = quad * 32 + lane;
    bool vec_ok = (ldy % 4 == 0) && (((uintptr_t)Y & 15) == 0);
#pragma unroll
    for (int p = 0; p < 8; ++p)
      if (p < ea.n_peers) vec_ok = vec_ok && (((uintptr_t)ea.peers[p] & 15) == 0);
    const bool bias_vec = (((uintptr_t)bias & 15) == 0);
    // column split: 32-column boxes; the second warp of a quadrant takes the upper half of the boxes.  A fused
    // (log-)softmax needs the whole row in one thread, so the first warp of the quadrant then takes every box.
    constexpr int N_BOXES = (BLOCK_N + 31) / 32;
    // Narrow heads (<= 64 columns, i.e. one box per warp): single pass — both warps of a quadrant keep their box in
    // registers, exchange (max, sum exp) through shared memory and normalise.  Wider heads: two passes by warp 0.
    constexpr bool FAST_HEAD = N_BOXES <= 2 && EW == EPI_WARPS;
    const bool use_fast_head = FAST_HEAD && head != FITGNN_HEAD_IDENTITY;
    float2* exch = reinterpret_cast<float2*>(reinterpret_cast<uint8_t*>(bars) + 256);  // [2][EPI_WARPS][32]
    const int ew = warp - EPI_WARP0;
    const int col_group = ew >> 2;
    // EW / 4 column groups share the boxes evenly; a two-pass (log-)softmax gives every box to group 0
    constexpr int GROUPS = EW / 4;
    constexpr int BOXES_PER_GROUP = (N_BOXES + GROUPS - 1) / GROUPS;
    const bool one_group = head != FITGNN_HEAD_IDENTITY && !FAST_HEAD;
    const int box_beg = one_group ? (col_group == 0 ? 0 : N_BOXES) : min(N_BOXES, col_group * BOXES_PER_GROUP);
    const int box_end = one_group ? N_BOXES : min(N_BOXES, box_beg + BOXES_PER_GROUP);
    uint32_t it = 0;
    // aggregation descriptor + dinv of this thread's row, fetched one tile ahead of its use
    unsigned long long desc_next = 0ull;
    float dr_next = 0.f, rs_next = 1.f;
    auto load_agg = [&](const Walk& wt) {
      desc_next = 0ull;
      dr_next = 0.f;
      rs_next = 1.f;
      if ((AGG || ea.row_scale) && valid(wt)) {
        const int64_t mm = tile_row0(wt) + row_in_tile;
        if (mm < M) {
          if (AGG) {
            desc_next = __ldg(ea.agg_desc + mm);
            dr_next = __ldg(ea.agg_dinv + mm);
          }
          if (ea.row_scale) rs_next = __ldg(ea.row_scale + mm);
        }
      }
    };
    load_agg(w0);
    Walk w_next = w0;
    for (Walk w = w0; valid(w); ++it, w = w_next) {
      const uint32_t acc = it % ACC_STAGES;
      const uint32_t acc_phase = (it / ACC_STAGES) & 1u;
      const int64_t tile_m0 = tile_row0(w);
      const int64_t m = tile_m0 + row_in_tile;
      const int n0 = w.nt * BLOCK_N;
      const unsigned long long desc = desc_next;
      const float dr = dr_next;
      const float rs = rs_next;
      advance(w_next);
      load_agg(w_next);
      const int agg_cnt = (int)(desc & 15ull);
      const int agg_max = AGG ? __reduce_max_sync(0xffffffffu, agg_cnt) : 0;
      mbar_wait(tfull_bar(acc), acc_phase);
      fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * BLOCK_N;
      const int64_t dest_row = (ea.row_map && m < M) ? (int64_t)__ldg(ea.row_map + m) : m;
      float* yrow = Y + dest_row * ldy + n0;
      float row_max = -INFINITY, row_sum = 0.f;
      bool exchanged = false, staged = false;
      const bool bulk_rows = FAST_HEAD && ea.bulk_rows != 0;
      // one linear [32 rows][ldy] fp32 buffer per TMEM lane quadrant (<= 8 KB), shared by the quadrant's two warps
      const uint32_t qbuf = smem_u32(staging) + (uint32_t)quad * 2u * EPI_BOX_BYTES;
      const uint32_t row_bytes = (uint32_t)ldy * 4u;
      auto stage_and_store = [&](const float (&vals)[32], bool have, int c0, int ncols) {
        // (a) the previous tile's bulk copies have finished reading the buffer, (b) both warps know it
        if (col_group == 0 && lane == 0) bulk_wait_read<0>();
        asm volatile("bar.sync %0, 64;" ::"r"(1 + quad) : "memory");
        if (have) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            if (j < ncols && c0 + j < (int)ldy) {
              const float x0 = (n0 + c0 + j < N) ? vals[j] : 0.f, x1 = (n0 + c0 + j + 1 < N) ? vals[j + 1] : 0.f;
              const float x2 = (n0 + c0 + j + 2 < N) ? vals[j + 2] : 0.f, x3 = (n0 + c0 + j + 3 < N) ? vals[j + 3] : 0.f;
              asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(qbuf + lane * row_bytes + (uint32_t)(c0 + j) * 4u),
                           "f"(x0), "f"(x1), "f"(x2), "f"(x3) : "memory");
            }
          }
        }
        fence_proxy_async();
        asm volatile("bar.sync %0, 64;" ::"r"(1 + quad) : "memory");
        if (col_group == 0) {
          // runs of consecutive destination rows -> one bulk copy per run and destination, issued by lane 0
          const int dr_ = (m < M) ? (int)dest_row : -1;
          const int prev = __shfl_up_sync(0xffffffffu, dr_, 1);
          const unsigned valid = __ballot_sync(0xffffffffu, dr_ >= 0);
          const unsigned starts = __ballot_sync(0xffffffffu, dr_ >= 0 && (lane == 0 || prev < 0 || dr_ != prev + 1));
          unsigned rem = starts;
          while (rem) {
            const int s0 = __ffs(rem) - 1;
            rem &= rem - 1;
            const unsigned stop = (rem | ~valid) & ~((2u << s0) - 1u);  // next run start or next invalid row after s0
            const int s1 = stop ? __ffs(stop) - 1 : 32;
            const int d0 = __shfl_sync(0xffffffffu, dr_, s0);
            if (lane == 0) {
              const int n_dst = ea.n_peers > 0 ? ea.n_peers : 1;
#pragma unroll
              for (int p = 0; p < 8; ++p) {  // constant indices: a dynamic one would copy the parameter array to the stack
                if (p < n_dst) {
                  float* base = ea.n_peers > 0 ? ea.peers[p] : Y;
                  bulk_store_1d(base + (int64_t)d0 * ldy, qbuf + (uint32_t)s0 * row_bytes, (uint32_t)(s1 - s0) * row_bytes);
                }
              }
            }
          }
          if (lane == 0) bulk_commit();
        }
        staged = true;
      };
      auto exchange_stats = [&](float lmax, float lsum) {
        // partner warp = same TMEM quadrant, other column group; buffers alternate by tile parity
        float2* mine = exch + ((it & 1) * EW + ew) * 32 + lane;
        const float2* theirs = exch + ((it & 1) * EW + (ew ^ 4)) * 32 + lane;
        *mine = make_float2(lmax, lsum);
        asm volatile("bar.sync %0, 64;" ::"r"(1 + quad) : "memory");
        const float2 o = *theirs;
        row_max = fmaxf(lmax, o.x);
        row_sum = (lsum > 0.f ? lsum * __expf(lmax - row_max) : 0.f) + (o.y > 0.f ? o.y * __expf(o.x - row_max) : 0.f);
        exchanged = true;
      };
      if (head != FITGNN_HEAD_IDENTITY && !FAST_HEAD && col_group == 0) {
        // pass 1: online max / sum of exp over the row (the whole row lives in this tile: N <= BLOCK_N)
        for (int c0 = 0; c0 < BLOCK_N; c0 += 16) {
          float v[16];
          tmem_ld16(taddr + c0, v);
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int n = n0 + c0 + j;
            if (n < N) {
              float x = v[j] + (bias ? __ldg(bias + n) : 0.f);
              if (act == FITGNN_ACT_ELU) x = elu1(x);
              const float nm = fmaxf(row_max, x);
              row_sum = row_sum * __expf(row_max - nm) + __expf(x - nm);
              row_max = nm;
            }
          }
        }
      }
      // only a two-pass (log-)softmax needs these here; computing them unconditionally put logf(0) and the 1/0 slow path
      // (a CALL that waits for every outstanding load, i.e. for the next tile's prefetched descriptors) into EVERY tile of
      // EVERY transform: 6.5 % of the fused-aggregation epilogue's samples (ncu r2s)
      float log_sum = 0.f, inv_sum = 0.f;
      if (head != FITGNN_HEAD_IDENTITY && !FAST_HEAD) {
        log_sum = logf(row_sum);
        inv_sum = 1.f / row_sum;
      }
      const uint32_t buf = smem_u32(staging) + (uint32_t)(warp - EPI_WARP0) * WARP_STAGE;
      const int m_base = (int)tile_m0 + quad * 32;
      for (int box = box_beg; box < box_end; ++box) {
        const int c0 = box * 32;
        if (n0 + c0 >= N) break;
        const int box_cols = (BLOCK_N - c0 >= 32) ? 32 : 16;  // BLOCK_N is a multiple of 16
        float v[32];
        // full boxes with a 16-byte aligned bias: the bias loads are issued BETWEEN the TMEM load and its wait (they used to
        // follow the wait, and the first FFMA then sat on the L1 round trip: 14 % of the per-box samples in ncu r2ai)
        // (not in the register-bound 12/16-warp aggregation epilogues: 32 more live registers spill there)
        constexpr bool BIAS_PRE = !(AGG && EW != EPI_WARPS);
        const bool bias_full = bias && bias_vec && n0 + c0 + 32 <= N;
        const bool bias_pre = BIAS_PRE && bias_full;
        float4 bq[8];
        auto bias4 = [&](int j) -> float4 {
          return BIAS_PRE ? bq[j >> 2] : __ldg(reinterpret_cast<const float4*>(bias + n0 + c0 + j));
        };
        if (box_cols == 32) {
          uint32_t r[32];
          tmem_ld32_issue(taddr + c0, r);
          if (bias_pre) {
#pragma unroll
            for (int j = 0; j < 8; ++j) bq[j] = __ldg(reinterpret_cast<const float4*>(bias + n0 + c0) + j);
          }
          tmem_ld32_wait(r);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        } else {
          if (bias_pre) {
#pragma unroll
            for (int j = 0; j < 8; ++j) bq[j] = __ldg(reinterpret_cast<const float4*>(bias + n0 + c0) + j);
          }
          float lo16[16];
          tmem_ld16(taddr + c0, lo16);
#pragma unroll
          for (int j = 0; j < 16; ++j) { v[j] = lo16[j]; v[16 + j] = 0.f; }
        }
        auto aggregate = [&](float (&v)[32]) {
          // normalised aggregation over the warp's aligned group (see EpiArgs); padding rows (dr = 0) give 0 * h = 0.
          // AGG == 1: applied to the ACTIVATED tile (the next layer's propagate).  AGG == 2: applied to the raw accumulators,
          // before bias and activation — act(Â·(A·W^T) + b), a whole GCNConv of the aligned pack in this one kernel.
          // (the A operand's padding rows must hold finite values: the engine's SpMM writes zeros there)
          // AGG_W columns at a time (16 when the register budget is 112 per thread, i.e. 16 epilogue warps)
#ifndef FG_AGG_W12
#define FG_AGG_W12 32  // 16-column chunks measured slower: 1.175 vs 1.149 ms (r2ap)
#endif
          constexpr int AGG_W = EW == EPI_WARPS_WIDE ? 16 : EW == EPI_WARPS_12 ? FG_AGG_W12 : 32;
#pragma unroll
          for (int h0 = 0; h0 < 32; h0 += AGG_W) {
            float u[AGG_W];
#pragma unroll
            for (int j = 0; j < AGG_W; ++j) {
              u[j] = v[h0 + j] * dr;
              v[h0 + j] = u[j];
            }
            for (int sl = 0; sl < agg_max; ++sl) {
              const bool on = sl < agg_cnt;
              const int src = on ? (int)((desc >> (4 + 5 * sl)) & 31ull) : lane;
#pragma unroll
              for (int j = 0; j < AGG_W; ++j) {
                const float tv = __shfl_sync(0xffffffffu, u[j], src);
                if (on) v[h0 + j] += tv;
              }
            }
            if (!ea.agg_defer_scale) {
#pragma unroll
              for (int j = 0; j < AGG_W; ++j) v[h0 + j] *= dr;
            }
          }
        };
        if (AGG == 2) aggregate(v);
        if (ea.row_scale) {  // act(rs * acc + bias): the scale rides on the bias add
          if (bias_full) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 b4 = bias4(j);
              v[j] = fmaf(v[j], rs, b4.x); v[j + 1] = fmaf(v[j + 1], rs, b4.y);
              v[j + 2] = fmaf(v[j + 2], rs, b4.z); v[j + 3] = fmaf(v[j + 3], rs, b4.w);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = fmaf(v[j], rs, (bias && n0 + c0 + j < N) ? __ldg(bias + n0 + c0 + j) : 0.f);
          }
        } else if (bias) {
          if (bias_full) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 b4 = bias4(j);
              v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (n0 + c0 + j < N) v[j] += __ldg(bias + n0 + c0 + j);
          }
        }
        if (act == FITGNN_ACT_ELU) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = elu1(v[j]);
        }
        if (AGG == 1) aggregate(v);
        if (use_fast_head) {
          float lmax = -INFINITY, lsum = 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (j < box_cols && n0 + c0 + j < N) lmax = fmaxf(lmax, v[j]);
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (j < box_cols && n0 + c0 + j < N) lsum += __expf(v[j] - lmax);
          exchange_stats(lmax, lsum);
          log_sum = logf(row_sum);
          inv_sum = 1.f / row_sum;
        }
        if (head == FITGNN_HEAD_LOG_SOFTMAX) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = v[j] - row_max - log_sum;
        } else if (head == FITGNN_HEAD_SOFTMAX) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __expf(v[j] - row_max) * inv_sum;
        }
        if (bulk_rows) {
          stage_and_store(v, true, c0, box_cols);
        } else if (tma_store) {
          // stage the box in this warp's 4 KB buffer (row = lane) and hand it to the TMA unit, which clips at the
          // tensor bounds.  fp32: 128-byte rows, 16-byte chunk c of row r at c ^ (r & 7).  bf16 hi/lo planes: two
          // 2 KB boxes of 64-byte rows, chunk c of row r at c ^ ((r >> 1) & 3).
          // (bulk async-groups belong to a thread: elect_one picks the same lane every time)
          if (elect_one()) bulk_wait_read<0>();  // the store(s) that last read this buffer have finished reading
          __syncwarp();
          if (tma_store == 3) {  // ONE fp16 plane (64-byte rows, the bf16 planes' swizzle)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint32_t h[4];
#pragma unroll
              for (int u = 0; u < 4; ++u) h[u] = pack_f16x2_rn(v[8 * j + 2 * u], v[8 * j + 2 * u + 1]);
              const uint32_t a = buf + lane * 64 + ((uint32_t)j ^ (uint32_t)((lane >> 1) & 3)) * 16;
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(h[0]), "r"(h[1]), "r"(h[2]), "r"(h[3])
                           : "memory");
            }
          } else if (tma_store == 2) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint32_t hi[4], lo[4];
#pragma unroll
              for (int u = 0; u < 4; ++u) split_bf16x2(v[8 * j + 2 * u], v[8 * j + 2 * u + 1], hi[u], lo[u]);
              const uint32_t a = buf + lane * 64 + ((uint32_t)j ^ (uint32_t)((lane >> 1) & 3)) * 16;
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(hi[0]), "r"(hi[1]), "r"(hi[2]),
                           "r"(hi[3]) : "memory");
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a + EPI_BOX_BYTES / 2), "r"(lo[0]),
                           "r"(lo[1]), "r"(lo[2]), "r"(lo[3]) : "memory");
            }
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const uint32_t a = buf + lane * 128 + ((uint32_t)j ^ (uint32_t)(lane & 7)) * 16;
              asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v[4 * j]), "f"(v[4 * j + 1]),
                           "f"(v[4 * j + 2]), "f"(v[4 * j + 3]) : "memory");
            }
          }
          fence_proxy_async();
          __syncwarp();
          if (elect_one() && !(ea.debug & 1)) {  // debug bit 0 (tuning gemm_debug, measurements only): drop the stores
            tma_store_2d(&map_y, buf, n0 + c0, m_base);
            if (tma_store == 2) tma_store_2d(&map_y_lo, buf + EPI_BOX_BYTES / 2, n0 + c0, m_base);
            bulk_commit();
          }
        } else if (m < M && dest_row >= 0) {
          // a row map with the pitch N rounded up to 4: the pitch-padding columns [N, ldy) are written as zeros, like the
          // bulk row copies do, so that what a caller's buffer holds does not depend on which store path ran
          const int n_end = (ea.row_map && ldy == (int64_t)((N + 3) & ~3)) ? (int)ldy : N;
          if (n0 + c0 + 32 > N) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (n0 + c0 + j >= N) v[j] = 0.f;
          }
          const int n_dst = ea.n_peers > 0 ? ea.n_peers : 1;
#pragma unroll
          for (int p = 0; p < 8; ++p) {
            if (p >= n_dst) break;
            float* yp = ea.n_peers > 0 ? ea.peers[p] + dest_row * ldy + n0 : yrow;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              if (vec_ok && j + 4 <= box_cols && n0 + c0 + j + 4 <= n_end) {
                *reinterpret_cast<float4*>(yp + c0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
              } else {
#pragma unroll
                for (int u = 0; u < 4; ++u)
                  if (j + u < box_cols && n0 + c0 + j + u < n_end) yp[c0 + j + u] = v[j + u];
              }
            }
          }
        }
      }
      if (use_fast_head && !exchanged) exchange_stats(-INFINITY, 0.f);  // no box this tile: still meet the partner
      if (bulk_rows && !staged) {
        const float none[32] = {};
        stage_and_store(none, false, 0, 0);
      }
      fence_before();
      __syncwarp();
      if (lane == 0) {  // this warp's quadrant of the accumulator is drained (pairs: tell the leader's MMA thread)
        if (CTA2 && !leader) mbar_arrive_remote(mapa_rank(tempty_bar(acc), 0));
        else mbar_arrive(tempty_bar(acc));
      }
    }
    if (tma_store || ea.bulk_rows) {  // smem must outlive the last bulk store (row-mapped path: lane 0 committed; boxes: the elected lane)
      if (lane == 0) bulk_wait_all();
      __syncwarp();
      if (elect_one()) bulk_wait_all();
    }
  }

  fence_before();
  __syncthreads();
  if (CTA2) cluster_sync_all();  // neither CTA frees tensor memory (or exits) while its peer still works on the pair's tile
  if (warp == 1) {
    fence_after();
    if (CTA2)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                   : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                   : "memory");
  }
}

// ---------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// bf16 [rows, cols] row-major with pitch ld (elements); box = BLOCK_K columns x box_rows rows, 128B swizzle,
// out-of-bounds elements read as zero
static int make_map(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  FG_REQUIRE(fn, FITGNN_ECUDA, "gemm_bf16x3: cuTensorMapEncodeTiled is not available from the driver");
  FG_REQUIRE(((uintptr_t)base & 15) == 0 && (ld * 2) % 16 == 0, FITGNN_EUNSUP,
             "gemm_bf16x3: bf16 planes need 16-byte aligned bases and a pitch that is a multiple of 8 elements");
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  const cuuint32_t box[2] = {(cuuint32_t)BLOCK_K, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FG_REQUIRE(r == CUDA_SUCCESS, FITGNN_ECUDA, "gemm_bf16x3: cuTensorMapEncodeTiled failed (%d)", (int)r);
  return FITGNN_OK;
}

// fp32 output [rows, cols] with pitch ld: 32 x 32 store boxes, 128B swizzle (matches the epilogue staging layout)
static int make_store_map(CUtensorMap* map, float* base, int64_t rows, int64_t cols, int64_t ld) {
  EncodeTiledFn fn = encode_fn();
  FG_REQUIRE(fn, FITGNN_ECUDA, "gemm_bf16x3: cuTensorMapEncodeTiled is not available from the driver");
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  const cuuint32_t box[2] = {32, 32};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FG_REQUIRE(r == CUDA_SUCCESS, FITGNN_ECUDA, "gemm_bf16x3: cuTensorMapEncodeTiled (store) failed (%d)", (int)r);
  return FITGNN_OK;
}

// bf16 output plane [rows, cols] with pitch ld: 32 x 32 store boxes (64-byte rows), 64B swizzle
static int make_store_map_bf16(CUtensorMap* map, void* base, int64_t rows, int64_t cols, int64_t ld) {
  EncodeTiledFn fn = encode_fn();
  FG_REQUIRE(fn, FITGNN_ECUDA, "gemm_bf16x3: cuTensorMapEncodeTiled is not available from the driver");
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  const cuuint32_t box[2] = {32, 32};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FG_REQUIRE(r == CUDA_SUCCESS, FITGNN_ECUDA, "gemm_bf16x3: cuTensorMapEncodeTiled (bf16 store) failed (%d)", (int)r);
  return FITGNN_OK;
}

#ifndef FG_AGG12_DEFAULT
#define FG_AGG12_DEFAULT 1
#endif
template <int BLOCK_N, bool GATHER, int AGG, int EW = EPI_WARPS, bool CTA2 = false>
static int launch(const GatherArgs& ga, const EpiArgs& ea, const CUtensorMap& a_hi, const CUtensorMap& a_lo, const void* W_hi, const void* W_lo, int64_t ldw,
                  const float* bias, int64_t M, int K, int N, int act, int head, float* Y, void* Y_lo, int64_t ldy,
                  int sms, cudaStream_t st) {
  CUtensorMap w_hi, w_lo;
  const int64_t w_rows = ea.m_batch_rows ? ea.w_rows_total : (int64_t)N;
  FG_TRY(make_map(&w_hi, W_hi, w_rows, K, ldw, CTA2 ? BLOCK_N / 2 : BLOCK_N));  // a CTA of a pair stages half of the B tile
  FG_TRY(make_map(&w_lo, W_lo ? W_lo : W_hi, w_rows, K, ldw, CTA2 ? BLOCK_N / 2 : BLOCK_N));  // unused with a single-plane W
  const size_t w_planes = ea.w_planes == 1 ? 1 : 2;
  CUtensorMap y_map, y_lo_map;
  int tma_store = ((ldy * 4) % 16 == 0 && ((uintptr_t)Y & 15) == 0) ? 1 : 0;
  y_map = w_hi;  // placeholders when unused
  y_lo_map = w_hi;
  if (ea.out_f16) {
    FG_REQUIRE(!Y_lo && !ea.row_map && (ldy * 2) % 16 == 0 && ((uintptr_t)Y & 15) == 0, FITGNN_EUNSUP,
               "gemm: fp16-plane output needs a 16-byte aligned plane with a pitch that is a multiple of 8, and no row map");
    tma_store = 3;
    FG_TRY(make_store_map_bf16(&y_map, Y, M, N, ldy));  // 16-bit elements: the map does not care which
  } else if (Y_lo) {
    FG_REQUIRE((ldy * 2) % 16 == 0 && ((uintptr_t)Y & 15) == 0 && ((uintptr_t)Y_lo & 15) == 0, FITGNN_EUNSUP,
               "gemm_bf16x3: split output needs 16-byte aligned planes and a pitch that is a multiple of 8");
    tma_store = 2;
    FG_TRY(make_store_map_bf16(&y_map, Y, M, N, ldy));
    FG_TRY(make_store_map_bf16(&y_lo_map, Y_lo, M, N, ldy));
  } else if (ea.row_map) {
    tma_store = 0;  // remapped rows: per-thread stores
  } else if (tma_store) {
    FG_TRY(make_store_map(&y_map, Y, M, N, ldy));
  }
  constexpr size_t SMEM_LIMIT = 227 * 1024;
  // staging + alignment slack + barriers/TMEM slot (256 B) + softmax exchange buffers (2 x 8 warps x 32 x float2)
  constexpr bool HALF_STAGE = BLOCK_N == 256 && (EW == EPI_WARPS_12 || (AGG && EW == EPI_WARPS_WIDE));
  const bool half_stage = HALF_STAGE || (CTA2 && ea.out_f16);  // must match the kernel's WARP_STAGE
  const size_t FIXED = (size_t)EW * (half_stage ? EPI_BOX_BYTES / 2 : EPI_BOX_BYTES) + 1024 + 256 +
                       (BLOCK_N <= 64 ? 2 * EW * 32 * 8 : 0);
  FG_REQUIRE(!HALF_STAGE || ea.out_f16, FITGNN_EINVAL, "gemm: the 12/16-epilogue-warp 256-column tile stages one fp16 plane only");
  constexpr int NTHREADS = 64 + 32 * EW + (GATHER ? 32 * GATHER_WARPS : 0);
  const int k_blocks = (K + BLOCK_K - 1) / BLOCK_K;
  const int n_tiles = (int)ceil_div(N, BLOCK_N);
  const int64_t m_tiles = ceil_div(M, BLOCK_M);
  const int64_t tiles = m_tiles * n_tiles;
  const size_t a_bytes = (size_t)(ea.a_planes == 1 ? 1 : 2) * A_PLANE_BYTES;  // stage share of A (one fp16 plane or hi + lo)
  const size_t stage_b = a_bytes + w_planes * BLOCK_N * BLOCK_K * 2;
  int n_stages = (int)((SMEM_LIMIT - FIXED) / stage_b);
  if (n_stages > 8) n_stages = 8;
  int grid = (int)(tiles < sms ? tiles : sms);
  size_t smem = (size_t)n_stages * stage_b + FIXED;
  // W-stationary plan: worth it when the resident weights fit beside >= 2 A stages and every CTA gets several m-blocks
  int w_stationary = 0;
  const size_t w_bytes = (size_t)k_blocks * w_planes * BLOCK_N * BLOCK_K * 2;
  if (!ea.m_batch_rows && w_bytes + 2 * a_bytes + FIXED <= SMEM_LIMIT && sms >= n_tiles && m_tiles >= 4 * (sms / n_tiles)) {
    w_stationary = 1;
    n_stages = (int)((SMEM_LIMIT - FIXED - w_bytes) / a_bytes);
    if (n_stages > 8) n_stages = 8;
    grid = (sms / n_tiles) * n_tiles;
    smem = w_bytes + (size_t)n_stages * a_bytes + FIXED;
  }
  if (!tuning().gemm_ws && w_stationary) {  // tuning override: force the streaming plan
    w_stationary = 0;
    n_stages = (int)((SMEM_LIMIT - FIXED) / stage_b);
    if (n_stages > 8) n_stages = 8;
    grid = (int)(tiles < sms ? tiles : sms);
    smem = (size_t)n_stages * stage_b + FIXED;
  }
  if (GATHER) {
    // the gather warps fill all k-blocks of a tile at once: needs the W-stationary plan with n_stages % k_blocks == 0
    FG_REQUIRE(w_stationary && k_blocks <= 2 && n_stages >= k_blocks, FITGNN_EUNSUP,
               "gcn_layer_fused: shape not eligible (needs K <= 128 and enough row blocks for the W-stationary plan)");
    n_stages = (n_stages / k_blocks) * k_blocks;
    smem = w_bytes + (size_t)n_stages * a_bytes + FIXED;
  }
  auto kern = gemm_bf16x3_kernel<BLOCK_N, GATHER, AGG, EW, CTA2>;
  static size_t smem_configured = 0;  // per instantiation; raised outside of stream capture by the first (warm-up) call
  if (smem > smem_configured) {
    FG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_LIMIT));
    smem_configured = SMEM_LIMIT;
  }
  if (CTA2) {
    // CTA pairs: streaming plan with half-B stages, one cluster of 2 CTAs per 256-row tile, persistent over the SM pairs
    const size_t b_half = w_planes * (size_t)(BLOCK_N / 2) * BLOCK_K * 2;  // this CTA's share of a k-block of W
    const size_t STAGE2 = a_bytes + b_half;
    w_stationary = 0;
    n_stages = (int)((SMEM_LIMIT - FIXED) / STAGE2);
    if (n_stages > 8) n_stages = 8;
    smem = (size_t)n_stages * STAGE2 + FIXED;
    const int64_t m_pair_tiles = ceil_div(M, 2 * BLOCK_M);
    const int64_t pair_tiles = m_pair_tiles * n_tiles;
    int64_t pairs = pair_tiles < sms / 2 ? pair_tiles : sms / 2;
    // W-stationary pairs: every CTA keeps its half of the pair's n-block for all k-blocks (fp16 single-plane W, K = 512:
    // 128 KB) and only A streams — the streaming pair kernel is bound by the L2 -> SM operand traffic (48 KB per k-block and
    // SM at the ~8 TB/s the chip's L2 delivers), this plan moves 16 KB.  Needs >= 3 A stages beside the weights and several
    // m-blocks per pair.  Tuning gemm_pair_ws = 0 forces the streaming plan.
    const size_t w_res = (size_t)k_blocks * b_half;
    const int64_t ws_pairs = (pairs / n_tiles) * n_tiles;
    if (tuning().gemm_pair_ws && !ea.m_batch_rows && w_res + 3 * a_bytes + FIXED <= SMEM_LIMIT && ws_pairs >= n_tiles &&
        m_pair_tiles >= 4 * (ws_pairs / n_tiles)) {
      w_stationary = 1;
      pairs = ws_pairs;
      n_stages = (int)((SMEM_LIMIT - FIXED - w_res) / a_bytes);
      if (n_stages > 8) n_stages = 8;
      smem = w_res + (size_t)n_stages * a_bytes + FIXED;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(2 * pairs));
    cfg.blockDim = dim3(NTHREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    FG_CUDA(cudaLaunchKernelEx(&cfg, kern, ga, ea, a_hi, a_lo, w_hi, w_lo, y_map, y_lo_map, tma_store, bias, M, K, N, act, head,
                               Y, ldy, w_stationary, n_stages));
    return FITGNN_OK;
  }
  kern<<<grid, NTHREADS, smem, st>>>(ga, ea, a_hi, a_lo, w_hi, w_lo, y_map, y_lo_map, tma_store, bias,
                                                              M, K, N, act, head, Y, ldy, w_stationary, n_stages);
  FG_LAUNCH_CHECK();
  return FITGNN_OK;
}

}  // namespace tc

int gemm_bf16x3(const void* A_hi, const void* A_lo, int64_t lda, const void* W_hi, const void* W_lo, int64_t ldw,
                const float* bias, int64_t M, int K, int N, int act, int head, float* Y, void* Y_lo, int64_t ldy,
                const uint64_t* agg_desc, const float* agg_dinv, const int32_t* row_map, float* const* peers, int n_peers,
                const float* row_scale, int agg_defer_scale, cudaStream_t st, int64_t m_batch_rows, int w_batch_rows,
                int64_t w_rows_total, int in_f16, int out_f16, int agg_pre) {
  FG_REQUIRE(!agg_pre || agg_desc, FITGNN_EINVAL, "gemm: agg_pre needs the aggregation descriptors");
  FG_REQUIRE(W_lo || in_f16, FITGNN_EINVAL, "gemm: a single-plane W (W_lo = NULL) needs the fp16 operand format");
  FG_REQUIRE(!in_f16 || !A_lo, FITGNN_EINVAL, "gemm: FP16X2 takes ONE fp16 A plane (A_lo must be NULL)");
  FG_REQUIRE(in_f16 || A_lo, FITGNN_EINVAL, "gemm: BF16X3 needs the A_lo plane");
  FG_REQUIRE(!out_f16 || (head == FITGNN_HEAD_IDENTITY && !Y_lo && !row_map), FITGNN_EUNSUP,
             "gemm: an fp16-plane output cannot carry a head, a lo plane or a row map");
  FG_REQUIRE(m_batch_rows == 0 || (m_batch_rows % 256 == 0 && M % m_batch_rows == 0 && w_batch_rows >= N && !agg_desc &&
                                   !row_map && head == FITGNN_HEAD_IDENTITY && w_rows_total >= (M / m_batch_rows) * w_batch_rows),
             FITGNN_EINVAL, "gemm_bf16x3: bad batching (m_batch_rows must be a multiple of 256 dividing M)");
  FG_REQUIRE(!Y_lo || head == FITGNN_HEAD_IDENTITY, FITGNN_EUNSUP, "gemm_bf16x3: split output cannot carry a head");
  FG_REQUIRE(n_peers >= 0 && n_peers <= 8 && (n_peers == 0 || (peers && row_map)), FITGNN_EINVAL,
             "gemm_bf16x3: peer stores need 1..8 peer bases and a row map");
  FG_REQUIRE(!agg_desc || (agg_dinv && head == FITGNN_HEAD_IDENTITY && !row_map && N > 128), FITGNN_EUNSUP,
             "gemm_bf16x3: the fused aggregation needs dinv, no head, no row map and a wide output (N > 128)");
  FG_REQUIRE(!row_map || !Y_lo, FITGNN_EUNSUP, "gemm_bf16x3: a row map needs fp32 output");
  FG_REQUIRE(head == FITGNN_HEAD_IDENTITY || N <= 256, FITGNN_EUNSUP,
             "gemm_bf16x3: a fused (log-)softmax head needs N <= 256 (got %d)", N);
  FG_REQUIRE(M < (1ll << 31) - 128, FITGNN_ERANGE, "gemm_bf16x3: M exceeds the TMA coordinate range");
  // persistent grids: one CTA per SM, minus the SMs left to a concurrent exchange kernel (fitgnn_peer_push launches clusters
  // of two, i.e. takes whole TPCs, so a CTA-pair GEMM loses the same number of SMs)
  int sms = sm_count() - tuning().sm_reserve;
  if (sms < 2) sms = 2;
  CUtensorMap a_hi, a_lo;
  FG_TRY(tc::make_map(&a_hi, A_hi, M, K, lda, tc::BLOCK_M));
  FG_TRY(tc::make_map(&a_lo, A_lo ? A_lo : A_hi, M, K, lda, tc::BLOCK_M));  // unused with a single-plane A
  const tc::GatherArgs ga{};
  tc::EpiArgs ea{reinterpret_cast<const unsigned long long*>(agg_desc), agg_dinv, row_map, {}, n_peers, 0, row_scale,
                 agg_defer_scale, m_batch_rows, w_batch_rows, w_rows_total, in_f16 ? 1 : 2, in_f16 ? 1 : 0, out_f16 ? 1 : 0,
                 W_lo ? 2 : 1, tuning().gemm_prefetch, tuning().gemm_debug};
  for (int p = 0; p < n_peers; ++p) ea.peers[p] = peers[p];
  if (n_peers > 0) Y = peers[0];  // alignment checks / unused fallbacks refer to a real buffer
  if (row_map && N <= 64 && ldy == (N + 3) / 4 * 4 && tuning().head_bulk) {
    bool aligned = ((uintptr_t)Y & 15) == 0;
    for (int p = 0; p < n_peers; ++p) aligned = aligned && ((uintptr_t)peers[p] & 15) == 0;
    ea.bulk_rows = aligned ? 1 : 0;
  }
  if (agg_desc && agg_pre) {
    // act(Â·(A·W^T) + b): the aggregation runs on the raw accumulators.  Hidden -> hidden layers (K > 128) on the fp16 plane
    // take the CTA-pair kernel with 12 epilogue warps: the exchange-heavy epilogue then overlaps a tensor-bound main loop
    // instead of idling the tensor cores behind a K = 100 transform.  Any other shape: the single-CTA 8-warp tile.
    if (K > 128 && out_f16 && in_f16 && M >= 4096 && tuning().gemm_pair)
      return tc::launch<256, false, 2, tc::EPI_WARPS_12, true>(ga, ea, a_hi, a_lo, W_hi, W_lo, ldw, bias, M, K, N, act, head, Y,
                                                               Y_lo, ldy, sms, st);
    return tc::launch<256, false, 2>(ga, ea, a_hi, a_lo, W_hi, W_lo, ldw, bias, M, K, N, act, head, Y, Y_lo, ldy, sms, st);
  }
  if (agg_desc) {
    // Tuning switch: 128-column tiles with 16 epilogue warps (4 per scheduler).  The small-K aggregation epilogue is
    // instruction-bound, yet the wide variant measured SLOWER (2.05 vs 1.91 ms on the products workload: twice as many
    // tiles, each warp handling a single box per tile), so the 256-column / 8-warp tile stays the default.
    if (tuning().agg_wide == 1)
      return tc::launch<128, false, true, tc::EPI_WARPS_WIDE>(ga, ea, a_hi, a_lo, W_hi, W_lo, ldw, bias, M, K, N, act, head, Y,
                                                              Y_lo, ldy, sms, st);
    // fp16-plane output: 12 epilogue warps (three per scheduler; the 2 KB boxes leave the smem for it) hide more of the
    // SHFL / MUFU latency of the exchange + ELU than 8: 1.38 -> 1.24 ms on the products workload; 16 warps at 96 registers
    // (agg_wide = 3): 1.34 ms.  agg_wide = 2 forces the 12-warp tile, -1 the 8-warp one.
    if (out_f16 && tuning().agg_wide == 3)
      return tc::launch<256, false, true, tc::EPI_WARPS_WIDE>(ga, ea, a_hi, a_lo, W_hi, W_lo, ldw, bias, M, K, N, act, head, Y,
                                                              Y_lo, ldy, sms, st);
    if (out_f16 && (tuning().agg_wide == 2 || (tuning().agg_wide == 0 && FG_AGG12_DEFAULT)))
      return tc::launch<256, false, true, tc::EPI_WARPS_12>(ga, ea, a_hi, a_lo, W_hi, W_lo, ldw, bias, M, K, N, act, head, Y,
                                                            Y_lo, ldy, sms, st);
    return tc::launch<256, false, true>(ga, ea, a_hi, a_lo, W_hi, W_lo, ldw, bias, M, K, N, act, head, Y, Y_lo, ldy, sms, st);
  }
#define FG_TC(BN) \
  return tc::launch<BN, false, false>(ga, ea, a_hi, a_lo, W_hi, W_lo, ldw, bias, M, K, N, act, head, Y, Y_lo, ldy, sms, st)
  if (N <= 16) FG_TC(16);
  if (N <= 32) FG_TC(32);
  if (N <= 48) FG_TC(48);
  if (N <= 64) FG_TC(64);
  if (N <= 128) FG_TC(128);
  // small-K wide-output transforms are epilogue-bound as well: with an fp16-plane output the 12-epilogue-warp tile
  // (see the AGG dispatch above; gemm_wide = -1 forbids it)
  if (K <= 128 && out_f16 && head == FITGNN_HEAD_IDENTITY && !row_map && tuning().gemm_wide >= 0 && FG_AGG12_DEFAULT)
    return tc::launch<256, false, false, tc::EPI_WARPS_12>(ga, ea, a_hi, a_lo, W_hi, W_lo, ldw, bias, M, K, N, act, head, Y,
                                                           Y_lo, ldy, sms, st);
  if (K <= 128 && head == FITGNN_HEAD_IDENTITY && tuning().gemm_wide)
    return tc::launch<128, false, false, tc::EPI_WARPS_WIDE>(ga, ea, a_hi, a_lo, W_hi, W_lo, ldw, bias, M, K, N, act, head, Y,
                                                             Y_lo, ldy, sms, st);
  // large-K wide transforms: CTA pairs (cta_group::2) halve the B bytes every SM has to ingest
  // (fp16-plane output: 12 epilogue warps — with ONE MMA per product the 8-warp epilogue, two latency-bound warps per
  // scheduler at IPC 0.37, was the bound of the pair kernel: ncu r2af, tensor pipe 36 % active; gemm_wide = -1 forbids it)
  if (K > 128 && head == FITGNN_HEAD_IDENTITY && !row_map && M >= 4096 && tuning().gemm_pair && out_f16 && tuning().gemm_wide >= 0)
    return tc::launch<256, false, false, tc::EPI_WARPS_12, true>(ga, ea, a_hi, a_lo, W_hi, W_lo, ldw, bias, M, K, N, act, head, Y,
                                                                 Y_lo, ldy, sms, st);
  if (K > 128 && head == FITGNN_HEAD_IDENTITY && !row_map && M >= 4096 && tuning().gemm_pair)
    return tc::launch<256, false, false, tc::EPI_WARPS, true>(ga, ea, a_hi, a_lo, W_hi, W_lo, ldw, bias, M, K, N, act, head, Y,
                                                              Y_lo, ldy, sms, st);
  FG_TC(256);
#undef FG_TC
}


// Y = act( (Â · X[src_index])[out_rows] · W^T + bias ) in one kernel (layer width K = 4 * nq <= 128, N = 512-style wide
// outputs).  Returns FITGNN_EUNSUP when the shape is not eligible so the caller can fall back to SpMM + GEMM.
int gcn_layer_fused(const int32_t* rowptr, const int32_t* col, const float* dinv, const float* X, int64_t ldx, int width,
                    const int32_t* src_index, const int32_t* out_rows, int64_t M, const void* W_hi, const void* W_lo,
                    int64_t ldw, const float* bias, int N, int act, float* Y, void* Y_lo, int64_t ldy, cudaStream_t st) {
  FG_REQUIRE(width % 4 == 0 && width <= 128 && ldx % 4 == 0 && ((uintptr_t)X & 15) == 0, FITGNN_EUNSUP,
             "gcn_layer_fused: feature width must be a multiple of 4 and <= 128 (got %d)", width);
  FG_REQUIRE(N > 128, FITGNN_EUNSUP, "gcn_layer_fused: only the wide-output tile (N > 128) is instantiated");
  FG_REQUIRE(M < (1ll << 31) - 128, FITGNN_ERANGE, "gcn_layer_fused: M exceeds the coordinate range");
  const int sms = sm_count();
  const int K = (width + 7) / 8 * 8;
  tc::GatherArgs ga{rowptr, col, dinv, X, src_index, out_rows, ldx, width / 4};
  CUtensorMap dummy;
  FG_TRY(tc::make_map(&dummy, W_hi, N, K, ldw, 16));  // placeholder for the unused A maps
  const tc::EpiArgs ea{nullptr, nullptr, nullptr, {}, 0, 0, nullptr, 0, 0, 0, 0, 2, 0, 0, 2, 0, 0};
  return tc::launch<256, true, false>(ga, ea, dummy, dummy, W_hi, W_lo, ldw, bias, M, K, N, act, FITGNN_HEAD_IDENTITY, Y,
                                      Y_lo, ldy, sms, st);
}

}  // namespace fitgnn
