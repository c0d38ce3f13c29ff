// CSR / pack builders: the packed block-diagonal CSR of all subgraphs, built once from the
// partition vector part[] (the column->row map of the coarsening matrix C).
//
//   fitgnn_csr_*   <- gcn_norm inside PyG GCNConv (call sites /root/reference/network.py:31,60,90,126,161,197)
//   fitgnn_pack_*  <- the per-cluster loop of coarsening_classification / coarsening_regression
//                     (/root/reference/utils.py:186-267, :269-350, :417-501, :503-584), with its helpers
//                     neighbour()/nodes_2_neighbours() (utils.py:52-62), Data.subgraph (utils.py:248) and
//                     the block-diagonal collation of G_DataLoader (run.py:336).
//
// Everything is expressed as 64-bit key generation -> radix sort -> run detection -> scatter, so the
// result is deterministic and independent of edge order (integer work, bit-exact by construction).
// Where the reference rescans all E edges per node / per cluster (O(N·E)), this is O(E log) total.
#include "common.cuh"

namespace fitgnn {

constexpr int BT = 256;  // builder block size
static inline unsigned nblk(int64_t n) { return (unsigned)ceil_div(n > 0 ? n : 1, BT); }

enum { C_ERR = 0, C_DROP = 1, C_A = 2, C_B = 3, C_CURSOR = 4, C_N = 8 };

__device__ __forceinline__ int find_u64(const uint64_t* __restrict__ a, int lo, int hi, uint64_t key) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// ---------------------------------------------------------------------------------------------
// shared CSR finishers
// ---------------------------------------------------------------------------------------------
__global__ void csr_col_kernel(const uint64_t* __restrict__ keys, int64_t nnz, int32_t* __restrict__ col) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nnz) col[i] = (int32_t)(keys[i] & 0xffffffffull);
}
__global__ void dinv_kernel(const int32_t* __restrict__ rowptr, int64_t n, float* __restrict__ dinv) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int deg = rowptr[r + 1] - rowptr[r];
  // PyG: deg.pow(-0.5), inf -> 0.  1/sqrtf is correctly rounded division of a correctly rounded sqrt.
  dinv[r] = deg > 0 ? 1.0f / sqrtf((float)deg) : 0.f;
}
static int finish_csr(const uint64_t* keys, int64_t nnz, int64_t n_rows, int32_t* rowptr, int32_t* col, float* dinv,
                      cudaStream_t st) {
  csr_col_kernel<<<nblk(nnz), BT, 0, st>>>(keys, nnz, col);
  FG_LAUNCH_CHECK();
  FG_TRY(segment_ptr_from_sorted(keys, nnz, 32, n_rows, rowptr, st));
  dinv_kernel<<<nblk(n_rows), BT, 0, st>>>(rowptr, n_rows, dinv);
  FG_LAUNCH_CHECK();
  return FITGNN_OK;
}

// ---------------------------------------------------------------------------------------------
// generic CSR from COO (drop-in GCNConv path)
// ---------------------------------------------------------------------------------------------
__global__ void csr_keys_kernel(const int64_t* __restrict__ ei, int64_t E, int64_t n, uint64_t* __restrict__ keys,
                                int32_t* __restrict__ ctr) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E + n) return;
  if (e >= E) {
    const uint64_t v = (uint64_t)(e - E);
    keys[e] = (v << 32) | v;
    return;
  }
  const int64_t s = ei[e], d = ei[E + e];
  if (s < 0 || s >= n || d < 0 || d >= n) {
    atomicExch(&ctr[C_ERR], 1);
    atomicAdd(&ctr[C_DROP], 1);
    keys[e] = (uint64_t)n << 32;
  } else if (s == d) {
    atomicAdd(&ctr[C_DROP], 1);
    keys[e] = (uint64_t)n << 32;
  } else {
    keys[e] = ((uint64_t)d << 32) | (uint64_t)s;
  }
}

// ---------------------------------------------------------------------------------------------
// pack helpers
// ---------------------------------------------------------------------------------------------
__global__ void inverse_perm_kernel(const int32_t* __restrict__ members, int64_t N, int32_t* __restrict__ pos) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) pos[members[i]] = (int32_t)i;
}
__global__ void iota_kernel(int32_t* out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (int32_t)i;
}
__global__ void fill_u8_kernel(uint8_t* out, int64_t n, uint8_t v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = v;
}
__global__ void copy_i32_kernel(const int32_t* __restrict__ in, int32_t* __restrict__ out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i];
}
__global__ void self_keys_kernel(uint64_t* __restrict__ keys, int64_t n) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n) keys[r] = ((uint64_t)r << 32) | (uint64_t)r;
}

// mode none: intra-cluster edges -> (pos[dst] << 32 | pos[src]); everything else -> sentinel.
// KEYS_EPT edges per thread, every level of the dependent chain (edge -> part[] -> pos[]) issued for all of them before the
// next level is touched (the 1-edge version was latency-bound on the L2 gathers: 3.4 ms for 123 M edges); one counter
// atomic per warp.
constexpr int KEYS_EPT = 4;
__global__ void __launch_bounds__(BT)
none_keys_kernel(const int64_t* __restrict__ ei, int64_t E, int64_t N, const int32_t* __restrict__ part,
                 const int32_t* __restrict__ pos, uint64_t* __restrict__ keys, int32_t* __restrict__ ctr) {
  const int64_t base = (int64_t)blockIdx.x * (BT * KEYS_EPT) + threadIdx.x;
  int64_t u[KEYS_EPT], v[KEYS_EPT];
#pragma unroll
  for (int j = 0; j < KEYS_EPT; ++j) {
    const int64_t e = base + (int64_t)j * BT;
    u[j] = e < E ? ei[e] : 0;
    v[j] = e < E ? ei[E + e] : 0;
  }
  bool inr[KEYS_EPT];
  int32_t pu[KEYS_EPT], pv[KEYS_EPT];
  bool bad = false;
#pragma unroll
  for (int j = 0; j < KEYS_EPT; ++j) {
    const bool live = base + (int64_t)j * BT < E;
    inr[j] = live && u[j] >= 0 && u[j] < N && v[j] >= 0 && v[j] < N;
    bad |= live && !inr[j];
    pu[j] = inr[j] ? __ldg(part + u[j]) : 0;
    pv[j] = inr[j] ? __ldg(part + v[j]) : 0;
  }
  int32_t qu[KEYS_EPT], qv[KEYS_EPT];
  bool keep[KEYS_EPT];
#pragma unroll
  for (int j = 0; j < KEYS_EPT; ++j) {
    keep[j] = inr[j] && u[j] != v[j] && pu[j] == pv[j];
    qu[j] = keep[j] ? __ldg(pos + u[j]) : 0;
    qv[j] = keep[j] ? __ldg(pos + v[j]) : 0;
  }
  int n_drop = 0;
#pragma unroll
  for (int j = 0; j < KEYS_EPT; ++j) {
    const int64_t e = base + (int64_t)j * BT;
    if (e < E) {
      keys[e] = keep[j] ? ((uint64_t)(uint32_t)qv[j] << 32) | (uint64_t)(uint32_t)qu[j] : (uint64_t)N << 32;
      n_drop += keep[j] ? 0 : 1;
    }
  }
  if (bad) atomicExch(&ctr[C_ERR], 1);
  n_drop = __reduce_add_sync(0xffffffffu, n_drop);
  if ((threadIdx.x & 31) == 0 && n_drop) atomicAdd(&ctr[C_DROP], n_drop);
}

// mode extra, membership keys: (part[v], v) for every node and (part[u], v) for every cross edge u->v
__global__ void extra_member_keys_kernel(const int64_t* __restrict__ ei, int64_t E, int64_t N, int64_t k,
                                         const int32_t* __restrict__ part, uint64_t* __restrict__ keys,
                                         int32_t* __restrict__ ctr) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N + E) return;
  if (i < N) {
    keys[i] = ((uint64_t)part[i] << 32) | (uint64_t)i;
    return;
  }
  const int64_t e = i - N;
  const int64_t u = ei[e], v = ei[E + e];
  bool keep = false;
  if (u < 0 || u >= N || v < 0 || v >= N) atomicExch(&ctr[C_ERR], 1);
  else keep = part[u] != part[v];
  if (keep) keys[i] = ((uint64_t)part[u] << 32) | (uint64_t)v;
  else {
    keys[i] = (uint64_t)k << 32;
    atomicAdd(&ctr[C_DROP], 1);
  }
}

__global__ void unique_flags_kernel(const uint64_t* __restrict__ keys, int64_t n, int shift,
                                    int32_t* __restrict__ flags) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flags[i] = (i == 0 || (keys[i] >> shift) != (keys[i - 1] >> shift)) ? 1 : 0;
}
// compact the run starts (w.r.t. key >> shift) of keys[0..n) to out[pos]
__global__ void compact_unique_kernel(const uint64_t* __restrict__ keys, int64_t n, int shift,
                                      const int32_t* __restrict__ pos, uint64_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (i == 0 || (keys[i] >> shift) != (keys[i - 1] >> shift)) out[pos[i]] = keys[i];
}

// out-edge list keyed by source (self loops dropped): (src << 32 | dst)
__global__ void src_keys_kernel(const int64_t* __restrict__ ei, int64_t E, int64_t N, uint64_t* __restrict__ keys,
                                int32_t* __restrict__ ctr) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int64_t u = ei[e], v = ei[E + e];
  if (u < 0 || u >= N || v < 0 || v >= N || u == v) {
    keys[e] = (uint64_t)N << 32;
    atomicAdd(&ctr[C_A], 1);
  } else {
    keys[e] = ((uint64_t)u << 32) | (uint64_t)v;
  }
}

// mode extra, induced edges: warp per pack row r = (s, a); for every out-edge a->b with (s, b) a member,
// COUNT: cnt[r] = #found      FILL: keys[off[r] + rank] = (row(b) << 32 | r)
template <bool FILL>
__global__ void __launch_bounds__(BT)
extra_edges_kernel(const uint64_t* __restrict__ rowkeys, int64_t n_rows, const int32_t* __restrict__ sub_ptr,
                   const uint64_t* __restrict__ out_keys, const int32_t* __restrict__ out_ptr,
                   int32_t* __restrict__ cnt, const int32_t* __restrict__ off, uint64_t* __restrict__ keys) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * (BT / 32) + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  const uint64_t rk = rowkeys[r];
  const uint64_t s = rk >> 32;
  const int a = (int)(rk & 0xffffffffull);
  const int lo = sub_ptr[s], hi = sub_ptr[s + 1];
  const int beg = out_ptr[a], end = out_ptr[a + 1];
  int total = 0;
  for (int e0 = beg; e0 < end; e0 += 32) {
    const int e = e0 + lane;
    int found = -1;
    if (e < end) {
      const uint64_t want = (s << 32) | (out_keys[e] & 0xffffffffull);
      const int p = find_u64(rowkeys, lo, hi, want);
      if (p < hi && rowkeys[p] == want) found = p;
    }
    const unsigned m = __ballot_sync(0xffffffffu, found >= 0);
    if (FILL && found >= 0) {
      const int rank = total + __popc(m & ((1u << lane) - 1u));
      keys[(int64_t)off[r] + rank] = ((uint64_t)found << 32) | (uint64_t)r;
    }
    total += __popc(m);
  }
  if (!FILL && lane == 0) cnt[r] = total;
}

__global__ void extra_rows_kernel(const uint64_t* __restrict__ rowkeys, int64_t n_rows,
                                  const int32_t* __restrict__ sub_ptr, const int32_t* __restrict__ part,
                                  const int32_t* __restrict__ members, const int32_t* __restrict__ member_ptr,
                                  int32_t* __restrict__ gid, uint8_t* __restrict__ is_core,
                                  uint8_t* __restrict__ mask, int32_t* __restrict__ core_rows) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  const uint64_t rk = rowkeys[r];
  const int s = (int)(rk >> 32);
  const int v = (int)(rk & 0xffffffffull);
  gid[r] = v;
  const bool core = part[v] == s;
  is_core[r] = core ? 1 : 0;
  // utils.py:260-261: mask = [True]*n_core + [False]*n_ext over the RE-SORTED node list (positional quirk)
  const int n_core_s = member_ptr[s + 1] - member_ptr[s];
  mask[r] = ((int)r - sub_ptr[s]) < n_core_s ? 1 : 0;
  if (core) {
    int lo = member_ptr[s], hi = member_ptr[s + 1];
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (members[mid] < v) lo = mid + 1; else hi = mid;
    }
    core_rows[lo] = (int32_t)r;
  }
}

// ---- mode cluster -----------------------------------------------------------------------------
struct ClusterBits {
  int bk, bn;  // bits of a cluster id (0..k) and of a node id (0..N-1)
};

// cross edges u->v (part[u] != part[v]) -> (s, c, u) triples; intra edges are only counted
__global__ void cluster_tri_keys_kernel(const int64_t* __restrict__ ei, int64_t E, int64_t N, int64_t k,
                                        const int32_t* __restrict__ part, ClusterBits cb, uint64_t* __restrict__ keys,
                                        int32_t* __restrict__ ctr) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int64_t u = ei[e], v = ei[E + e];
  const uint64_t sentinel = (uint64_t)k << (cb.bk + cb.bn);
  if (u < 0 || u >= N || v < 0 || v >= N) {
    atomicExch(&ctr[C_ERR], 1);
    atomicAdd(&ctr[C_DROP], 1);
    keys[e] = sentinel;
    return;
  }
  const int s = part[u], c = part[v];
  if (s == c) {
    atomicAdd(&ctr[C_DROP], 1);
    if (u != v) atomicAdd(&ctr[C_A], 1);  // intra-cluster directed edge
    keys[e] = sentinel;
  } else {
    keys[e] = ((uint64_t)s << (cb.bk + cb.bn)) | ((uint64_t)c << cb.bn) | (uint64_t)u;
  }
}

// per unique triple: its pair index; per unique pair: (s,c) key, first-seen key (s, min u, c) and payload
__global__ void cluster_compact_kernel(const uint64_t* __restrict__ keys, int64_t n, ClusterBits cb,
                                       const int32_t* __restrict__ posT, const int32_t* __restrict__ posP,
                                       uint64_t* __restrict__ tri, int32_t* __restrict__ tri_pair,
                                       uint64_t* __restrict__ pair_sc, uint64_t* __restrict__ pair_order,
                                       uint32_t* __restrict__ pair_idx) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t key = keys[i];
  const bool newT = (i == 0) || key != keys[i - 1];
  const bool newP = (i == 0) || (key >> cb.bn) != (keys[i - 1] >> cb.bn);
  if (!newT) return;
  const int32_t p = posP[i] + (newP ? 1 : 0) - 1;
  tri[posT[i]] = key;
  tri_pair[posT[i]] = p;
  if (newP) {
    const uint64_t sc = key >> cb.bn;
    const uint64_t s = sc >> cb.bk, c = sc & ((1ull << cb.bk) - 1ull), u = key & ((1ull << cb.bn) - 1ull);
    pair_sc[p] = sc;
    pair_order[p] = (s << (cb.bk + cb.bn)) | (u << cb.bk) | c;  // utils.py:195-213 first-seen order
    pair_idx[p] = (uint32_t)p;
  }
}

__global__ void cluster_rank_kernel(const uint64_t* __restrict__ pair_order_sorted,
                                    const uint32_t* __restrict__ perm, int64_t Pn, ClusterBits cb,
                                    const int32_t* __restrict__ pstart, int32_t* __restrict__ cl_rank) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= Pn) return;
  const uint64_t s = pair_order_sorted[j] >> (cb.bk + cb.bn);
  cl_rank[perm[j]] = (int32_t)j - pstart[s];
}

__global__ void add_i32_kernel(const int32_t* __restrict__ a, const int32_t* __restrict__ b, int32_t* __restrict__ out,
                               int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = a[i] + b[i];
}

// cluster<->cluster edges: warp per pair i = (s, a); for b in Ac[a] with (s, b) also a pair j: edge i -> j
template <bool FILL>
__global__ void __launch_bounds__(BT)
cluster_cc_kernel(const uint64_t* __restrict__ pair_sc, int64_t Pn, ClusterBits cb, const int32_t* __restrict__ pstart,
                  const int32_t* __restrict__ ac_rowptr, const int32_t* __restrict__ ac_col,
                  const int32_t* __restrict__ sub_ptr, const int32_t* __restrict__ member_ptr,
                  const int32_t* __restrict__ cl_rank, int32_t* __restrict__ cnt, const int32_t* __restrict__ off,
                  uint64_t* __restrict__ keys) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * (BT / 32) + (threadIdx.x >> 5);
  if (i >= Pn) return;
  const uint64_t sc = pair_sc[i];
  const uint64_t s = sc >> cb.bk;
  const int a = (int)(sc & ((1ull << cb.bk) - 1ull));
  const int lo = pstart[s], hi = pstart[s + 1];
  const int beg = ac_rowptr[a], end = ac_rowptr[a + 1];
  const int row_base = sub_ptr[s] + (member_ptr[s + 1] - member_ptr[s]);
  const int row_i = row_base + cl_rank[i];
  int total = 0;
  for (int e0 = beg; e0 < end; e0 += 32) {
    const int e = e0 + lane;
    int found = -1;
    if (e < end) {
      const uint64_t want = (s << cb.bk) | (uint64_t)ac_col[e];
      const int p = find_u64(pair_sc, lo, hi, want);
      if (p < hi && pair_sc[p] == want) found = p;
    }
    const unsigned m = __ballot_sync(0xffffffffu, found >= 0);
    if (FILL && found >= 0) {
      const int rank = total + __popc(m & ((1u << lane) - 1u));
      const int row_j = row_base + cl_rank[found];
      keys[(int64_t)off[i] + rank] = ((uint64_t)row_j << 32) | (uint64_t)row_i;
    }
    total += __popc(m);
  }
  if (!FILL && lane == 0) cnt[i] = total;
}

// core<->core edges inside a cluster, written through an atomic cursor (order fixed later by the sort)
__global__ void cluster_intra_keys_kernel(const int64_t* __restrict__ ei, int64_t E, int64_t N,
                                          const int32_t* __restrict__ part, const int32_t* __restrict__ pos,
                                          const int32_t* __restrict__ member_ptr, const int32_t* __restrict__ sub_ptr,
                                          uint64_t* __restrict__ keys, int32_t* __restrict__ ctr) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int64_t u = ei[e], v = ei[E + e];
  if (u < 0 || u >= N || v < 0 || v >= N || u == v) return;
  const int s = part[u];
  if (s != part[v]) return;
  const int base = sub_ptr[s] - member_ptr[s];
  const int slot = atomicAdd(&ctr[C_CURSOR], 1);
  keys[slot] = ((uint64_t)(base + pos[v]) << 32) | (uint64_t)(base + pos[u]);
}

// node<->cluster-node edges, both directions, once per unique (s, c, u) triple (utils.py:214-222)
__global__ void cluster_nc_keys_kernel(const uint64_t* __restrict__ tri, const int32_t* __restrict__ tri_pair,
                                       int64_t T, ClusterBits cb, const int32_t* __restrict__ pos,
                                       const int32_t* __restrict__ member_ptr, const int32_t* __restrict__ sub_ptr,
                                       const int32_t* __restrict__ cl_rank, uint64_t* __restrict__ keys) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const uint64_t key = tri[t];
  const uint64_t s = key >> (cb.bk + cb.bn);
  const int u = (int)(key & ((1ull << cb.bn) - 1ull));
  const int ru = sub_ptr[s] - member_ptr[s] + pos[u];
  const int rc = sub_ptr[s] + (member_ptr[s + 1] - member_ptr[s]) + cl_rank[tri_pair[t]];
  keys[2 * t] = ((uint64_t)rc << 32) | (uint64_t)ru;      // node -> cluster node
  keys[2 * t + 1] = ((uint64_t)ru << 32) | (uint64_t)rc;  // cluster node -> node
}

__global__ void cluster_rows_kernel(int64_t N, int64_t Pn, ClusterBits cb, const int32_t* __restrict__ members,
                                    const int32_t* __restrict__ part, const int32_t* __restrict__ member_ptr,
                                    const int32_t* __restrict__ sub_ptr, const uint64_t* __restrict__ pair_sc,
                                    const int32_t* __restrict__ cl_rank, int32_t* __restrict__ gid,
                                    uint8_t* __restrict__ is_core, uint8_t* __restrict__ mask,
                                    int32_t* __restrict__ core_rows) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) {  // i-th node in (part, id) order
    const int v = members[i];
    const int s = part[v];
    const int r = sub_ptr[s] - member_ptr[s] + (int)i;
    gid[r] = v;
    is_core[r] = 1;
    mask[r] = 1;  // utils.py:262-263: positional mask is correct in cluster mode
    core_rows[i] = r;
  } else if (i < N + Pn) {
    const int64_t p = i - N;
    const uint64_t sc = pair_sc[p];
    const uint64_t s = sc >> cb.bk;
    const int c = (int)(sc & ((1ull << cb.bk) - 1ull));
    const int r = sub_ptr[s] + (member_ptr[s + 1] - member_ptr[s]) + cl_rank[p];
    gid[r] = (int32_t)(N + c);
    is_core[r] = 0;
    mask[r] = 0;
  }
}

}  // namespace fitgnn

using namespace fitgnn;

// =================================================================================================
// generic CSR
// =================================================================================================
extern "C" size_t fitgnn_csr_workspace_bytes(int64_t E, int64_t n) {
  const int64_t m = (E > 0 ? E : 0) + (n > 0 ? n : 0) + 1;
  return 1024 + align_up((size_t)m * 8) + sort_ws_bytes(m);
}

extern "C" int fitgnn_csr_plan(const int64_t* edge_index, int64_t E, int64_t n, void* ws, size_t ws_bytes,
                               int64_t* host_nnz, void* stream) {
  FG_REQUIRE(E >= 0 && n >= 0 && ws && host_nnz && (E == 0 || edge_index), FITGNN_EINVAL, "csr_plan: bad arguments");
  FG_REQUIRE(E + n < (1ll << 31) - 8192, FITGNN_ERANGE, "csr_plan: E + n = %lld exceeds int32 indexing",
             (long long)(E + n));
  cudaStream_t st = as_stream(stream);
  Bump b(ws, ws_bytes);
  int32_t* ctr = b.take<int32_t>(C_N);
  uint64_t* keys = b.take<uint64_t>((size_t)(E + n + 1));
  FG_REQUIRE(b.ok, FITGNN_EWS, "csr_plan: workspace too small");
  FG_CUDA(cudaMemsetAsync(ctr, 0, C_N * sizeof(int32_t), st));
  if (E + n > 0) {
    csr_keys_kernel<<<nblk(E + n), BT, 0, st>>>(edge_index, E, n, keys, ctr);
    FG_LAUNCH_CHECK();
    FG_TRY(sort_u64_mask(keys, nullptr, E + n, field_mask((uint64_t)n, (uint64_t)n), b.here(), b.left(), st));
  }
  int32_t h[C_N];
  FG_CUDA(cudaMemcpyAsync(h, ctr, sizeof(h), cudaMemcpyDeviceToHost, st));
  FG_CUDA(cudaStreamSynchronize(st));
  FG_REQUIRE(h[C_ERR] == 0, FITGNN_EINVAL, "csr_plan: edge_index holds node ids outside [0,%lld)", (long long)n);
  *host_nnz = E + n - h[C_DROP];
  // remember the sizes for the fill call in the (otherwise unused) tail of the counter block
  const int64_t dims[2] = {E, *host_nnz};
  FG_CUDA(cudaMemcpyAsync(ctr + 4, dims, sizeof(dims), cudaMemcpyHostToDevice, st));  // 4 int32 = 2 int64
  FG_CUDA(cudaStreamSynchronize(st));
  return FITGNN_OK;
}

extern "C" int fitgnn_csr_fill(int64_t n, void* ws, size_t ws_bytes, int32_t* rowptr, int32_t* col, float* dinv,
                               void* stream) {
  FG_REQUIRE(n >= 0 && ws && rowptr && dinv, FITGNN_EINVAL, "csr_fill: bad arguments");
  cudaStream_t st = as_stream(stream);
  Bump b(ws, ws_bytes);
  int32_t* ctr = b.take<int32_t>(C_N);
  int64_t dims[2];
  FG_CUDA(cudaMemcpyAsync(dims, ctr + 4, sizeof(dims), cudaMemcpyDeviceToHost, st));
  FG_CUDA(cudaStreamSynchronize(st));
  const int64_t E = dims[0], nnz = dims[1];
  uint64_t* keys = b.take<uint64_t>((size_t)(E + n + 1));
  FG_REQUIRE(b.ok, FITGNN_EWS, "csr_fill: workspace too small");
  FG_REQUIRE(nnz == 0 || col, FITGNN_EINVAL, "csr_fill: null col");
  return finish_csr(keys, nnz, n, rowptr, col, dinv, st);
}

// =================================================================================================
// raw CSR (drop-in SAGEConv path): the edges exactly as given — self loops kept, none added, duplicates kept
// =================================================================================================
namespace fitgnn {
__global__ void csr_raw_keys_kernel(const int64_t* __restrict__ ei, int64_t E, int64_t n, uint64_t* __restrict__ keys,
                                    int32_t* __restrict__ ctr) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int64_t s = ei[e], d = ei[E + e];
  if (s < 0 || s >= n || d < 0 || d >= n) {
    atomicExch(&ctr[C_ERR], 1);
    atomicAdd(&ctr[C_DROP], 1);
    keys[e] = (uint64_t)n << 32;
  } else {
    keys[e] = ((uint64_t)d << 32) | (uint64_t)s;
  }
}
}  // namespace fitgnn

extern "C" int fitgnn_csr_raw_plan(const int64_t* edge_index, int64_t E, int64_t n, void* ws, size_t ws_bytes,
                                   int64_t* host_nnz, void* stream) {
  FG_REQUIRE(E >= 0 && n >= 0 && ws && host_nnz && (E == 0 || edge_index), FITGNN_EINVAL, "csr_raw_plan: bad arguments");
  FG_REQUIRE(E + n < (1ll << 31) - 8192, FITGNN_ERANGE, "csr_raw_plan: E + n = %lld exceeds int32 indexing",
             (long long)(E + n));
  cudaStream_t st = as_stream(stream);
  Bump b(ws, ws_bytes);
  int32_t* ctr = b.take<int32_t>(C_N);
  uint64_t* keys = b.take<uint64_t>((size_t)(E + n + 1));  // same layout as fitgnn_csr_plan (workspace size shared)
  FG_REQUIRE(b.ok, FITGNN_EWS, "csr_raw_plan: workspace too small");
  FG_CUDA(cudaMemsetAsync(ctr, 0, C_N * sizeof(int32_t), st));
  if (E > 0) {
    csr_raw_keys_kernel<<<nblk(E), BT, 0, st>>>(edge_index, E, n, keys, ctr);
    FG_LAUNCH_CHECK();
    FG_TRY(sort_u64_mask(keys, nullptr, E, field_mask((uint64_t)n, (uint64_t)n), b.here(), b.left(), st));
  }
  int32_t h[C_N];
  FG_CUDA(cudaMemcpyAsync(h, ctr, sizeof(h), cudaMemcpyDeviceToHost, st));
  FG_CUDA(cudaStreamSynchronize(st));
  FG_REQUIRE(h[C_ERR] == 0, FITGNN_EINVAL, "csr_raw_plan: edge_index holds node ids outside [0,%lld)", (long long)n);
  *host_nnz = E;
  const int64_t dims[2] = {E, E};
  FG_CUDA(cudaMemcpyAsync(ctr + 4, dims, sizeof(dims), cudaMemcpyHostToDevice, st));
  FG_CUDA(cudaStreamSynchronize(st));
  return FITGNN_OK;
}

extern "C" int fitgnn_csr_raw_fill(int64_t n, void* ws, size_t ws_bytes, int32_t* rowptr, int32_t* col, void* stream) {
  FG_REQUIRE(n >= 0 && ws && rowptr, FITGNN_EINVAL, "csr_raw_fill: bad arguments");
  cudaStream_t st = as_stream(stream);
  Bump b(ws, ws_bytes);
  int32_t* ctr = b.take<int32_t>(C_N);
  int64_t dims[2];
  FG_CUDA(cudaMemcpyAsync(dims, ctr + 4, sizeof(dims), cudaMemcpyDeviceToHost, st));
  FG_CUDA(cudaStreamSynchronize(st));
  const int64_t E = dims[0], nnz = dims[1];
  uint64_t* keys = b.take<uint64_t>((size_t)(E + n + 1));
  FG_REQUIRE(b.ok, FITGNN_EWS, "csr_raw_fill: workspace too small");
  FG_REQUIRE(nnz == 0 || col, FITGNN_EINVAL, "csr_raw_fill: null col");
  csr_col_kernel<<<nblk(nnz), BT, 0, st>>>(keys, nnz, col);
  FG_LAUNCH_CHECK();
  return segment_ptr_from_sorted(keys, nnz, 32, n, rowptr, st);
}

// =================================================================================================
// pack builder
// =================================================================================================
namespace {

// workspace layout shared by plan and fill (recomputed identically in both from E, N, k, mode)
struct PackWs {
  int32_t* ctr;
  int32_t *members, *member_ptr, *pos;  // nodes grouped by (part, id); pos = inverse permutation
  // none
  uint64_t* keys;  // [E + N]
  // extra
  uint64_t* mkeys;      // [N + E] membership keys, then compacted in place into rowkeys
  int32_t* mflags;      // [N + E + 1]
  uint64_t* rowkeys;    // [N + E]
  int32_t* sub_ptr;     // [k + 1]
  uint64_t* out_keys;   // [E] (src, dst) sorted
  int32_t* out_ptr;     // [N + 1]
  int32_t* cnt;         // [N + E + 1] -> offsets
  // cluster
  uint64_t* tkeys;      // [E]
  int32_t *posT, *posP; // [E + 1]
  uint64_t* tri;        // [E]
  int32_t* tri_pair;    // [E]
  uint64_t *pair_sc, *pair_order;  // [E]
  uint32_t* pair_idx;   // [E]
  int32_t *pstart, *cl_rank, *ccnt;  // [k+1], [E], [E+1]
  void* scratch;
  size_t scratch_bytes;
  bool ok;
};

size_t pack_scratch_bytes(int64_t E, int64_t N) { return sort_ws_bytes(E + N + 1) + scan_ws_bytes(E + N + 2) + 1024; }

PackWs carve(void* ws, size_t ws_bytes, int64_t E, int64_t N, int64_t k, int mode) {
  PackWs w{};
  Bump b(ws, ws_bytes);
  const size_t e = (size_t)E + 1, n = (size_t)N + 1, kk = (size_t)k + 2;
  w.ctr = b.take<int32_t>(C_N);
  w.members = b.take<int32_t>(n);
  w.member_ptr = b.take<int32_t>(kk);
  w.pos = b.take<int32_t>(n);
  if (mode == FITGNN_MODE_NONE) {
    w.keys = b.take<uint64_t>(e + n);
  } else if (mode == FITGNN_MODE_EXTRA) {
    w.mkeys = b.take<uint64_t>(e + n);
    w.mflags = b.take<int32_t>(e + n + 1);
    w.rowkeys = b.take<uint64_t>(e + n);
    w.sub_ptr = b.take<int32_t>(kk);
    w.out_keys = b.take<uint64_t>(e);
    w.out_ptr = b.take<int32_t>(n + 1);
    w.cnt = b.take<int32_t>(e + n + 1);
  } else {
    w.tkeys = b.take<uint64_t>(e);
    w.posT = b.take<int32_t>(e + 1);
    w.posP = b.take<int32_t>(e + 1);
    w.tri = b.take<uint64_t>(e);
    w.tri_pair = b.take<int32_t>(e);
    w.pair_sc = b.take<uint64_t>(e);
    w.pair_order = b.take<uint64_t>(e);
    w.pair_idx = b.take<uint32_t>(e);
    w.pstart = b.take<int32_t>(kk);
    w.cl_rank = b.take<int32_t>(e);
    w.ccnt = b.take<int32_t>(e + 1);
    w.sub_ptr = b.take<int32_t>(kk);
  }
  w.scratch = b.here();
  w.scratch_bytes = b.left();
  w.ok = b.ok && w.scratch_bytes >= pack_scratch_bytes(E, N);
  return w;
}

size_t carve_bytes(int64_t E, int64_t N, int64_t k, int mode) {
  // run the bump allocator over a fake huge region to measure the fixed part
  Bump b(nullptr, (size_t)1 << 62);
  const size_t e = (size_t)E + 1, n = (size_t)N + 1, kk = (size_t)k + 2;
  b.take<int32_t>(C_N); b.take<int32_t>(n); b.take<int32_t>(kk); b.take<int32_t>(n);
  if (mode == FITGNN_MODE_NONE) {
    b.take<uint64_t>(e + n);
  } else if (mode == FITGNN_MODE_EXTRA) {
    b.take<uint64_t>(e + n); b.take<int32_t>(e + n + 1); b.take<uint64_t>(e + n); b.take<int32_t>(kk);
    b.take<uint64_t>(e); b.take<int32_t>(n + 1); b.take<int32_t>(e + n + 1);
  } else {
    b.take<uint64_t>(e); b.take<int32_t>(e + 1); b.take<int32_t>(e + 1); b.take<uint64_t>(e); b.take<int32_t>(e);
    b.take<uint64_t>(e); b.take<uint64_t>(e); b.take<uint32_t>(e); b.take<int32_t>(kk); b.take<int32_t>(e);
    b.take<int32_t>(e + 1); b.take<int32_t>(kk);
  }
  return b.off;
}

int read_ctr(const int32_t* ctr, int32_t* h, cudaStream_t st) {
  FG_CUDA(cudaMemcpyAsync(h, ctr, C_N * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  FG_CUDA(cudaStreamSynchronize(st));
  return FITGNN_OK;
}
int read_i32(const int32_t* p, int32_t* h, cudaStream_t st) {
  FG_CUDA(cudaMemcpyAsync(h, p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  FG_CUDA(cudaStreamSynchronize(st));
  return FITGNN_OK;
}

}  // namespace

extern "C" size_t fitgnn_pack_workspace_bytes(int64_t E, int64_t N, int64_t k, int mode, int64_t ac_nnz) {
  (void)ac_nnz;
  if (E < 0) E = 0;
  if (N < 0) N = 0;
  if (k < 0) k = 0;
  return carve_bytes(E, N, k, mode) + pack_scratch_bytes(E, N) + fitgnn_group_workspace_bytes(N, k) + 4096;
}

// priv[] slots of fitgnn_plan
enum { P_E = 0, P_N, P_K, P_MODE, P_EI, P_PART, P_ACP, P_ACC, P_T, P_PN, P_NINTRA, P_NCC, P_EPRIME, P_BK, P_BN };

extern "C" int fitgnn_pack_plan(const int64_t* edge_index, int64_t E, int64_t N, const int32_t* part, int64_t k,
                                int mode, const int32_t* ac_rowptr, const int32_t* ac_col, int64_t ac_nnz, void* ws,
                                size_t ws_bytes, fitgnn_plan* plan, void* stream) {
  FG_REQUIRE(plan && ws && part && E >= 0 && N > 0 && k > 0 && (E == 0 || edge_index), FITGNN_EINVAL,
             "pack_plan: bad arguments");
  FG_REQUIRE(mode == FITGNN_MODE_NONE || mode == FITGNN_MODE_EXTRA || mode == FITGNN_MODE_CLUSTER, FITGNN_EINVAL,
             "pack_plan: unknown mode %d", mode);
  FG_REQUIRE(mode != FITGNN_MODE_CLUSTER || (ac_rowptr && (ac_nnz == 0 || ac_col)), FITGNN_EINVAL,
             "pack_plan: cluster mode needs the coarsened adjacency (ac_rowptr/ac_col)");
  FG_REQUIRE(E + N < (1ll << 31) - 16384 && k < (1ll << 31), FITGNN_ERANGE, "pack_plan: E + N exceeds int32 indexing");
  cudaStream_t st = as_stream(stream);
  PackWs w = carve(ws, ws_bytes, E, N, k, mode);
  FG_REQUIRE(w.ok, FITGNN_EWS, "pack_plan: workspace too small (%zu bytes)", ws_bytes);
  for (int i = 0; i < 27; ++i) plan->priv[i] = 0;
  plan->priv[P_E] = E; plan->priv[P_N] = N; plan->priv[P_K] = k; plan->priv[P_MODE] = mode;
  plan->priv[P_EI] = (int64_t)(uintptr_t)edge_index; plan->priv[P_PART] = (int64_t)(uintptr_t)part;
  plan->priv[P_ACP] = (int64_t)(uintptr_t)ac_rowptr; plan->priv[P_ACC] = (int64_t)(uintptr_t)ac_col;
  plan->fill_ws_bytes = 0;

  FG_CUDA(cudaMemsetAsync(w.ctr, 0, C_N * sizeof(int32_t), st));
  FG_TRY(fitgnn_group_by_part(part, N, k, w.members, w.member_ptr, w.scratch, w.scratch_bytes, stream));
  inverse_perm_kernel<<<nblk(N), BT, 0, st>>>(w.members, N, w.pos);
  FG_LAUNCH_CHECK();
  int32_t h[C_N];

  if (mode == FITGNN_MODE_NONE) {
    if (E > 0) {
      none_keys_kernel<<<(unsigned)ceil_div(E, (int64_t)BT * KEYS_EPT), BT, 0, st>>>(edge_index, E, N, part, w.pos, w.keys, w.ctr);
      FG_LAUNCH_CHECK();
    }
    self_keys_kernel<<<nblk(N), BT, 0, st>>>(w.keys + E, N);
    FG_LAUNCH_CHECK();
    FG_TRY(sort_u64_mask(w.keys, nullptr, E + N, field_mask((uint64_t)N, (uint64_t)N), w.scratch, w.scratch_bytes, st));
    FG_TRY(read_ctr(w.ctr, h, st));
    FG_REQUIRE(h[C_ERR] == 0, FITGNN_EINVAL, "pack_plan: edge_index holds node ids outside [0,%lld)", (long long)N);
    plan->n_rows = N; plan->nnz = E + N - h[C_DROP]; plan->n_sub = k; plan->n_core = N; plan->n_src = N;
    return FITGNN_OK;
  }

  if (mode == FITGNN_MODE_EXTRA) {
    const int64_t M = N + E;
    extra_member_keys_kernel<<<nblk(M), BT, 0, st>>>(edge_index, E, N, k, part, w.mkeys, w.ctr);
    FG_LAUNCH_CHECK();
    FG_TRY(sort_u64_mask(w.mkeys, nullptr, M, field_mask((uint64_t)k, (uint64_t)N), w.scratch, w.scratch_bytes, st));
    FG_TRY(read_ctr(w.ctr, h, st));
    FG_REQUIRE(h[C_ERR] == 0, FITGNN_EINVAL, "pack_plan: edge_index holds node ids outside [0,%lld)", (long long)N);
    const int64_t n_valid = M - h[C_DROP];
    unique_flags_kernel<<<nblk(n_valid), BT, 0, st>>>(w.mkeys, n_valid, 0, w.mflags);
    FG_LAUNCH_CHECK();
    FG_TRY(scan_i32(w.mflags, n_valid, w.mflags, n_valid + 1, w.scratch, w.scratch_bytes, st));
    int32_t n_rows = 0;
    FG_TRY(read_i32(w.mflags + n_valid, &n_rows, st));
    compact_unique_kernel<<<nblk(n_valid), BT, 0, st>>>(w.mkeys, n_valid, 0, w.mflags, w.rowkeys);
    FG_LAUNCH_CHECK();
    FG_TRY(segment_ptr_from_sorted(w.rowkeys, n_rows, 32, k, w.sub_ptr, st));
    // out-edge CSR of the original graph
    int64_t E2 = 0;
    if (E > 0) {
      src_keys_kernel<<<nblk(E), BT, 0, st>>>(edge_index, E, N, w.out_keys, w.ctr);
      FG_LAUNCH_CHECK();
      FG_TRY(sort_u64_mask(w.out_keys, nullptr, E, field_mask((uint64_t)N, (uint64_t)N), w.scratch, w.scratch_bytes, st));
      FG_TRY(read_ctr(w.ctr, h, st));
      E2 = E - h[C_A];
    }
    FG_TRY(segment_ptr_from_sorted(w.out_keys, E2, 32, N, w.out_ptr, st));
    extra_edges_kernel<false><<<(unsigned)ceil_div(n_rows, BT / 32), BT, 0, st>>>(
        w.rowkeys, n_rows, w.sub_ptr, w.out_keys, w.out_ptr, w.cnt, nullptr, nullptr);
    FG_LAUNCH_CHECK();
    FG_TRY(scan_i32(w.cnt, n_rows, w.cnt, n_rows + 1, w.scratch, w.scratch_bytes, st));
    int32_t e_prime = 0;
    FG_TRY(read_i32(w.cnt + n_rows, &e_prime, st));
    plan->n_rows = n_rows; plan->nnz = (int64_t)e_prime + n_rows; plan->n_sub = k; plan->n_core = N; plan->n_src = N;
    plan->priv[P_EPRIME] = e_prime;
    FG_REQUIRE(plan->nnz < (1ll << 31) - 16384, FITGNN_ERANGE, "pack_plan: nnz = %lld exceeds int32 indexing",
               (long long)plan->nnz);
    plan->fill_ws_bytes = (int64_t)(align_up((size_t)(plan->nnz + 1) * 8) + sort_ws_bytes(plan->nnz) + 1024);
    return FITGNN_OK;
  }

  // ---- cluster ----
  ClusterBits cb{bits_for((uint64_t)k), bits_for((uint64_t)(N > 1 ? N - 1 : 1))};
  FG_REQUIRE(2 * cb.bk + cb.bn <= 64, FITGNN_ERANGE,
             "pack_plan: (cluster, cluster, node) key needs %d bits > 64 (k=%lld, N=%lld)", 2 * cb.bk + cb.bn,
             (long long)k, (long long)N);
  plan->priv[P_BK] = cb.bk; plan->priv[P_BN] = cb.bn;
  int64_t T = 0, Pn = 0, n_intra = 0, n_cc = 0;
  if (E > 0) {
    cluster_tri_keys_kernel<<<nblk(E), BT, 0, st>>>(edge_index, E, N, k, part, cb, w.tkeys, w.ctr);
    FG_LAUNCH_CHECK();
    FG_TRY(sort_u64(w.tkeys, nullptr, E, 2 * cb.bk + cb.bn, w.scratch, w.scratch_bytes, st));
    FG_TRY(read_ctr(w.ctr, h, st));
    FG_REQUIRE(h[C_ERR] == 0, FITGNN_EINVAL, "pack_plan: edge_index holds node ids outside [0,%lld)", (long long)N);
    const int64_t n_cross = E - h[C_DROP];
    n_intra = h[C_A];
    if (n_cross > 0) {
      unique_flags_kernel<<<nblk(n_cross), BT, 0, st>>>(w.tkeys, n_cross, 0, w.posT);
      FG_LAUNCH_CHECK();
      unique_flags_kernel<<<nblk(n_cross), BT, 0, st>>>(w.tkeys, n_cross, cb.bn, w.posP);
      FG_LAUNCH_CHECK();
      FG_TRY(scan_i32(w.posT, n_cross, w.posT, n_cross + 1, w.scratch, w.scratch_bytes, st));
      FG_TRY(scan_i32(w.posP, n_cross, w.posP, n_cross + 1, w.scratch, w.scratch_bytes, st));
      int32_t t32 = 0, p32 = 0;
      FG_TRY(read_i32(w.posT + n_cross, &t32, st));
      FG_TRY(read_i32(w.posP + n_cross, &p32, st));
      T = t32; Pn = p32;
      cluster_compact_kernel<<<nblk(n_cross), BT, 0, st>>>(w.tkeys, n_cross, cb, w.posT, w.posP, w.tri, w.tri_pair,
                                                           w.pair_sc, w.pair_order, w.pair_idx);
      FG_LAUNCH_CHECK();
    }
  }
  FG_TRY(segment_ptr_from_sorted(w.pair_sc, Pn, cb.bk, k, w.pstart, st));
  if (Pn > 0) {
    FG_TRY(sort_u64(w.pair_order, w.pair_idx, Pn, 2 * cb.bk + cb.bn, w.scratch, w.scratch_bytes, st));
    cluster_rank_kernel<<<nblk(Pn), BT, 0, st>>>(w.pair_order, w.pair_idx, Pn, cb, w.pstart, w.cl_rank);
    FG_LAUNCH_CHECK();
  }
  add_i32_kernel<<<nblk(k + 1), BT, 0, st>>>(w.member_ptr, w.pstart, w.sub_ptr, k + 1);
  FG_LAUNCH_CHECK();
  if (Pn > 0) {
    cluster_cc_kernel<false><<<(unsigned)ceil_div(Pn, BT / 32), BT, 0, st>>>(
        w.pair_sc, Pn, cb, w.pstart, ac_rowptr, ac_col, w.sub_ptr, w.member_ptr, w.cl_rank, w.ccnt, nullptr, nullptr);
    FG_LAUNCH_CHECK();
    FG_TRY(scan_i32(w.ccnt, Pn, w.ccnt, Pn + 1, w.scratch, w.scratch_bytes, st));
    int32_t c32 = 0;
    FG_TRY(read_i32(w.ccnt + Pn, &c32, st));
    n_cc = c32;
  }
  plan->n_rows = N + Pn; plan->n_sub = k; plan->n_core = N; plan->n_src = N + k;
  plan->nnz = n_intra + 2 * T + n_cc + plan->n_rows;
  plan->priv[P_T] = T; plan->priv[P_PN] = Pn; plan->priv[P_NINTRA] = n_intra; plan->priv[P_NCC] = n_cc;
  FG_REQUIRE(plan->nnz < (1ll << 31) - 16384 && plan->n_rows < (1ll << 31) - 16384, FITGNN_ERANGE,
             "pack_plan: nnz = %lld exceeds int32 indexing", (long long)plan->nnz);
  plan->fill_ws_bytes = (int64_t)(align_up((size_t)(plan->nnz + 1) * 8) + sort_ws_bytes(plan->nnz) + 1024);
  return FITGNN_OK;
}

extern "C" int fitgnn_pack_fill(const fitgnn_plan* plan, const fitgnn_pack* out, void* ws, size_t ws_bytes, void* ws2,
                                size_t ws2_bytes, void* stream) {
  FG_REQUIRE(plan && out && ws, FITGNN_EINVAL, "pack_fill: bad arguments");
  FG_REQUIRE(out->rowptr && out->col && out->dinv && out->gid && out->sub_ptr && out->core_rows && out->is_core &&
                 out->mask, FITGNN_EINVAL, "pack_fill: pack arrays must be allocated by the caller");
  FG_REQUIRE(out->n_rows == plan->n_rows && out->nnz == plan->nnz && out->n_sub == plan->n_sub &&
                 out->n_core == plan->n_core, FITGNN_EINVAL, "pack_fill: pack sizes do not match the plan");
  cudaStream_t st = as_stream(stream);
  const int64_t E = plan->priv[P_E], N = plan->priv[P_N], k = plan->priv[P_K];
  const int mode = (int)plan->priv[P_MODE];
  const int64_t* ei = reinterpret_cast<const int64_t*>((uintptr_t)plan->priv[P_EI]);
  const int32_t* part = reinterpret_cast<const int32_t*>((uintptr_t)plan->priv[P_PART]);
  PackWs w = carve(ws, ws_bytes, E, N, k, mode);
  FG_REQUIRE(w.ok, FITGNN_EWS, "pack_fill: workspace too small");
  int32_t* rowptr = const_cast<int32_t*>(out->rowptr);
  int32_t* col = const_cast<int32_t*>(out->col);
  float* dinv = const_cast<float*>(out->dinv);
  int32_t* gid = const_cast<int32_t*>(out->gid);
  int32_t* sub_ptr = const_cast<int32_t*>(out->sub_ptr);
  int32_t* core_rows = const_cast<int32_t*>(out->core_rows);
  uint8_t* is_core = const_cast<uint8_t*>(out->is_core);
  uint8_t* mask = const_cast<uint8_t*>(out->mask);
  const int64_t n_rows = plan->n_rows, nnz = plan->nnz;

  if (mode == FITGNN_MODE_NONE) {
    FG_TRY(finish_csr(w.keys, nnz, n_rows, rowptr, col, dinv, st));
    copy_i32_kernel<<<nblk(N), BT, 0, st>>>(w.members, gid, N);
    copy_i32_kernel<<<nblk(k + 1), BT, 0, st>>>(w.member_ptr, sub_ptr, k + 1);
    iota_kernel<<<nblk(N), BT, 0, st>>>(core_rows, N);
    fill_u8_kernel<<<nblk(N), BT, 0, st>>>(is_core, N, 1);
    fill_u8_kernel<<<nblk(N), BT, 0, st>>>(mask, N, 1);
    FG_LAUNCH_CHECK();
    return FITGNN_OK;
  }

  FG_REQUIRE(ws2 && ws2_bytes >= (size_t)plan->fill_ws_bytes, FITGNN_EWS,
             "pack_fill: second workspace needs %lld bytes", (long long)plan->fill_ws_bytes);
  Bump b2(ws2, ws2_bytes);
  uint64_t* keys = b2.take<uint64_t>((size_t)nnz + 1);
  FG_REQUIRE(b2.ok, FITGNN_EWS, "pack_fill: second workspace too small");

  if (mode == FITGNN_MODE_EXTRA) {
    const int64_t e_prime = plan->priv[P_EPRIME];
    extra_edges_kernel<true><<<(unsigned)ceil_div(n_rows, BT / 32), BT, 0, st>>>(
        w.rowkeys, n_rows, w.sub_ptr, w.out_keys, w.out_ptr, nullptr, w.cnt, keys);
    FG_LAUNCH_CHECK();
    self_keys_kernel<<<nblk(n_rows), BT, 0, st>>>(keys + e_prime, n_rows);
    FG_LAUNCH_CHECK();
    FG_TRY(sort_u64_mask(keys, nullptr, nnz, field_mask((uint64_t)n_rows, (uint64_t)n_rows), b2.here(), b2.left(), st));
    FG_TRY(finish_csr(keys, nnz, n_rows, rowptr, col, dinv, st));
    copy_i32_kernel<<<nblk(k + 1), BT, 0, st>>>(w.sub_ptr, sub_ptr, k + 1);
    extra_rows_kernel<<<nblk(n_rows), BT, 0, st>>>(w.rowkeys, n_rows, w.sub_ptr, part, w.members, w.member_ptr, gid,
                                                   is_core, mask, core_rows);
    FG_LAUNCH_CHECK();
    return FITGNN_OK;
  }

  // ---- cluster ----
  ClusterBits cb{(int)plan->priv[P_BK], (int)plan->priv[P_BN]};
  const int64_t T = plan->priv[P_T], Pn = plan->priv[P_PN], n_intra = plan->priv[P_NINTRA], n_cc = plan->priv[P_NCC];
  const int32_t* ac_rowptr = reinterpret_cast<const int32_t*>((uintptr_t)plan->priv[P_ACP]);
  const int32_t* ac_col = reinterpret_cast<const int32_t*>((uintptr_t)plan->priv[P_ACC]);
  FG_CUDA(cudaMemsetAsync(w.ctr + C_CURSOR, 0, sizeof(int32_t), st));
  if (E > 0) {
    cluster_intra_keys_kernel<<<nblk(E), BT, 0, st>>>(ei, E, N, part, w.pos, w.member_ptr, w.sub_ptr, keys, w.ctr);
    FG_LAUNCH_CHECK();
  }
  if (T > 0) {
    cluster_nc_keys_kernel<<<nblk(T), BT, 0, st>>>(w.tri, w.tri_pair, T, cb, w.pos, w.member_ptr, w.sub_ptr, w.cl_rank,
                                                   keys + n_intra);
    FG_LAUNCH_CHECK();
  }
  if (Pn > 0 && n_cc > 0) {
    cluster_cc_kernel<true><<<(unsigned)ceil_div(Pn, BT / 32), BT, 0, st>>>(
        w.pair_sc, Pn, cb, w.pstart, ac_rowptr, ac_col, w.sub_ptr, w.member_ptr, w.cl_rank, nullptr, w.ccnt,
        keys + n_intra + 2 * T);
    FG_LAUNCH_CHECK();
  }
  self_keys_kernel<<<nblk(n_rows), BT, 0, st>>>(keys + n_intra + 2 * T + n_cc, n_rows);
  FG_LAUNCH_CHECK();
  FG_TRY(sort_u64_mask(keys, nullptr, nnz, field_mask((uint64_t)n_rows, (uint64_t)n_rows), b2.here(), b2.left(), st));
  FG_TRY(finish_csr(keys, nnz, n_rows, rowptr, col, dinv, st));
  copy_i32_kernel<<<nblk(k + 1), BT, 0, st>>>(w.sub_ptr, sub_ptr, k + 1);
  cluster_rows_kernel<<<nblk(N + Pn), BT, 0, st>>>(N, Pn, cb, w.members, part, w.member_ptr, w.sub_ptr, w.pair_sc,
                                                   w.cl_rank, gid, is_core, mask, core_rows);
  FG_LAUNCH_CHECK();
  return FITGNN_OK;
}
