// tlc_common.cuh -- shared device-side definitions for the sm_100a kernels of the vicinity
// persistence path.  One CTA ("team") works on one target at a time; every per-target array lives in
// a chunk arena in HBM (SoA, addressed through per-target offsets), hot per-vertex state is staged in
// shared memory when it fits.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/tlc_b200.h"

namespace tlc {

struct GraphView {
  int32_t N;
  int64_t nnz;
  const int32_t* rowptr;  // [N+1]
  const int32_t* col;     // [nnz] ascending per row
  const double* kappa;    // [nnz]
  // [nnz] interleaved row records {u32 neighbour id, u32 0, f64 weight = kappa + 1}: ONE 128-bit load per row entry on
  // the graph-row route of kernel 1b (the weight is the host's IEEE double add, bit-identical to __dadd_rn(kappa, 1.0))
  const uint4* rec;
};

// All device pointers of one chunk of targets.  Vertex-indexed arrays are addressed at voff[t],
// edge-indexed ones at eoff[t], pair arrays at poff(t) = voff[t] + eoff[t] + t (capacity n+m+1).
struct ChunkView {
  int32_t T;
  const int32_t* tgt;   // [T][2] graph ids
  const int64_t* tidx;  // [T] row in the caller's output
  const int64_t* voff;  // [T+1]
  const int64_t* eoff;  // [T+1]
  const int64_t* aoff;  // [T]   start of the target's adjacency segment (capacity: sum of the vicinity's graph degrees)
  int32_t *tn, *tm, *tlu, *tlv, *tnp, *tnpos, *tnneg, *tncls;
  int32_t *tnb, *tminv, *tmaxv;  // kernel 2v: #blocks of the vertex order (-1: diagram already written, nothing to sweep), local ids of the essential pair
  int32_t no_fast = 0;           // kernel 2v: 1 = never take the essential-pair-only shortcut
  uint8_t* tstatus;
  int* fb_counter;  // device counter: targets kernel 3v handed back
  uint8_t* tfb;  // 1: the vertex-ordered sweep (kernel 3v) did not run / bailed out -> edge-sorted kernels 2 + 3 do the ascending sweep
  // vertex-indexed
  int32_t *vert, *vcls, *vs0, *vs1, *vs2, *neg;
  double *fval, *d1, *d2;
  unsigned long long *v64a, *v64b, *v64c;
  int32_t *vord, *vrank;  // kernel 2v: rank -> local id, local id -> rank in the (value, id) vertex order
  // (n+1)-per-target arrays, addressed at voff[t] + t
  int32_t *bfirst;  // first rank of every block of the vertex order | flags in bits 31, 30 (kernel 2v), [nb] = n
  // induced adjacency (kernel 1), both directions: row of local vertex x = [astart[x], astart[x] + adeg[x])
  // inside the target's segment, which starts at aoff[t]; a row's capacity is the vertex's degree in the graph,
  // adeg of it are used; rows ascending in local id
  int32_t *astart, *adeg;  // vertex-indexed
  float* aminw;            // vertex-indexed: smallest incident weight, rounded down (settling criterion of kernel 1b)
  uint32_t* anb;           // [sum D_S] neighbour local ids
  double* aw;              // [sum D_S] kappa + 1
  // GRAPH-ROW route (dbm != nullptr): no adjacency is materialised.  Row of local vertex x = the graph's CSR row of
  // vert[x]: astart[x] = rowptr[vert[x]] (absolute position in gcol / gkappa), adeg[x] = graph degree; an entry is
  // an induced neighbour iff its graph id is in the target's vicinity bitmap dbm[t][0..W), its local id is the
  // bitmap rank (word prefix dbm[t][W..2W) + popcount below the bit).  anb / aw are not written.
  uint32_t* dbm;         // [T][2W]
  int32_t W;             // bitmap words = ceil(N / 32)
  const int32_t* gcol;   // the graph's col[]
  const double* gkappa;  // the graph's kappa[]
  int32_t count_m;       // graph-row route: kernel 1b counts the induced edges into tm[] (the counting pass skipped them)
  // edge-indexed (canonical lexicographic (lo, hi) edge list: kernel 1c, only for the edge-sorted kernels)
  int32_t *elo, *ehi, *pos, *arank;
  double* ew;
  uint32_t *ord_asc, *ord_desc, *sp0, *sp1;
  unsigned long long *sk0, *sk1;
  uint8_t* isneg;
  // pair-indexed
  uint8_t* pkind;
  int32_t *pbv, *pdv;
  double *pbirth, *pdeath;
  __host__ __device__ int64_t poff(int t) const { return voff[t] + eoff[t] + t; }
};

struct Params {
  int32_t hop, mode, descriptor, resolution;
  uint32_t flags, img_mask;
};

// ---------------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ unsigned lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// bit pattern of +inf: the distance of a vertex no relaxation has reached (distances are compared as u64 bit patterns)
constexpr unsigned long long INF_BITS = 0x7ff0000000000000ull;

__device__ __forceinline__ bool test_bit(const uint32_t* bm, int32_t y) { return (bm[y >> 5] >> (y & 31)) & 1u; }

__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) { const unsigned long long u = __shfl_xor_sync(0xffffffffu, v, o); v = u < v ? u : v; }
  return v;
}

// graph-row route: local id of graph node g in the vicinity whose bitmap / word prefix is bm[0..W) / bm[W..2W), -1 if absent
__device__ __forceinline__ int bitmap_rank(const uint32_t* bm, int W, int g) {
  const uint32_t word = bm[g >> 5];
  if (!((word >> (g & 31)) & 1u)) return -1;
  return (int)bm[W + (g >> 5)] + __popc(word & ((1u << (g & 31)) - 1u));
}

// word w of the vicinity bitmap from the two closed k-hop ball bitmaps of the target (u, v), by vicinity mode
//   EDGE: ball(u) & ball(v) (riccidist2dgm.py:311-316) | NODE: ball(u) (data_utils_NC.py:97-100) | EDGE_FORCED: (& ) + [u, v]
//   (data_utils_LP.py:111) | EDGE_UNION: ball(u) | ball(v) (riccidist2dgm.py:242-247) | EDGE_REMOVEINTER: (|) - (&) + [u, v] (:289-296)
__device__ __forceinline__ uint32_t combine_balls(int mode, uint32_t bu, uint32_t bv, int w, int u, int v) {
  uint32_t x;
  if (mode == TLC_MODE_NODE) x = bu;
  else if (mode == TLC_MODE_EDGE_UNION) x = bu | bv;
  else if (mode == TLC_MODE_EDGE_REMOVEINTER) x = bu ^ bv;
  else x = bu & bv;
  if (mode == TLC_MODE_EDGE_FORCED || mode == TLC_MODE_EDGE_REMOVEINTER) {
    if (w == (u >> 5)) x |= 1u << (u & 31);
    if (w == (v >> 5)) x |= 1u << (v & 31);
  }
  return x;
}

// order-preserving map double -> u64 (all finite values, -0 < +0 irrelevant here)
__device__ __forceinline__ unsigned long long f64_to_ordered(double x) {
  unsigned long long b = (unsigned long long)__double_as_longlong(x);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}

__device__ __forceinline__ double ordered_to_f64(unsigned long long k) {  // inverse of f64_to_ordered
  const unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}

// block-wide exclusive scan of `n` ints in (global or shared) memory, in place; returns the total.
// Each thread owns a contiguous slice; `sh` needs blockDim.x + 1 ints.  All threads must call.
__device__ inline int block_exclusive_scan(int32_t* data, int n, int32_t* sh) {
  const int nt = blockDim.x, tid = threadIdx.x;
  const int per = (n + nt - 1) / nt;
  const int lo = min(tid * per, n), hi = min(lo + per, n);
  int s = 0;
  for (int i = lo; i < hi; i++) s += data[i];
  sh[tid] = s;
  __syncthreads();
  // Hillis-Steele over nt entries (nt <= 1024)
  for (int off = 1; off < nt; off <<= 1) {
    int v = (tid >= off) ? sh[tid - off] : 0;
    __syncthreads();
    sh[tid] += v;
    __syncthreads();
  }
  int total = sh[nt - 1];
  int run = sh[tid] - s;  // exclusive prefix of this thread's slice
  __syncthreads();
  for (int i = lo; i < hi; i++) {
    int v = data[i];
    data[i] = run;
    run += v;
  }
  __syncthreads();
  return total;
}

// exclusive scan of data[0..cnt) in shared memory, two barriers; returns the total.  `wsum` needs 33 ints.  All threads call.
__device__ inline int block_scan_shfl(int32_t* data, int cnt, int32_t* wsum) {
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = (nt + 31) >> 5;
  const int per = (cnt + nt - 1) / nt;
  const int lo = min(tid * per, cnt), hi = min(lo + per, cnt);
  int s = 0;
  for (int i = lo; i < hi; i++) s += data[i];
  int inc = s;
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
  if (lane == 31) wsum[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    const int wv = lane < nw ? wsum[lane] : 0;
    int winc = wv;
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= o) winc += v; }
    if (lane < nw) wsum[lane] = winc - wv;
    if (lane == 31) wsum[32] = winc;
  }
  __syncthreads();
  int run = wsum[wid] + inc - s;
  for (int i = lo; i < hi; i++) { const int v = data[i]; data[i] = run; run += v; }
  return wsum[32];
}

__device__ inline int block_reduce_sum(int v, int32_t* sh) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if (lane_id() == 0) sh[w] = v;
  __syncthreads();
  int t = 0;
  for (int i = 0; i < nw; i++) t += sh[i];
  __syncthreads();
  return t;
}

__device__ inline double block_reduce_max(double v, double* sh) {
  for (int o = 16; o; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  const int w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if (lane_id() == 0) sh[w] = v;
  __syncthreads();
  double t = sh[0];
  for (int i = 1; i < nw; i++) t = fmax(t, sh[i]);
  __syncthreads();
  return t;
}

// ---------------------------------------------------------------------------------------------
// the reference's arithmetic, one definition for every kernel (the parity tests pin each IEEE operation order)
// ---------------------------------------------------------------------------------------------
// dict_node[u] KeyError (riccidist2dgm.py:353): an endpoint outside the graph; the reference graph has no isolated nodes
__device__ __forceinline__ bool unknown_target(const GraphView& g, int32_t u, int32_t v, bool node_mode) {
  bool bad = u < 0 || u >= g.N || (!node_mode && (v < 0 || v >= g.N));
  if (!bad) bad = g.rowptr[u + 1] == g.rowptr[u] || (!node_mode && g.rowptr[v + 1] == g.rowptr[v]);
  return bad;
}

// kernels 1b / 1t, graph-row route: the vicinity bitmap of target t from its cached balls into bm[0..W) and its word-prefix
// ranks into bm[W..2W) (both in shared memory), copied to c.dbm for kernels 2v / 3v; returns n.  The whole CTA calls.
// nodes = set(nodes_u) & set(nodes_v), canonical local ids = ranks   riccidist2dgm.py:311-316
__device__ __forceinline__ int graph_row_bitmap(const ChunkView& c, int t, const uint32_t* ball_cache, int W, int32_t u,
                                                int32_t v, bool node_mode, uint32_t* bm, int32_t* wsum) {
  const int tid = threadIdx.x, nt = blockDim.x;
  const uint32_t* __restrict__ bu = ball_cache + (size_t)u * W;
  const uint32_t* __restrict__ bv = ball_cache + (size_t)v * W;
  for (int w = tid; w < W; w += nt) {
    const uint32_t x = node_mode ? bu[w] : (bu[w] & bv[w]);
    bm[w] = x;
    bm[W + w] = __popc(x);
  }
  __syncthreads();
  const int n = block_scan_shfl(reinterpret_cast<int32_t*>(bm + W), W, wsum);
  __syncthreads();
  uint32_t* gb = c.dbm + (size_t)t * 2 * W;
  for (int w = tid; w < 2 * W; w += nt) gb[w] = bm[w];
  return n;
}

// nx.NodeNotFound (a root outside the vicinity) / nx.NetworkXNoPath -> dist = 100   riccidist2dgm.py:31-32,36-37
constexpr double NO_PATH_DIST = 100.0;

// `if x in [root_1, root_2]`: all three attributes 0   riccidist2dgm.py:22-25
template <typename T>
__device__ __forceinline__ void zero_roots(T* d1, T* d2, int lu, int lv) {
  d1[lu] = T(0); d2[lu] = T(0); d1[lv] = T(0); d2[lv] = T(0);
}

struct PySum {  // CPython's float sum(): first item exact, then Neumaier (3.12+) or plain adds   SURVEY.md F5
  double s, c;
  int k;
};
__device__ __forceinline__ void pysum_add(PySum& p, double x, bool plain) {
  if (p.k == 0) { p.s = x; p.k = 1; return; }
  if (plain) { p.s = __dadd_rn(p.s, x); return; }
  const double t = __dadd_rn(p.s, x);
  if (fabs(p.s) >= fabs(x)) p.c = __dadd_rn(p.c, __dadd_rn(__dadd_rn(p.s, -t), x));
  else p.c = __dadd_rn(p.c, __dadd_rn(__dadd_rn(x, -t), p.s));
  p.s = t;
}
__device__ __forceinline__ double pysum_get(const PySum& p, bool plain) {
  if (p.k == 0) return 0.0;
  if (!plain && p.c != 0.0 && isfinite(p.c)) return __dadd_rn(p.s, p.c);
  return p.s;
}

// build_fv's descriptor of one vertex from its distances a, b to the two roots   riccidist2dgm.py:47-53 ; data_utils_NC.py:52-54
__device__ __forceinline__ double fv_descriptor(int descriptor, bool node_mode, double a, double b) {
  if (descriptor == TLC_DESC_MIN) return fmin(a, b);
  if (descriptor == TLC_DESC_MAX) return fmax(a, b);
  return node_mode ? a : __dadd_rn(a, b);
}
// build_fv's normalisers (:54-56): smax / ssum, the vicinity's largest MAX / SUM descriptor, + 1e-10 with TLC_F_NORM_EPS.
// Without it a zero normaliser raises ZeroDivisionError (the target gets zeros, :356-357): returns false.
__device__ __forceinline__ bool fv_normalisers(uint32_t flags, double& smax, double& ssum) {
  if (flags & TLC_F_NORM_EPS) { smax = __dadd_rn(smax, 1e-10); ssum = __dadd_rn(ssum, 1e-10); return true; }
  return !(smax == 0.0 || ssum == 0.0);
}
__device__ __forceinline__ double fv_value(int descriptor, bool node_mode, bool norm, double smax, double ssum, double a,
                                           double b) {
  double f = fv_descriptor(descriptor, node_mode, a, b);
  if (norm) f = __ddiv_rn(f, descriptor == TLC_DESC_SUM ? ssum : smax);
  return f;
}

// find with path halving   accelerated_PD.py:53-58
template <typename PT>
__device__ __forceinline__ int uf_find(PT* p, int x) {
  for (;;) {
    const int px = (int)p[x];
    if (px == x) return x;
    const int gp = (int)p[px];
    p[x] = (PT)gp;
    x = gp;
  }
}

// the persistence image's per-point factors: PersistenceImager.transform (PersistenceImager.pyx:352-388), isotropic
// sigma = 1, skew (persistence = death - birth, :366)
__device__ __forceinline__ double norm_cdf(double x) {  // erfc(-x / sqrt(2)) / 2   :60
  return erfc(-x / 1.4142135623730951) * 0.5;
}
__device__ __forceinline__ double norm_pdf(double x) {  // d norm_cdf / dx = exp(-x^2 / 2) / sqrt(2 pi)
  return exp(-0.5 * x * x) * 0.3989422804014327;
}
__device__ __forceinline__ double ramp_weight(double pers) {  // linear_ramp defaults  :22-28
  return pers < 0.0 ? 0.0 : (pers > 1.0 ? 1.0 : pers);
}
// the point's CDF differences over the pixels of both axes, mesh i * step (i = 0 .. res)   :302-314,385-388
__device__ __forceinline__ void cdf_diffs(int res, double step, double birth, double pers, double* gb, double* gp) {
  double pb = norm_cdf(0.0 - birth), pp = norm_cdf(0.0 - pers);
#pragma unroll
  for (int i = 1; i <= res; i++) {
    const double pt = i * step;
    const double cb = norm_cdf(pt - birth), cp = norm_cdf(pt - pers);
    gb[i - 1] = cb - pb; gp[i - 1] = cp - pp;
    pb = cb; pp = cp;
  }
}

// ---------------------------------------------------------------------------------------------
// kernel launchers (defined in the k*.cu files), all asynchronous on `st`
// ---------------------------------------------------------------------------------------------
struct VicinityScratch {
  uint32_t* bitmaps;  // global fallback: [grid][2*W] words when the bitmaps do not fit shared memory
  int32_t* queue;     // [grid][2*N] frontier queues, only for hop > 2
  int grid;
  // ball cache (per graph and hop): the closed k-hop ball of a node is shared by every target incident to it, so
  // it is expanded once and kept as a bitmap row; a vicinity is then the AND of two rows.  nullptr: expand per target.
  uint32_t* ball_cache;            // [N][W]
  unsigned long long* ball_acc;    // [N][2]: expanded degree sum, rowptr pairs read (algorithmic-byte accounting)
  int32_t* ball_state;             // [N]: 0 not cached, 1 claimed for this call, 2 cached
  int32_t* ball_list;              // [N] nodes to expand in this call
  int* ball_count;
};

void launch_vicinity_sizes(const GraphView& g, const Params& p, const int32_t* targets, int64_t E, int32_t* out_n,
                           int32_t* out_m, int32_t* out_ds, uint8_t* out_status, double* out_bytes,
                           const VicinityScratch& vs, int* work_counter, cudaStream_t st);
// graph-row route: n, D_S, status (needs the ball cache); out_m receives a planning estimate, kernel 1b counts m
void launch_vicinity_light(const GraphView& g, const Params& p, const int32_t* targets, int64_t E, int32_t* out_n,
                           int32_t* out_m, int32_t* out_ds, uint8_t* out_status, double* out_bytes,
                           const VicinityScratch& vs, int sm_count, cudaStream_t st);
void launch_vicinity_fill(const GraphView& g, const Params& p, const ChunkView& c, const VicinityScratch& vs,
                          int* work_counter, cudaStream_t st);
void launch_filtration(const Params& p, const ChunkView& c, int t0, int cnt, int block, int64_t n_max, cudaStream_t st);
void launch_degree_filtration(const Params& p, const ChunkView& c, cudaStream_t st);
void launch_hks_filtration(const Params& p, const ChunkView& c, double t, int64_t n_max, cudaStream_t st);
// graph-row route: builds the vicinity (bitmap, ranks, vertex list, roots, status) itself and runs the shortest-path
// phases over the graph's own CSR rows filtered by the bitmap (everything L2-resident, no adjacency in HBM)
void launch_filtration_direct(const GraphView& g, const Params& p, const ChunkView& c, const VicinityScratch& vs,
                              const float* gminw, int t0, int cnt, int block, int64_t n_max, cudaStream_t st);
// canonical edge list (elo, ehi, ew) from the adjacency; fb_only: only for targets with tfb[t] != 0
void launch_edgelist(const Params& p, const ChunkView& c, int block, int fb_only, cudaStream_t st);
// sweep_mask: bit 0 ascending, bit 1 descending.  fb_only: the ascending sweep only for targets with tfb[t] != 0.
void launch_sort(const Params& p, const ChunkView& c, int block, int sweep_mask, int fb_only, cudaStream_t st);
void launch_union_find(const Params& p, const ChunkView& c, int block, int smem_ints, int build_lists, int sweep_mask,
                       int fb_only, cudaStream_t st);
void launch_vorder(const Params& p, const ChunkView& c, int t0, int cnt, int block, int64_t n_max, cudaStream_t st);
void launch_sweep(const Params& p, const ChunkView& c, int t0, int cnt, int64_t n_max, cudaStream_t st);
void launch_loops(const Params& p, const ChunkView& c, int block, int smem_ints, int64_t n_max, cudaStream_t st);
void launch_pimg(const Params& p, const ChunkView& c, double* out_pi, float* out_pi_f32, uint8_t* out_status,
                 int block, cudaStream_t st);
void launch_pimg_batch(const int64_t* poff, const double* birth, const double* death, const uint8_t* kind,
                       uint32_t img_mask, int res, int64_t D, double* out, cudaStream_t st);
void launch_pimg_batch_grad(const int64_t* poff, const double* birth, const double* death, const uint8_t* kind,
                            uint32_t img_mask, int res, int64_t D, const double* grad_out, double* grad_birth,
                            double* grad_death, cudaStream_t st);
uint64_t wasserstein_workspace_bytes(int64_t D, int64_t Px, int64_t Py);
void launch_wasserstein(const int64_t* poff_x, const double* bx, const double* dx, const uint8_t* kx,
                        const int64_t* poff_y, const double* by, const double* dy, const uint8_t* ky, uint32_t mask,
                        double order, double internal_p, int64_t D, void* ws, uint64_t ws_bytes, double* dist,
                        int64_t* match_x, int64_t* match_y, cudaStream_t st);
void launch_wasserstein_grad(const int64_t* poff_x, const double* bx, const double* dx, const uint8_t* kx,
                             const int64_t* poff_y, const double* by, const double* dy, const uint8_t* ky,
                             uint32_t mask, double order, double internal_p, int64_t D, const double* dist,
                             const int64_t* match_x, const int64_t* match_y, const double* grad_out, double* gbx,
                             double* gdx, double* gby, double* gdy, cudaStream_t st);

void launch_gather_rows(const double* table, int64_t rows, int r2, const int64_t* index, int64_t start, int64_t n,
                        float* out, int* bad, int sm_count, cudaStream_t st);

void launch_scatter_rows(const double* src_pi, const float* src_pi32, const uint8_t* src_st, const int64_t* idx, int64_t k,
                         int r2, double* dst_pi, float* dst_pi32, uint8_t* dst_st, int sm_count, cudaStream_t st);

// kernel 1t (k1t_sssp_table.cu): per-root shortest-path tables, [N][N] entries, row r over the subgraph induced by r's
// k-hop ball (the tables hold one hop at a time), rows built on demand.  Three arrays, split by the pass that reads them:
// kernel 1t's class pass reads D and P of every vertex of S (dense rows: neighbouring vertices of S share their sectors),
// only the valid vertices' output pass reads Q and W, together in one 16-byte load.
struct SsspTables {
  double* D;       // fl-distance from the root (bit pattern of the Dijkstra fixpoint), +inf outside the ball / unreachable
  int32_t* P;      // tree parent (graph id), -1 for the root / unreachable
  double2* QW;     // {Q, W}: python-order path sum x -> root (100 where unreachable), weight kappa + 1 of the tree edge
                   // (x, P[x]) (0 without one)
  int32_t* state;  // [N] 0 row not built, 1 claimed in this call, 2 built
  int32_t* list;   // [N] roots to build in this call
  int* count;
};
void launch_sssp_build(const GraphView& g, const Params& p, const int32_t* targets, int64_t E, const SsspTables& tb,
                       const uint32_t* ball_cache, const float* gminw, double* pw_scratch, int grid, cudaStream_t st);
size_t sssp_build_smem(int N);
void launch_filtration_table(const GraphView& g, const Params& p, const ChunkView& c, const VicinityScratch& vs,
                             const SsspTables& tb, const int32_t* n_of, int t0, int cnt, int block, int64_t n_min,
                             int64_t n_max, cudaStream_t st);
size_t filtration_table_smem(int N, int64_t n_max);

// kernel 6 (k6_ricci.cu): Ollivier-Ricci curvature (Sinkhorn) of a host-prepared edge list
void launch_ricci(const int32_t* rowptr, const int32_t* col, const uint32_t* ball1, const uint32_t* ball2, int W,
                  const int64_t* epos, const int64_t* emir, const int32_t* esrc, int64_t E, double alpha, const double* kval4,
                  const double* wsum, double wnb, int topk, int max_iter, double stop_thr, int cap, bool codes_smem,
                  uint8_t* slab, size_t slab_stride, int grid, double* out, int32_t* iters, cudaStream_t st);
size_t ricci_smem_bytes(int cap, bool codes_smem);

// kernel S (k0_small.cu): the whole path for small vicinities in one launch per size class
struct SmallDiag {  // optional diagram output: pairs of row t at poff[t] (capacity n + m + 2 per row)
  const int64_t* poff;
  int32_t* np;
  uint8_t* kind;
  int32_t *bv, *dv;
  double *birth, *death;
  int graph_ids = 0;  // 1: birth / death vertices as graph ids (default: local ids)
  int want_desc = 1;  // 0: ascending sweep only (PD_up and [min,max])
};
struct SmallStats {  // device accumulators of one call
  unsigned long long handled[3];  // rows finished by class A / B / C (any status)
  unsigned long long live, sum_n, sum_m;  // over the rows with status <= TRIVIAL
  double bytes;                   // their compulsory bytes B_e (SURVEY.md 8d)
};
void launch_small(const GraphView& g, const Params& p, const int32_t* targets, int64_t E, const VicinityScratch& vs,
                  double* out_pi, float* out_pi32, uint8_t* out_status, int32_t* list_b, int32_t* list_c, int32_t* list_big,
                  int* counters, int32_t* out_n, int32_t* out_m, const SmallDiag* diag, SmallStats* stats, int sm_count,
                  int phases, cudaStream_t st, int32_t* list_b2 = nullptr);
// rows of a sub-list: sub[i] = targets[list[i]], idx[i] = list[i]
void launch_gather_targets(const int32_t* targets, const int32_t* list, int64_t k, int32_t* sub, int64_t* idx, cudaStream_t st);

// kernel 7 (k7_diagrams.cu): the diagrams of a batch call.  A pair array set (structure of arrays, graph vertex ids).
struct DiagArea {
  uint8_t* kind;
  int32_t *bv, *dv;
  double *birth, *death;
};
// pairs a target's diagram holds: those of the statuses kernel S and the staged pipeline report pairs for
__host__ __device__ inline int diag_pairs(uint8_t status, int32_t np) {
  return (status <= TLC_ST_TRIVIAL || status == TLC_ST_NO_TREE_EDGES) && np > 0 ? np : 0;
}
// the chunk's pairs into `area` at dst[t] - area_base, graph ids; np_out / soff_out[rows[t]] = count / dst[t] (rows[t] < 0: skipped)
void launch_export_pairs(const ChunkView& c, const int64_t* dst, const int64_t* rows, const DiagArea& area,
                         int64_t area_base, int32_t* np_out, int64_t* soff_out, int sm_count, cudaStream_t st);
// poff[0..E] = exclusive scan of np[0..E)
void launch_scan_counts(const int32_t* np, int64_t E, int64_t* poff, cudaStream_t st);
// out[poff[t] ..] = segment t of the staging (offsets soff[t] < split_at in a, the others in b at soff[t] - split_at);
// NULL arrays of `out` are skipped
void launch_gather_pairs(const int32_t* np, const int64_t* soff, const int64_t* poff, int64_t E, const DiagArea& a,
                         const DiagArea& b, int64_t split_at, const DiagArea& out, int sm_count, cudaStream_t st);

// kernel 9 (k9_graph_pd.cu): diagrams of a batch of caller-supplied graphs (tlc_graph_batch_*).  Graph t owns vertices
// noff[t] .. noff[t+1] and edges eoff[t] .. eoff[t+1] of (ea, eb), batch-global ids; its pairs are staged at soff[t] =
// noff[t] + eoff[t] + t (capacity n + m + 1), np[t] / status[t] are its pair count (0 unless the status has pairs) and status
struct GraphBatchView {
  int64_t D;
  const int64_t *noff, *eoff, *soff;
  const int32_t *ea, *eb;
  const double* f;
  uint32_t flags;
  DiagArea stage;
  int32_t* np;
  uint8_t* status;
};
// the fused route's size classes (kernel S's): a warp per graph, a 128-thread CTA, a 256-thread CTA
constexpr int GRAPH_A_N = 64, GRAPH_A_M = 256, GRAPH_B_N = 256, GRAPH_B_M = 2048, GRAPH_C_N = 1024, GRAPH_C_M = 4096;
// lists[c] / counts[c]: the graphs of class c
void launch_graph_pd_small(const GraphBatchView& b, const int32_t* const lists[3], const int counts[3], cudaStream_t st);
// staged route: c.tidx[s] = graph of staged entry s, c.voff / c.eoff its segments in the arena
void launch_graph_fill(const GraphBatchView& b, const ChunkView& c, int sm_count, cudaStream_t st);
void launch_graph_export(const GraphBatchView& b, const ChunkView& c, int sm_count, cudaStream_t st);
// cnt int32[N], lst int32[2 (N + M + D)]: scratch
void launch_graph_grad(const GraphBatchView& b, const int64_t* poff, const int32_t* bv, const int32_t* dv, const double* gb,
                       const double* gd, int32_t* cnt, int32_t* lst, double* grad_f, int sm_count, cudaStream_t st);

// kernel 10 (k10_vicinity_batch.cu): vicinities in graph-batch layout (tlc_vicinity_batch_dev) and the device-side check
// of a graph batch in canonical form (tlc_graph_batch_create_dev).
// export: chunk target t's vertices, edges (local id + voff[row]) and filtration values to voff[row] / eoff[row], row =
// c.tidx[t]; its final status (a connected check over its edges turns OK / TRIVIAL into DISCONNECTED) to status[row].
// bad_desc: every OK / TRIVIAL target reports BAD_DESCRIPTOR (written by the host) and gets NaN values.  NULL arrays are
// skipped.
void launch_vicinity_export(const ChunkView& c, const int64_t* voff, const int64_t* eoff, int32_t* vert, int32_t* ea,
                            int32_t* eb, double* fval, uint8_t* status, int bad_desc, cudaStream_t st);
// the first edge k (in index order) that breaks canonical form, as first = k * 4 + reason (reason: 0 endpoint outside its
// graph, 1 self-loop, 2 ea > eb, 3 not strictly after edge k - 1); first is left as it was (all ones) when there is none.
// noff / eoff must be monotone (checked on the host).
constexpr int BATCH_BAD_RANGE = 0, BATCH_BAD_LOOP = 1, BATCH_BAD_ORIENT = 2, BATCH_BAD_ORDER = 3;
void launch_batch_check(int64_t D, int64_t M, const int64_t* noff, const int64_t* eoff, const int32_t* ea, const int32_t* eb,
                        unsigned long long* first, int sm_count, cudaStream_t st);

// multi-GPU exchange by peer stores (k5_gather.cu): the tables of all ranks, this rank's own included
constexpr int PEER_MAX = 16;
constexpr size_t PEER_HEADER_BYTES = 256;  // [u32 arrival counter | pad] in front of the float32 rows
struct PeerTables {
  int n;
  void* table[PEER_MAX];
};
void launch_peer_scatter(const float* src_pi32, const uint8_t* src_st, const int64_t* row_index, int64_t k, int r2,
                         const PeerTables& pt, unsigned int* ticket, int sm_count, cudaStream_t st);
void launch_peer_wait(const unsigned int* flag, unsigned int target, cudaStream_t st);

int64_t launch_count();
void count_launch();
int vicinity_grid(int device, const GraphView& g, const Params& p, size_t* bitmap_words, bool* use_smem);
// expand (once) the balls of the targets' endpoints that are not cached yet (targets == nullptr: of every node)
void launch_ball_cache(const GraphView& g, const Params& p, const int32_t* targets, int64_t E, const VicinityScratch& vs,
                       cudaStream_t st);

}  // namespace tlc
