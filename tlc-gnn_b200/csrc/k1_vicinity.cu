// k1_vicinity.cu -- kernel 1: batched k-hop vicinity extraction on the CSR graph.
//
// Replaces riccidist2dgm.py:311-316 (two nx.bfs_edges balls, set intersection, G.subgraph) and
// Knowledge_Distillation/data_utils_NC.py:97-100 (node-centred ball).
//
// One CTA per target at a time (persistent grid, targets handed out by an atomic counter).  The two
// closed balls are bitmaps over the N graph nodes (shared memory when 2*ceil(N/32) words fit, else a
// per-CTA slab in HBM); the vicinity is their AND.  Local vertex ids are ranks in the bitmap
// (word-prefix popcounts), which yields the canonical ascending-id order for free; induced edges are
// emitted lexicographically (lo,hi) by a count / scan / ballot-compacted fill over the CSR rows.
//
// Two entry points share the traversal: a counting pass (n, m per target -> the host sizes the chunk
// arena) and the fill pass (vertex list, induced edges with weight kappa+1, local root ids).
#include <algorithm>

#include "tlc_common.cuh"

namespace tlc {

namespace {

constexpr int K1_BLOCK = 256;

struct K1Shared {
  int32_t scan[K1_BLOCK + 1];
  int32_t red[32];
  int32_t qcnt[2];
  int32_t target;
  int32_t next;   // next bitmap word (a batch of <= 32 vicinity vertices) to hand to a warp
  int32_t ecur;   // fill: adjacency entries reserved so far
  // per warp, for the batch of 32 rows in flight: degree prefix, write cursors, row starts, smallest weights
  int32_t bcnt[K1_BLOCK / 32][32], bmin[K1_BLOCK / 32][32], bra[K1_BLOCK / 32][32], bmw[K1_BLOCK / 32][32];
  unsigned long long dacc;  // algorithmic-byte accounting: sum of expanded degrees (D_u + D_v + D_S)
  unsigned long long xacc;  // ... and number of rowptr pairs read (X)
};

__device__ __forceinline__ bool set_bit(uint32_t* bm, int32_t y) {  // returns true if newly set
  const uint32_t bit = 1u << (y & 31);
  if (bm[y >> 5] & bit) return false;
  return (atomicOr(&bm[y >> 5], bit) & bit) == 0;
}

// a warp walks the CSR row [a, b) of col[]: the 16-byte aligned body with coalesced 128-bit loads (four neighbour ids per
// lane and load, LDG.E.128), the unaligned head and the tail with 32-bit loads.  f(y) is called once per entry.
template <typename F>
__device__ __forceinline__ void warp_row_v4(const int32_t* __restrict__ col, int32_t a, int32_t b, int lane, F f) {
  const int32_t a4 = min(b, (a + 3) & ~3);           // first 4-aligned index (cudaMalloc'ed col[] is 256-byte aligned)
  const int32_t b4 = a4 + ((b - a4) & ~3);           // end of the whole int4 groups
  if (a + lane < a4) f(col[a + lane]);               // head: < 4 entries
  for (int32_t e = a4 + 4 * lane; e < b4; e += 128) {
    const int4 v = __ldg(reinterpret_cast<const int4*>(col + e));
    f(v.x); f(v.y); f(v.z); f(v.w);
  }
  if (b4 + lane < b) f(col[b4 + lane]);              // tail: < 4 entries
}

// closed ball of radius hop around root into bm (bm zeroed by the caller).
// nodes_u = [root] + [x for _, x in nx.bfs_edges(G, root, depth_limit=hop)]   riccidist2dgm.py:311-312
__device__ void ball(const GraphView& g, int32_t root, int hop, uint32_t* bm, int32_t* q0, int32_t* q1,
                     K1Shared& sh) {
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  if (tid == 0) bm[root >> 5] |= 1u << (root & 31);
  __syncthreads();
  if (hop <= 0) return;
  const int32_t r0 = g.rowptr[root], r1 = g.rowptr[root + 1];
  if (tid == 0) { sh.dacc += (unsigned long long)(r1 - r0); sh.xacc += 1; }
  // depth 1: the CSR row of the root, every warp a 128-entry slice of it (128-bit loads)
  for (int32_t s0 = r0 + wid * 128; s0 < r1; s0 += nw * 128)
    warp_row_v4(g.col, s0, min(s0 + 128, r1), lane, [&](int32_t y) { set_bit(bm, y); });
  __syncthreads();
  if (hop == 1) return;
  // depth 2: one warp per depth-1 vertex, lanes stride its row (coalesced)
  const bool push = hop > 2;
  if (tid == 0) sh.qcnt[0] = 0;
  __syncthreads();
  for (int32_t i = r0 + wid; i < r1; i += nw) {
    const int32_t x = g.col[i];
    const int32_t a = g.rowptr[x], b = g.rowptr[x + 1];
    if (lane == 0) { atomicAdd(&sh.dacc, (unsigned long long)(b - a)); atomicAdd(&sh.xacc, 1ull); }
    warp_row_v4(g.col, a, b, lane, [&](int32_t y) { if (set_bit(bm, y) && push) q0[atomicAdd(&sh.qcnt[0], 1)] = y; });
  }
  __syncthreads();
  // depth >= 3: explicit frontier queues (HBM slabs); newly set bits form the next frontier
  int32_t* cur = q0;
  int32_t* nxt = q1;
  int ci = 0;
  for (int d = 2; d < hop; d++) {
    const int cnt = sh.qcnt[ci];
    if (tid == 0) sh.qcnt[ci ^ 1] = 0;
    __syncthreads();
    if (cnt == 0) break;
    const bool push2 = d + 1 < hop;
    for (int i = wid; i < cnt; i += nw) {
      const int32_t x = cur[i];
      const int32_t a = g.rowptr[x], b = g.rowptr[x + 1];
      if (lane == 0) { atomicAdd(&sh.dacc, (unsigned long long)(b - a)); atomicAdd(&sh.xacc, 1ull); }
      warp_row_v4(g.col, a, b, lane, [&](int32_t y) { if (set_bit(bm, y) && push2) nxt[atomicAdd(&sh.qcnt[ci ^ 1], 1)] = y; });
    }
    __syncthreads();
    int32_t* t = cur; cur = nxt; nxt = t;
    ci ^= 1;
  }
  __syncthreads();
}

// ball(u) & ball(v) -> iw (in bm_u) ; word-prefix popcounts -> wbase (in bm_v) ; returns n
__device__ int build_vicinity(const GraphView& g, const Params& p, int32_t u, int32_t v, int W, uint32_t* bm_u,
                              uint32_t* bm_v, int32_t* q0, int32_t* q1, K1Shared& sh, const VicinityScratch& vs) {
  const int tid = threadIdx.x, nt = blockDim.x;
  if (vs.ball_cache) {  // both balls are cached rows: nodes = set(nodes_u) & set(nodes_v)   :315
    const uint32_t* __restrict__ bu = vs.ball_cache + (size_t)u * W;
    const uint32_t* __restrict__ bv = vs.ball_cache + (size_t)v * W;
    const bool edge = p.mode != TLC_MODE_NODE;
    for (int w = tid; w < W; w += nt) {
      const uint32_t x = combine_balls(p.mode, bu[w], edge ? bv[w] : 0u, w, u, v);
      bm_u[w] = x;
      bm_v[w] = __popc(x);
    }
    if (tid == 0) {
      sh.dacc = vs.ball_acc[2 * (size_t)u] + (edge ? vs.ball_acc[2 * (size_t)v] : 0ull);
      sh.xacc = vs.ball_acc[2 * (size_t)u + 1] + (edge ? vs.ball_acc[2 * (size_t)v + 1] : 0ull);
    }
    __syncthreads();
    return block_exclusive_scan(reinterpret_cast<int32_t*>(bm_v), W, sh.scan);
  }
  for (int w = tid; w < 2 * W; w += nt) bm_u[w] = 0;  // bm_v follows bm_u
  __syncthreads();
  ball(g, u, p.hop, bm_u, q0, q1, sh);
  if (p.mode != TLC_MODE_NODE) {
    ball(g, v, p.hop, bm_v, q0, q1, sh);
    for (int w = tid; w < W; w += nt) {  // nodes = set(nodes_u) & set(nodes_v)   :315 (or the mode's other combination)
      const uint32_t x = combine_balls(p.mode, bm_u[w], bm_v[w], w, u, v);
      bm_u[w] = x;
      bm_v[w] = __popc(x);
    }
  } else {
    for (int w = tid; w < W; w += nt) bm_v[w] = __popc(bm_u[w]);
  }
  __syncthreads();
  return block_exclusive_scan(reinterpret_cast<int32_t*>(bm_v), W, sh.scan);
}

__device__ __forceinline__ int32_t local_id(const uint32_t* iw, const uint32_t* wbase, int32_t y) {
  return (int32_t)wbase[y >> 5] + __popc(iw[y >> 5] & ((1u << (y & 31)) - 1u));
}

// ---- ball cache ----
__global__ void ball_mark_kernel(const int32_t* __restrict__ targets, int64_t E, int node_mode, GraphView g,
                                 VicinityScratch vs) {
  const int64_t total = 2 * E;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    if (node_mode && (i & 1)) continue;
    const int32_t x = targets[i];
    if (x < 0 || x >= g.N || g.rowptr[x + 1] == g.rowptr[x]) continue;
    if (vs.ball_state[x] == 0 && atomicCAS(&vs.ball_state[x], 0, 1) == 0) vs.ball_list[atomicAdd(vs.ball_count, 1)] = x;
  }
}

__global__ void ball_mark_all_kernel(GraphView g, VicinityScratch vs) {  // every node with an edge whose ball is not cached yet
  for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < g.N; x += gridDim.x * blockDim.x) {
    if (g.rowptr[x + 1] == g.rowptr[x]) continue;
    if (vs.ball_state[x] == 0 && atomicCAS(&vs.ball_state[x], 0, 1) == 0) vs.ball_list[atomicAdd(vs.ball_count, 1)] = x;
  }
}

__global__ void __launch_bounds__(K1_BLOCK)
ball_build_kernel(GraphView g, Params p, VicinityScratch vs, int W, int bm_in_smem) {
  extern __shared__ uint32_t dyn_smem[];
  __shared__ K1Shared sh;
  const int tid = threadIdx.x, nt = blockDim.x;
  uint32_t* bm = bm_in_smem ? dyn_smem : vs.bitmaps + (size_t)blockIdx.x * 2 * W;
  int32_t* q0 = vs.queue ? vs.queue + (size_t)blockIdx.x * 2 * g.N : nullptr;
  int32_t* q1 = q0 ? q0 + g.N : nullptr;
  const int cnt = *vs.ball_count;
  for (int idx = blockIdx.x; idx < cnt; idx += gridDim.x) {
    const int32_t root = vs.ball_list[idx];
    __syncthreads();
    for (int w = tid; w < W; w += nt) bm[w] = 0;
    if (tid == 0) { sh.dacc = 0; sh.xacc = 0; }
    __syncthreads();
    ball(g, root, p.hop, bm, q0, q1, sh);
    uint32_t* row = vs.ball_cache + (size_t)root * W;
    for (int w = tid; w < W; w += nt) row[w] = bm[w];
    if (tid == 0) {
      vs.ball_acc[2 * (size_t)root] = sh.dacc;
      vs.ball_acc[2 * (size_t)root + 1] = sh.xacc;
      vs.ball_state[root] = 2;
    }
  }
}

// Counting pass of the GRAPH-ROW route: n, D_S and the status only -- the induced edges are not counted here (the
// filtration kernel counts them while it reads the rows anyway).  One warp per target: the vicinity is the AND of two
// cached ball bitmaps, n its popcount, D_S the sum of the members' graph degrees.
__global__ void __launch_bounds__(256)
vicinity_light_kernel(GraphView g, Params p, const int32_t* __restrict__ targets, int64_t E, int32_t* out_n, int32_t* out_m,
                      int32_t* out_ds, uint8_t* out_status, double* out_bytes, VicinityScratch vs, int W) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const bool node_mode = p.mode == TLC_MODE_NODE;
  for (int64_t t = warp; t < E; t += nwarps) {
    const int32_t u = targets[2 * t], v = targets[2 * t + 1];
    if (unknown_target(g, u, v, node_mode)) {
      if (lane == 0) { out_n[t] = 0; out_m[t] = 0; out_ds[t] = 0; out_status[t] = TLC_ST_UNKNOWN_NODE; if (out_bytes) out_bytes[t] = 0.0; }
      continue;
    }
    const uint32_t* __restrict__ bu = vs.ball_cache + (size_t)u * W;
    const uint32_t* __restrict__ bv = vs.ball_cache + (size_t)v * W;
    int n = 0;
    long long ds = 0;
    for (int w = lane; w < W; w += 32) {
      uint32_t bits = node_mode ? bu[w] : (bu[w] & bv[w]);
      n += __popc(bits);
      while (bits) {
        const int x = w * 32 + __ffs(bits) - 1;
        bits &= bits - 1;
        ds += g.rowptr[x + 1] - g.rowptr[x];
      }
    }
    for (int o = 16; o; o >>= 1) { n += __shfl_xor_sync(0xffffffffu, n, o); ds += __shfl_xor_sync(0xffffffffu, ds, o); }
    if (lane == 0) {
      out_n[t] = n;
      out_m[t] = (int32_t)(ds / 3);  // planning estimate only (CTA width class); the exact count comes from kernel 1b
      out_ds[t] = (int32_t)ds;
      uint8_t st = TLC_ST_OK;
      if (n == 0 || (node_mode && n == 1)) st = TLC_ST_EMPTY;  // :318 / data_utils_NC.py:103-104 (lone centre <=> no edge)
      out_status[t] = st;
      if (out_bytes) {  // compulsory bytes B_e (SURVEY.md 8d) WITHOUT the 16 m term, added once m is known
        const unsigned long long dacc = vs.ball_acc[2 * (size_t)u] + (node_mode ? 0ull : vs.ball_acc[2 * (size_t)v]) + (unsigned long long)ds;
        const unsigned long long xacc = vs.ball_acc[2 * (size_t)u + 1] + (node_mode ? 0ull : vs.ball_acc[2 * (size_t)v + 1]);
        out_bytes[t] = 4.0 * (double)dacc + 8.0 * (double)(xacc + (unsigned long long)n) + 4.0 * p.resolution * p.resolution;
      }
    }
  }
}

template <bool FILL>
__global__ void __launch_bounds__(K1_BLOCK)
vicinity_kernel(GraphView g, Params p, const int32_t* __restrict__ targets, int64_t E, int32_t* out_n, int32_t* out_m,
                int32_t* out_ds, uint8_t* out_status, double* out_bytes, ChunkView c, VicinityScratch vs, int* work_counter,
                int W, int bm_in_smem) {
  extern __shared__ uint32_t dyn_smem[];
  __shared__ K1Shared sh;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5;
  uint32_t* bm_u = bm_in_smem ? dyn_smem : vs.bitmaps + (size_t)blockIdx.x * 2 * W;
  uint32_t* bm_v = bm_u + W;
  int32_t* q0 = vs.queue ? vs.queue + (size_t)blockIdx.x * 2 * g.N : nullptr;
  int32_t* q1 = q0 ? q0 + g.N : nullptr;

  for (;;) {
    __syncthreads();
    if (tid == 0) sh.target = atomicAdd(work_counter, 1);
    __syncthreads();
    const int64_t t = sh.target;
    if (t >= E) break;
    const int64_t ti = FILL ? c.tidx[t] : t;
    const int32_t u = targets[2 * ti], v = targets[2 * ti + 1];
    const bool node_mode = p.mode == TLC_MODE_NODE;
    if (unknown_target(g, u, v, node_mode)) {
      if (tid == 0) {
        if (!FILL) { out_n[t] = 0; out_m[t] = 0; out_ds[t] = 0; out_status[t] = TLC_ST_UNKNOWN_NODE; }
        else { c.tn[t] = 0; c.tm[t] = 0; c.tnp[t] = 0; c.tnpos[t] = 0; c.tnneg[t] = 0; c.tlu[t] = -1; c.tlv[t] = -1;
               c.tstatus[t] = TLC_ST_UNKNOWN_NODE; }
      }
      continue;
    }
    if (tid == 0) { sh.dacc = 0; sh.xacc = 0; }
    __syncthreads();
    const int n = build_vicinity(g, p, u, v, W, bm_u, bm_v, q0, q1, sh, vs);
    const uint32_t* iw = bm_u;
    const uint32_t* wbase = bm_v;

    if (!FILL) {
      // counting pass: every induced edge is seen from both ends -> m = (sum over vicinity rows of kept entries) / 2
      if (tid == 0) { sh.next = 0; sh.ecur = 0; }
      __syncthreads();
      int msum = 0;
      int32_t* binc = sh.bcnt[wid];  // per warp: inclusive degree prefix / row starts of the batch
      int32_t* bra = sh.bmin[wid];
      for (;;) {
        int w = 0;
        if (lane == 0) w = atomicAdd(&sh.next, 1);
        w = __shfl_sync(0xffffffffu, w, 0);
        if (w >= W) break;
        const uint32_t bits = iw[w];
        if (!bits) continue;
        const bool has = (bits >> lane) & 1u;
        const int32_t x = w * 32 + lane;
        const int32_t ra = has ? g.rowptr[x] : 0;
        const int dg = has ? g.rowptr[x + 1] - ra : 0;
        int inc = dg;
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
        const int total = __shfl_sync(0xffffffffu, inc, 31);
        __syncwarp();
        binc[lane] = inc;
        bra[lane] = ra - (inc - dg);  // entry e of row r sits at col[bra[r] + e]
        __syncwarp();
        if (lane == 0) atomicAdd(&sh.ecur, total);
        // every lane walks the concatenated rows with its own monotone row pointer (no shuffles in the loop)
        int r = 0, nxt = binc[0];
        constexpr int CU = 4;
        for (int e0 = lane; e0 < total; e0 += 32 * CU) {
          int32_t yy[CU];
#pragma unroll
          for (int k = 0; k < CU; k++) {
            const int e = e0 + 32 * k;
            if (e < total) {
              while (e >= nxt) nxt = binc[++r];
              yy[k] = g.col[bra[r] + e];
            } else yy[k] = -1;
          }
#pragma unroll
          for (int k = 0; k < CU; k++) msum += (yy[k] >= 0 && test_bit(iw, yy[k])) ? 1 : 0;
        }
        __syncwarp();
      }
      const int m = block_reduce_sum(msum, sh.red) / 2;
      if (tid == 0) {
        sh.dacc += (unsigned long long)sh.ecur;
        out_n[t] = n;
        out_m[t] = m;
        out_ds[t] = sh.ecur;  // D_S: sum of the vicinity vertices' degrees = capacity of the adjacency segment
        uint8_t st = TLC_ST_OK;
        if (n == 0) st = TLC_ST_EMPTY;                          // assert len(components) == 1 fails  :318
        else if ((node_mode || p.mode == TLC_MODE_EDGE_FORCED) && m == 0) st = TLC_ST_EMPTY;  // `return None, None` data_utils_NC.py:103-104, data_utils_LP.py:117-118
        out_status[t] = st;
        // compulsory bytes B_e (SURVEY.md 8d): int32 neighbour reads of both expansions and of the induced
        // scan, rowptr pairs, f64 weight per induced directed edge, fp32 image
        if (out_bytes)
          out_bytes[t] = 4.0 * (double)sh.dacc + 8.0 * (double)(sh.xacc + (unsigned long long)n) + 16.0 * (double)m +
                         4.0 * p.resolution * p.resolution;
      }
      continue;
    }

    // ---- fill: vertex list, then the induced adjacency (both directions, rows ascending) ----
    const int64_t vo = c.voff[t], ao = c.aoff[t];
    for (int w = tid; w < W; w += nt) {
      uint32_t bits = iw[w];
      int32_t lx = (int32_t)wbase[w];
      while (bits) {
        const int b = __ffs(bits) - 1;
        bits &= bits - 1;
        c.vert[vo + lx++] = w * 32 + b;
      }
    }
    if (tid == 0) { sh.next = 0; sh.ecur = 0; }
    __syncthreads();
    // a warp takes the next bitmap word (batch of <= 32 vertices), reserves the batch's rows (capacity = graph
    // degree) in the target's adjacency segment with one atomic, and writes local neighbour ids + weights kappa+1
    // compacted at each row's start, in row order: ONE walk over the concatenated rows
    int32_t* binc = sh.bcnt[wid];   // inclusive degree prefix of the batch
    int32_t* bcur = sh.bmin[wid];   // running write cursor of every row
    int32_t* bra = sh.bra[wid];
    int32_t* bmw = sh.bmw[wid];     // smallest kept weight of each row (float bits, rounded down)
    int kept_total = 0;
    for (;;) {
      int w = 0;
      if (lane == 0) w = atomicAdd(&sh.next, 1);
      w = __shfl_sync(0xffffffffu, w, 0);
      if (w >= W) break;
      const uint32_t bits = iw[w];
      if (!bits) continue;
      const bool has = (bits >> lane) & 1u;
      const int32_t x = w * 32 + lane;
      const int lx = (int)wbase[w] + __popc(bits & lanemask_lt());
      const int32_t ra = has ? g.rowptr[x] : 0;
      const int dg = has ? g.rowptr[x + 1] - ra : 0;
      int inc = dg;
      for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
      const int total = __shfl_sync(0xffffffffu, inc, 31);
      int start = 0;
      if (lane == 0) start = atomicAdd(&sh.ecur, total);
      start = __shfl_sync(0xffffffffu, start, 0);
      const int rbase = start + inc - dg;
      __syncwarp();
      binc[lane] = inc;
      bra[lane] = ra - (inc - dg);
      bcur[lane] = rbase;
      bmw[lane] = 0x7f7fffff;  // FLT_MAX
      __syncwarp();
      int r = 0, nxt = binc[0];
      constexpr int CU = 4;
      for (int e0 = 0; e0 < total; e0 += 32 * CU) {
        int32_t yy[CU];
        int rw[CU], aa[CU];
#pragma unroll
        for (int k = 0; k < CU; k++) {
          const int e = e0 + 32 * k + lane;
          if (e < total) {
            while (e >= nxt) nxt = binc[++r];
            rw[k] = r;
            aa[k] = bra[r] + e;
            yy[k] = g.col[aa[k]];
          } else { rw[k] = 32 + lane; aa[k] = 0; yy[k] = -1; }  // idle lanes: a row of their own
        }
#pragma unroll
        for (int k = 0; k < CU; k++) {
          if (e0 + 32 * k >= total) break;  // uniform
          const bool keep = yy[k] >= 0 && test_bit(iw, yy[k]);
          const unsigned km = __ballot_sync(0xffffffffu, keep);
          // lanes of one row are contiguous: segment = [first lane of my row, first lane of the next row)
          const int up = __shfl_up_sync(0xffffffffu, rw[k], 1);
          const unsigned chg = __ballot_sync(0xffffffffu, lane == 0 || up != rw[k]);
          const int s0 = 31 - __clz(chg & (lanemask_lt() | (1u << lane)));
          const unsigned above = chg & ~((2u << lane) - 1u);  // segment starts above my lane
          const int s1 = above ? __ffs(above) - 1 : 32;
          const unsigned seg = (s1 == 32 ? 0xffffffffu : ((1u << s1) - 1u)) & ~((1u << s0) - 1u);
          const int cur = rw[k] < 32 ? bcur[rw[k]] : 0;
          __syncwarp();
          if (keep) {
            const int64_t o = ao + cur + __popc(km & seg & lanemask_lt());
            const double wgt = g.kappa[aa[k]] + 1.0;  // graph[a][b]['weight'] = kappa + 1   riccidist2dgm.py:225
            c.anb[o] = (uint32_t)local_id(iw, wbase, yy[k]);
            c.aw[o] = wgt;
            atomicMin(&bmw[rw[k]], __float_as_int(__double2float_rd(wgt)));  // positive floats order like ints
          }
          if (lane == s1 - 1 && rw[k] < 32) bcur[rw[k]] = cur + __popc(km & seg);
          __syncwarp();
        }
      }
      __syncwarp();
      if (has) {
        const int cntl = bcur[lane] - rbase;
        c.astart[vo + lx] = rbase;
        c.adeg[vo + lx] = cntl;
        c.aminw[vo + lx] = __int_as_float(bmw[lane]);  // smallest incident weight, rounded down
        kept_total += cntl;
      }
      __syncwarp();
    }
    const int m = block_reduce_sum(kept_total, sh.red) / 2;
    if (tid == 0) {
      c.tn[t] = n;
      c.tm[t] = m;
      const bool u_in = test_bit(iw, u);
      const bool v_in = node_mode ? u_in : test_bit(iw, v);
      c.tlu[t] = u_in ? local_id(iw, wbase, u) : -1;
      c.tlv[t] = node_mode ? c.tlu[t] : (v_in ? local_id(iw, wbase, v) : -1);
      uint8_t st = (u_in && v_in) ? TLC_ST_OK : TLC_ST_TRIVIAL;
      if (n == 0 || ((node_mode || p.mode == TLC_MODE_EDGE_FORCED) && m == 0)) st = TLC_ST_EMPTY;  // :318 / data_utils_NC.py:103-104
      c.tstatus[t] = st;
      c.tnp[t] = 0; c.tnpos[t] = 0; c.tnneg[t] = 0; c.tncls[t] = 0;
    }
  }
}

}  // namespace

int vicinity_grid(int device, const GraphView& g, const Params& p, size_t* bitmap_words, bool* use_smem) {
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  const size_t W = ((size_t)g.N + 31) / 32;
  *bitmap_words = W;
  const size_t need = 2 * W * sizeof(uint32_t);
  *use_smem = need <= 96 * 1024;
  int per_sm = 4;
  if (*use_smem && need > 0) {
    const size_t fit = (size_t)(200 * 1024) / (need + 2048);
    per_sm = (int)(fit < 1 ? 1 : (fit > 6 ? 6 : fit));
  }
  return prop.multiProcessorCount * per_sm;
}

static void set_smem(const void* fn, size_t bytes) {
  if (bytes > 48 * 1024) cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// targets == nullptr: the ball of every node with an edge (kernel 1t's table build needs them all)
void launch_ball_cache(const GraphView& g, const Params& p, const int32_t* targets, int64_t E, const VicinityScratch& vs,
                       cudaStream_t st) {
  if (!vs.ball_cache || (targets && E <= 0)) return;
  const int W = (g.N + 31) / 32;
  const bool smem = vs.bitmaps == nullptr;
  const size_t bytes = smem ? (size_t)2 * W * 4 : 0;
  cudaMemsetAsync(vs.ball_count, 0, sizeof(int), st);
  if (targets) {
    const int mgrid = (int)std::min<int64_t>((2 * E + 255) / 256, 4096);
    ball_mark_kernel<<<mgrid, 256, 0, st>>>(targets, E, p.mode == TLC_MODE_NODE ? 1 : 0, g, vs);
  } else {
    ball_mark_all_kernel<<<(g.N + 255) / 256, 256, 0, st>>>(g, vs);
  }
  count_launch();
  set_smem((const void*)ball_build_kernel, bytes);
  ball_build_kernel<<<vs.grid, K1_BLOCK, bytes, st>>>(g, p, vs, W, smem ? 1 : 0);
  count_launch();
}

void launch_vicinity_sizes(const GraphView& g, const Params& p, const int32_t* targets, int64_t E, int32_t* out_n,
                           int32_t* out_m, int32_t* out_ds, uint8_t* out_status, double* out_bytes,
                           const VicinityScratch& vs, int* work_counter, cudaStream_t st) {
  const int W = (g.N + 31) / 32;
  const bool smem = vs.bitmaps == nullptr;
  const size_t bytes = smem ? (size_t)2 * W * 4 : 0;
  set_smem((const void*)vicinity_kernel<false>, bytes);
  cudaMemsetAsync(work_counter, 0, sizeof(int), st);
  ChunkView dummy{};
  vicinity_kernel<false><<<vs.grid, K1_BLOCK, bytes, st>>>(g, p, targets, E, out_n, out_m, out_ds, out_status, out_bytes, dummy, vs,
                                                          work_counter, W, smem ? 1 : 0);
  count_launch();
}

void launch_vicinity_light(const GraphView& g, const Params& p, const int32_t* targets, int64_t E, int32_t* out_n,
                           int32_t* out_m, int32_t* out_ds, uint8_t* out_status, double* out_bytes,
                           const VicinityScratch& vs, int sm_count, cudaStream_t st) {
  const int W = (g.N + 31) / 32;
  const int64_t want = (E * 32 + 255) / 256;
  const int grid = (int)std::min<int64_t>(want, (int64_t)sm_count * 8);
  vicinity_light_kernel<<<grid, 256, 0, st>>>(g, p, targets, E, out_n, out_m, out_ds, out_status, out_bytes, vs, W);
  count_launch();
}

void launch_vicinity_fill(const GraphView& g, const Params& p, const ChunkView& c, const VicinityScratch& vs,
                          int* work_counter, cudaStream_t st) {
  const int W = (g.N + 31) / 32;
  const bool smem = vs.bitmaps == nullptr;
  const size_t bytes = smem ? (size_t)2 * W * 4 : 0;
  set_smem((const void*)vicinity_kernel<true>, bytes);
  cudaMemsetAsync(work_counter, 0, sizeof(int), st);
  const int grid = vs.grid < c.T ? vs.grid : c.T;
  vicinity_kernel<true><<<grid, K1_BLOCK, bytes, st>>>(g, p, c.tgt, c.T, nullptr, nullptr, nullptr, nullptr, nullptr, c, vs, work_counter,
                                                      W, smem ? 1 : 0);
  count_launch();
}

}  // namespace tlc
