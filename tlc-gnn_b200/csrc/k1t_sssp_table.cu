// k1t_sssp_table.cu -- kernel 1t: the node filtration from a per-ROOT shortest-path table of the root's k-hop ball.
//
// build_fv (riccidist2dgm.py:20-61) needs, for a target (u, v), the shortest-path distances from u and from v INSIDE the
// vicinity S.  Kernel 1b runs one Dijkstra per root and target.  On graphs small enough to afford O(N^2) entries the
// same values come from a table that is built ONCE per graph, hop k and root r over G'_r, the subgraph of G induced by
// r's closed k-hop ball:
//     D_r[x] = least fixpoint of d[y] = min_x fl(d[x] + w(x, y)) on G'_r       (what Dijkstra returns, fl(+) monotone)
//     P_r[x] = smallest id y with fl(D_r[y] + w(y, x)) == D_r[x]               (the tree rule of kernel 1b / the oracle)
//     Q_r[x] = python-order sum of the weights along x -> P_r[x] -> ... -> r   (:30,35, SURVEY.md F5)
//     W_r[x] = w(x, P_r[x]), the weight of the tree edge (the walks of the vertices below need it term by term)
// The proof below needs two facts: S is a vertex subset of G'_r, and the edges of S are edges of G'_r.  Both hold on
// the two modes that reach this kernel: TLC_MODE_EDGE (S = ball(u) & ball(v), induced) and TLC_MODE_NODE (S = ball(u));
// not on FORCED, UNION or REMOVEINTER, whose S leaves a root's ball (the host never gives those the tables).
// For a vicinity S containing r call x VALID when its whole tree branch x -> ... -> r lies in S.  Then, exactly:
//   * d_S[x] == D_r[x]: d_S >= D_r (fewer edges), and along the branch d_S[x] <= fl(d_S[p] + w) = fl(D_r[p] + w) = D_r[x];
//   * the tree parent inside S is P_r[x]: every candidate y in S (fl(d_S[y] + w) == d_S[x]) is a candidate in G'_r as
//     well (D_r[y] <= d_S[y] and D_r[x] is minimal), and P_r[x], the smallest candidate of G'_r, lies in S with d_S = D_r;
//   * hence the path and its python-order sum are Q_r[x].
// The ball table leaves no more vertices invalid than a table over the whole graph G would: if x's branch in G's tree
// lies in S, then along that branch (induction from r) the G'_r values equal G's -- D' >= D (fewer edges), the G branch
// is a path of G'_r so D' <= D, and every G'_r candidate for the parent is a G candidate, so the smallest is the same.
// Whole-graph shortest paths often leave the ball (weights kappa + 1 lie in (0.1, 1.9): a cheap path to a 2-hop vertex
// through a hub 3 hops away); inside the ball most of those vertices become valid.
// The other vertices of S (their branch leaves S: 5 % of the Computers-shaped 2-hop vicinities, from 2 % on the largest
// quarter to 17 % on the smallest -- scripts/table_census.py; 10 % with whole-graph tables)
// get their distance from the same fixpoint restricted to them, the valid vertices acting as settled sources: ONE pass of
// "pull" relaxations over THEIR graph rows (which also lists the adjacencies among the invalid vertices), further rounds
// over that list only, then the tree rule and the path walk (parents and tree-edge weights of all vertices in shared
// memory by then).  Results are bit-identical to kernel 1b (tests: the parity suite runs both; TLC_F_NO_TABLE selects
// kernel 1b).
//
// Rows read per target drop from 2 x D_S (every row of the vicinity, once per root) to the rows of the invalid
// vertices; the table rows of u and v (D, P, {Q, W}: 28 N bytes each) are gathered through the vertex list instead.
#include <cstdlib>

#include <cstdio>
#include <cstring>

#include "tlc_common.cuh"

namespace tlc {
namespace {

// ---------------------------------------------------------------------------------------------------------------------
// table build: one CTA per root, the root's ball, distances + parents in shared memory
// ---------------------------------------------------------------------------------------------------------------------
__global__ void sssp_mark_kernel(const int32_t* __restrict__ targets, int64_t E, int node_mode, GraphView g, SsspTables tb) {
  const int64_t total = 2 * E;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    if (node_mode && (i & 1)) continue;
    const int32_t x = targets[i];
    if (x < 0 || x >= g.N || g.rowptr[x + 1] == g.rowptr[x]) continue;
    if (tb.state[x] == 0 && atomicCAS(&tb.state[x], 0, 1) == 0) tb.list[atomicAdd(tb.count, 1)] = x;
  }
}

__global__ void sssp_mark_all_kernel(GraphView g, SsspTables tb) {  // every node with an edge whose row does not exist yet
  for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < g.N; x += gridDim.x * blockDim.x) {
    if (g.rowptr[x + 1] == g.rowptr[x]) continue;
    if (tb.state[x] == 0 && atomicCAS(&tb.state[x], 0, 1) == 0) tb.list[atomicAdd(tb.count, 1)] = x;
  }
}

constexpr int BQ = 2048;  // vertices settled per phase at most
struct BuildShared {
  int32_t q[BQ];
  int32_t qn, qhead;
  unsigned long long dmin;
  int32_t any;
};

// The graph of root r's table is G'_r, the subgraph induced by r's closed k-hop ball (the ball cache row of r, which must
// hold the call's hop): an edge is relaxed only into a member of the ball.  Vertices outside it keep D = +inf, P = -1,
// Q = NO_PATH_DIST, W = 0 (kernel 1t never reads them: S is a subset of the ball).  gminw, the smallest weight of a
// vertex's WHOLE-graph row, stays a valid settling margin: the edges of G'_r into x are a subset of those of G, so their
// smallest weight is at least gminw[x].  The host launches one CTA per SM (pw_scratch has one row per CTA); saying so in
// the launch bounds lets ptxas use up to 64 registers instead of spilling at 32.
__global__ void __launch_bounds__(1024, 1) sssp_build_kernel(GraphView g, SsspTables tb, const uint32_t* __restrict__ ball_cache,
                                                          const float* __restrict__ gminw, double* __restrict__ pw_scratch,
                                                          int plain) {
  extern __shared__ __align__(16) unsigned long long bsm[];
  __shared__ BuildShared sh;
  const int N = g.N, W = (N + 31) / 32;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  unsigned long long* dist = bsm;                                   // [N]
  int32_t* par = reinterpret_cast<int32_t*>(bsm + N);               // [N]
  uint32_t* ball = reinterpret_cast<uint32_t*>(par + N);            // [W]  the root's ball
  uint8_t* state = reinterpret_cast<uint8_t*>(ball + W);            // [N]  0 far, 1 tentative, 2 done
  double* pw = pw_scratch + (size_t)blockIdx.x * N;                 // weight of the parent edge (global scratch of this CTA)
  const int cnt = *tb.count;
  for (int idx = blockIdx.x; idx < cnt; idx += gridDim.x) {
    const int32_t root = tb.list[idx];
    __syncthreads();
    for (int x = tid; x < N; x += nt) { dist[x] = INF_BITS; state[x] = 0; par[x] = -1; }
    for (int w = tid; w < W; w += nt) ball[w] = ball_cache[(size_t)root * W + w];
    __syncthreads();
    if (tid == 0) { dist[root] = 0ull; state[root] = 1; }
    __syncthreads();
    for (int phase = 0; phase < 2 * N + 2; phase++) {
      // smallest tentative distance
      if (tid == 0) { sh.dmin = INF_BITS; sh.qn = 0; sh.qhead = 0; }
      __syncthreads();
      unsigned long long lm = INF_BITS;
      for (int x = tid; x < N; x += nt) if (state[x] == 1) { const unsigned long long d = dist[x]; lm = d < lm ? d : lm; }
      lm = warp_min_u64(lm);
      if (lane == 0 && lm != INF_BITS) atomicMin(&sh.dmin, lm);
      __syncthreads();
      const unsigned long long dminb = sh.dmin;
      if (dminb == INF_BITS) break;
      const double dmin = __longlong_as_double((long long)dminb);
      // settle every tentative x with d[x] <= fl(dmin + minw[x])   (Crauser et al.'s IN criterion, exact by monotonicity of fl)
      for (int x = tid; x < N; x += nt) {
        if (state[x] != 1) continue;
        if (__longlong_as_double((long long)dist[x]) <= __dadd_rn(dmin, (double)gminw[x])) {
          const int pos = atomicAdd(&sh.qn, 1);
          if (pos < BQ) { state[x] = 2; sh.q[pos] = x; }
        }
      }
      __syncthreads();
      const int qn = min(sh.qn, BQ);
      // relax the settled rows: a warp per row, rows handed out by a shared counter
      for (;;) {
        int i = 0;
        if (lane == 0) i = atomicAdd(&sh.qhead, 1);
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i >= qn) break;
        const int x = sh.q[i];
        const double dx = __longlong_as_double((long long)dist[x]);
        const int a = g.rowptr[x], b = g.rowptr[x + 1];
        for (int e = a + lane; e < b; e += 32) {
          const int y = g.col[e];
          if (!test_bit(ball, y)) continue;
          const unsigned long long tbv = (unsigned long long)__double_as_longlong(__dadd_rn(dx, __dadd_rn(g.kappa[e], 1.0)));
          if (tbv < dist[y]) { atomicMin(&dist[y], tbv); if (state[y] == 0) state[y] = 1; }
        }
      }
      __syncthreads();
    }
    __syncthreads();
    // tree rule: parent[x] = smallest id y with fl(d[y] + w) == d[x] (rows ascend: the first matching position)
    for (int x = wid; x < N; x += nw) {
      const unsigned long long dxb = dist[x];
      if (x == root || dxb == INF_BITS) continue;
      const int a = g.rowptr[x], b = g.rowptr[x + 1];
      for (int e0 = a; e0 < b; e0 += 32) {
        const int e = e0 + lane;
        bool hit = false;
        double w = 0.0;
        int y = 0;
        if (e < b) {
          y = g.col[e];
          w = __dadd_rn(g.kappa[e], 1.0);
          const unsigned long long dyb = dist[y];
          hit = dyb != INF_BITS && (unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dyb), w)) == dxb;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, hit);
        if (bal) {
          if (lane == __ffs(bal) - 1) { par[x] = y; pw[x] = w; }
          break;
        }
      }
    }
    __threadfence_block();
    __syncthreads();
    // outputs: D (bit pattern as double), P, {Q (python-order path sum; 100 where the root does not reach x:
    // riccidist2dgm.py:31-32), W}
    double* Drow = tb.D + (size_t)root * N;
    int32_t* Prow = tb.P + (size_t)root * N;
    double2* QWrow = tb.QW + (size_t)root * N;
    for (int x = tid; x < N; x += nt) {
      const unsigned long long dxb = dist[x];
      const int32_t px = par[x];
      double res;
      if (x == root) res = 0.0;
      else if (dxb == INF_BITS || px < 0) res = NO_PATH_DIST;
      else {
        PySum ps{0.0, 0.0, 0};
        int y = x, guard = 0;
        while (y != root && guard++ <= N) { pysum_add(ps, pw[y], plain != 0); y = par[y]; }
        res = pysum_get(ps, plain != 0);
      }
      Drow[x] = __longlong_as_double((long long)dxb);
      Prow[x] = px;
      QWrow[x] = make_double2(res, px >= 0 ? pw[x] : 0.0);
    }
    __syncthreads();
    if (tid == 0) { __threadfence(); tb.state[root] = 2; }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// kernel 1t proper: one CTA per target of the graph-row route
// ---------------------------------------------------------------------------------------------------------------------
struct TableShared {
  double redd[32];
  int32_t wsum[33];
  int32_t ninv;     // invalid vertices of the current root
  int32_t nextra;   // further chunks of their long rows
  int32_t dinv;     // sum of their graph degrees
  int32_t nia;      // entries of the list of invalid-invalid adjacencies
  int32_t any;
};
#ifdef T1_PROFILE
__device__ unsigned long long g_t1prof[24];
#define TPROF(i) do { if (tid == 0) { const long long tnow_ = clock64(); atomicAdd(&g_t1prof[i], (unsigned long long)(tnow_ - tprev_)); tprev_ = tnow_; } } while (0)
#else
#define TPROF(i) do { } while (0)
#endif


__global__ void __launch_bounds__(1024) filtration_table_kernel(Params p, ChunkView c, int t0, int cap, GraphView g,
                                                                const uint32_t* __restrict__ ball_cache, SsspTables tb, int W) {
  extern __shared__ __align__(16) unsigned long long dynt[];
  __shared__ TableShared sh;
  const int t = t0 + blockIdx.x;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  const bool node_mode = p.mode == TLC_MODE_NODE;
  const int64_t vo = c.voff[t];
  const int N = g.N;
  // dynamic shared memory: dist u64[cap] | parent local id u16[cap] | class u8[cap] | bitmap + ranks u32[2W] | local ids u16[N]
  unsigned long long* dist = dynt;
  uint16_t* parl = reinterpret_cast<uint16_t*>(dynt + cap);
  uint8_t* cls = reinterpret_cast<uint8_t*>(parl + cap);
  uint32_t* bm = reinterpret_cast<uint32_t*>(reinterpret_cast<unsigned char*>(dynt) + (size_t)cap * 11);
  uint16_t* lid = reinterpret_cast<uint16_t*>(bm + 2 * W);

#ifdef T1_PROFILE
  long long tprev_ = clock64();
#endif
  // ---- 0. the vicinity (as kernel 1b's graph-row prologue): nodes = set(nodes_u) & set(nodes_v), local ids = ranks   :311-316
  const int64_t ti = c.tidx[t];
  const int32_t u = c.tgt[2 * ti], v = c.tgt[2 * ti + 1];
  if (unknown_target(g, u, v, node_mode)) {
    if (tid == 0) { c.tn[t] = 0; c.tnp[t] = 0; c.tnpos[t] = 0; c.tnneg[t] = 0; c.tlu[t] = -1; c.tlv[t] = -1;
                    c.tstatus[t] = TLC_ST_UNKNOWN_NODE; }
    return;
  }
  const int n = graph_row_bitmap(c, t, ball_cache, W, u, v, node_mode, bm, sh.wsum);
  {
    uint32_t* l32 = reinterpret_cast<uint32_t*>(lid);
    for (int i = tid; i < (N + 1) / 2; i += nt) l32[i] = 0xffffffffu;
  }
  __syncthreads();
  for (int w = wid; w < W; w += nw) {  // a warp per bitmap word: vertex list, graph rows, graph id -> local id
    const uint32_t bits = bm[w];
    if (!((bits >> lane) & 1u)) continue;
    const int lx = (int)bm[W + w] + __popc(bits & lanemask_lt());
    const int32_t x = w * 32 + lane;
    const int32_t ra = g.rowptr[x];
    c.vert[vo + lx] = x;
    c.astart[vo + lx] = ra;
    c.adeg[vo + lx] = g.rowptr[x + 1] - ra;
    lid[x] = (uint16_t)lx;
  }
  const int lu = bitmap_rank(bm, W, u);
  const int lv = node_mode ? lu : bitmap_rank(bm, W, v);
  uint8_t st0 = (lu >= 0 && lv >= 0) ? TLC_ST_OK : TLC_ST_TRIVIAL;
  if (n == 0 || (node_mode && n == 1)) st0 = TLC_ST_EMPTY;  // :318 / data_utils_NC.py:103-104
  if (tid == 0) {
    c.tn[t] = n; c.tlu[t] = lu; c.tlv[t] = lv; c.tstatus[t] = st0;
    if (c.count_m) c.tm[t] = 0;  // batch call: the induced edges are not counted on this route (nobody reads all rows)
    c.tnp[t] = 0; c.tnpos[t] = 0; c.tnneg[t] = 0; c.tncls[t] = 0;
  }
  __syncthreads();
      TPROF(0);
  if (n == 0 || st0 > TLC_ST_TRIVIAL) return;

  const int32_t* __restrict__ vert = c.vert + vo;
  double* d1 = c.d1 + vo;
  double* d2 = c.d2 + vo;
  double* fval = c.fval + vo;
  int32_t* hint = c.neg + vo;     // tree parent towards the last root (kernel 2v's "neighbour in an earlier block" hint)
  int32_t* hint0 = c.vcls + vo;   // ... and towards the first root
  int32_t* inv = c.vs0 + vo;      // list of the invalid vertices of the current root
  int32_t* extra = c.vs1 + vo;    // further row chunks of the long invalid rows: local vertex id << 12 | chunk
  int32_t* bpos = c.vs2 + vo;     // per vertex: smallest row position of a tree-parent candidate
  uint32_t* iap = reinterpret_cast<uint32_t*>(c.vord + vo);   // invalid-invalid adjacency: vertex << 16 | neighbour ...
  int32_t* iaq = c.vrank + vo;                                // ... and the row position of the entry; slots n .. 2n - 1:
  uint2* ia2 = reinterpret_cast<uint2*>(c.v64a + vo);
  uint2* ia3 = reinterpret_cast<uint2*>(c.v64c + vo);
  uint2* ia4 = reinterpret_cast<uint2*>(c.fval + vo);       // (the filtration values are written at the very end)
  const bool roots_in = lu >= 0 && lv >= 0;
  const bool plain = (p.flags & TLC_F_SUM_PLAIN) != 0;
  const bool two = roots_in && !node_mode && lu != lv;
  constexpr uint8_t UNKNOWN = 0, VALID = 1, INVALID = 2, UNREACH = 3;

  if (!roots_in) {
    // nx.NodeNotFound for every vertex
    for (int x = tid; x < n; x += nt) { d1[x] = NO_PATH_DIST; d2[x] = NO_PATH_DIST; hint[x] = -1; hint0[x] = -1; }
  } else {
    for (int r = 0; r < (two ? 2 : 1); r++) {
      const int root = r == 0 ? lu : lv;
      const int32_t groot = r == 0 ? u : v;
      const double* __restrict__ Drow = tb.D + (size_t)groot * N;
      const int32_t* __restrict__ Prow = tb.P + (size_t)groot * N;
      const double2* __restrict__ QWrow = tb.QW + (size_t)groot * N;
      double* out = r == 0 ? d1 : d2;
      int32_t* hnt = r == 0 ? hint0 : hint;
      if (tid == 0) { sh.ninv = 0; sh.nextra = 0; sh.dinv = 0; sh.nia = 0; }
      // ---- 1. classes: the branch of x stays in S <=> its table parent is in S and is valid itself ----
      // Four vertices per thread with their loads in flight together: first their graph ids, then their D and P, only
      // then the local ids of the parents (each vertex alone would be two dependent global round trips)
      for (int x0 = tid; x0 < n; x0 += 4 * nt) {
        int32_t gx4[4];
#pragma unroll
        for (int k = 0; k < 4; k++) { const int x = x0 + k * nt; gx4[k] = x < n ? vert[x] : -1; }
        double d4[4];
        int32_t p4[4];
#pragma unroll
        for (int k = 0; k < 4; k++) { d4[k] = gx4[k] >= 0 ? Drow[gx4[k]] : 0.0; p4[k] = gx4[k] >= 0 ? Prow[gx4[k]] : -1; }
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const int x = x0 + k * nt;
          if (x >= n) continue;
          uint8_t cl;
          uint16_t pl = 0xffff;
          if (x == root) cl = VALID;
          else {
            const int32_t gp = p4[k];
            pl = gp >= 0 ? lid[gp] : (uint16_t)0xffff;
            cl = pl == 0xffff ? INVALID : UNKNOWN;
          }
          cls[x] = cl; parl[x] = pl;
          dist[x] = (unsigned long long)__double_as_longlong(d4[k]);
          if (r == 0) { hint[x] = -1; hint0[x] = -1; }
        }
      }
      __syncthreads();
      TPROF(1);
      for (int round = 0; round <= n; round++) {
        int ch = 0;
        for (int x = tid; x < n; x += nt) {
          if (cls[x] != UNKNOWN) continue;
          const uint8_t pc = cls[parl[x]];
          if (pc != UNKNOWN) { cls[x] = pc; ch = 1; }   // (a stale read only delays the vertex to the next round)
          else ch = 1;
        }
        if (!__syncthreads_or(ch)) break;
      }
      TPROF(2);
      // ---- 2. the invalid vertices, their distances by pull relaxations over their own graph rows ----
      // Work items are row CHUNKS: item i < ninv is the first chunk of invalid vertex i, the further chunks of the long
      // rows (hubs) are listed once per root in extra[] -- a hub's row is then spread over many warps instead of stalling
      // one.  A chunk's best candidate goes into the vertex's distance with a shared-memory atomic min.
      for (int x0 = 0; x0 < n; x0 += nt) {
        const int x = x0 + tid;
        const bool iv = x < n && cls[x] == INVALID;
        const unsigned bal = __ballot_sync(0xffffffffu, iv);
        int base = 0;
        if (bal && lane == 0) base = atomicAdd(&sh.ninv, __popc(bal));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (iv) {
          const int32_t gx = vert[x];
          inv[base + __popc(bal & lanemask_lt())] = x;
          dist[x] = INF_BITS; bpos[x] = 0x7fffffff;
          atomicAdd(&sh.dinv, g.rowptr[gx + 1] - g.rowptr[gx]);
        }
      }
      __syncthreads();
      TPROF(3);
      const int ninv = sh.ninv;
      // chunk size: EIGHT LANES walk a chunk together (one 128-byte line of records per step); about four chunks per
      // 8-lane group, between 32 and 512 records -- then doubled until the extra chunks fit the n slots of extra[]
      int chunk = min(512, max(32, ((sh.dinv / (nt / 2) + 31) / 32) * 32));
      while (sh.dinv / chunk > n / 2) chunk *= 2;
      for (int i = tid; i < ninv; i += nt) {
        const int32_t gx = vert[inv[i]];
        const int cnt = (g.rowptr[gx + 1] - g.rowptr[gx] + chunk - 1) / chunk;
        if (cnt > 1) {
          const int at = atomicAdd(&sh.nextra, cnt - 1);
          for (int j = 1; j < cnt; j++) extra[at + j - 1] = (inv[i] << 12) | j;
        }
      }
      __syncthreads();
      TPROF(4);
      const int nextra = sh.nextra, nitems = ninv + nextra;
      // Eight lanes walk a chunk: their 16-byte record loads fall into one 128-byte line per step (one L1 wavefront; a lane
      // per chunk costs a wavefront per record, a warp per chunk leaves most lanes idle on these 25 - 100-record rows and
      // pays a 32-lane reduction per row -- both measured slower).  Four loads in flight per lane, a 3-step reduction.
      const int l8 = lane & 7, grp = tid >> 3, ngrp = nt >> 3;
      const unsigned gm = 0xffu << (lane & 24);  // the lanes of this 8-lane group
      constexpr int ITEM_RESCAN = 1 << 30;  // item flag: its invalid neighbours did not all fit the list -> later rounds reread the chunk
      auto item_bounds = [&](int i, int& x, int& a, int& b, bool flagged_only) {
        const int raw = i < ninv ? inv[i] : extra[i - ninv];
        const int pk = i < ninv ? ((raw & 0xffff) << 12) : (raw & (ITEM_RESCAN - 1));
        x = pk >> 12;
        const int ra = c.astart[vo + x];
        a = ra + (pk & 4095) * chunk;
        b = min(ra + c.adeg[vo + x], a + chunk);
        if (flagged_only && !(raw & ITEM_RESCAN)) b = a;
      };
      // The FIRST round reads every invalid row once.  The valid neighbours' distances are final: their candidates never
      // need a second look.  The invalid neighbours go into a list of (vertex, neighbour, row position) entries -- the
      // graph among the invalid vertices, a few entries per vertex, every pair once (weights are symmetric, the later
      // rounds relax an entry both ways) -- and the following rounds run over that list only
      // (measured: 3 rounds, the second changes 2 - 5 % of the vertices, the third none).  A list that outgrows its 4n
      // slots (small vicinities that are mostly invalid) sends the root back to rounds over the rows.
      auto ia_put = [&](int k, uint32_t pr, int pos) {
        if (k < n) { iap[k] = pr; iaq[k] = pos; }
        else if (k < 2 * n) ia2[k - n] = make_uint2(pr, (uint32_t)pos);
        else if (k < 3 * n) ia3[k - 2 * n] = make_uint2(pr, (uint32_t)pos);
        else if (k < 4 * n) ia4[k - 3 * n] = make_uint2(pr, (uint32_t)pos);
      };
      auto ia_get = [&](int k, uint32_t& pr, int& pos) {
        if (k < n) { pr = iap[k]; pos = iaq[k]; return; }
        const uint2 v2 = k < 2 * n ? ia2[k - n] : k < 3 * n ? ia3[k - 2 * n] : ia4[k - 3 * n];
        pr = v2.x; pos = (int)v2.y;
      };
      // List slots without atomics: every warp owns a region of 4n / nw slots and counts its entries in a register (one
      // warp vote per record slot; the single shared counter this replaces serialised 2 600 atomics per root -- 100 k cycles,
      // most of the first round).  The later rounds: a warp walks its own region.
      const int capw = (4 * n) / nw;
      int cntw = 0;
      auto relax_rows = [&](bool first) -> int {
        int ch = 0;
        for (int kb = 0; kb * ngrp < nitems; kb += 8) {   // (uniform trip counts: the shuffles below are group-wide)
          // the group's next eight items, their bounds fetched lane-parallel (vertex -> row start, degree: a dependent chain)
          int mx = 0, ma = 0, mb = 0;
          { const int itl = (kb + l8) * ngrp + grp; if (itl < nitems) item_bounds(itl, mx, ma, mb, !first); }
          for (int j = 0; j < 8; j++) {
            const int x = __shfl_sync(gm, mx, j, 8), a = __shfl_sync(gm, ma, j, 8), b = __shfl_sync(gm, mb, j, 8);
            int trips = (b - a + 31) >> 5;  // the longest of the warp's four chunks: the votes below are warp-wide
            trips = max(trips, __shfl_xor_sync(0xffffffffu, trips, 8));
            trips = max(trips, __shfl_xor_sync(0xffffffffu, trips, 16));
            unsigned long long best = INF_BITS;
            for (int t5 = 0; t5 < trips; t5++) {
              const int e0 = a + l8 + 32 * t5;
              uint4 rc[4];
#pragma unroll
              for (int q = 0; q < 4; q++) rc[q] = e0 + 8 * q < b ? __ldg(g.rec + e0 + 8 * q) : make_uint4(0xffffffffu, 0u, 0u, 0u);
#pragma unroll
              for (int q = 0; q < 4; q++) {
                uint16_t ly = 0xffff;
                if (rc[q].x != 0xffffffffu) ly = lid[rc[q].x];
                if (first) {
                  const bool need = ly != 0xffff && (int)ly > x && cls[ly] == INVALID;  // (a pair is listed once, by its smaller end)
                  const unsigned m = __ballot_sync(0xffffffffu, need);
                  if (need) {
                    const int slot = cntw + __popc(m & lanemask_lt());
                    if (slot < capw) ia_put(wid * capw + slot, ((uint32_t)x << 16) | ly, e0 + 8 * q);
                  }
                  cntw += __popc(m);
                }
                if (ly == 0xffff) continue;
                const double w = __hiloint2double((int)rc[q].w, (int)rc[q].z);
                const unsigned long long dyb = dist[ly];
                if (!first && cls[ly] == INVALID) {  // a reread chunk also pushes: the pairs it would have listed go both ways
                  const unsigned long long dxb = dist[x];
                  if (dxb != INF_BITS) {
                    const unsigned long long c2 = (unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dxb), w));
                    if (c2 < dyb && c2 < atomicMin(&dist[ly], c2)) ch = 1;
                  }
                }
                if (dyb == INF_BITS) continue;
                const unsigned long long cand = (unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dyb), w));
                best = cand < best ? cand : best;
              }
            }
#pragma unroll
            for (int o = 4; o; o >>= 1) { const unsigned long long u2 = __shfl_xor_sync(gm, best, o); best = u2 < best ? u2 : best; }
            if (l8 == 0 && b > a && best < dist[x] && best < atomicMin(&dist[x], best)) ch = 1;
            if (first && cntw > capw && l8 == 0 && b > a) {  // the warp's region is full: this chunk stays on the row path
              const int itj = (kb + j) * ngrp + grp;
              if (itj < ninv) inv[itj] |= ITEM_RESCAN; else extra[itj - ninv] |= ITEM_RESCAN;
            }
          }
        }
        return ch;
      };
      relax_rows(true);
      const bool full = __syncthreads_or(cntw > capw ? 1 : 0) != 0;  // some chunks are flagged for rereading
      TPROF(5);
      const int nlist = min(cntw, capw);
      // the first 128 entries of the warp's region stay in registers over the rounds (vertex pair + edge weight): a round is
      // then shared-memory work only, not two dependent global loads per entry
      uint32_t epr[4];
      double ewt[4];
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const int k = lane + 32 * i;
        epr[i] = 0xffffffffu; ewt[i] = 0.0;
        if (k < nlist) {
          int pos;
          ia_get(wid * capw + k, epr[i], pos);
          const uint4 rc = __ldg(g.rec + pos);
          ewt[i] = __hiloint2double((int)rc.w, (int)rc.z);
        }
      }
#ifdef T1_PROFILE
      long long tlr0_ = clock64();
      int nrounds_ = 0;
#endif
      for (int round = 1; round <= ninv + 1; round++) {
        int ch = 0;
#ifdef T1_PROFILE
        nrounds_++;
#endif
#pragma unroll
        for (int i = 0; i < 4; i++) {
          if (epr[i] == 0xffffffffu) continue;
          const int x = (int)(epr[i] >> 16), ly = (int)(epr[i] & 0xffffu);
          const unsigned long long dyb = dist[ly], dxb = dist[x];
          if (dyb != INF_BITS) {
            const unsigned long long cand = (unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dyb), ewt[i]));
            if (cand < dxb && cand < atomicMin(&dist[x], cand)) ch = 1;
          }
          if (dxb != INF_BITS) {
            const unsigned long long c2 = (unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dxb), ewt[i]));
            if (c2 < dyb && c2 < atomicMin(&dist[ly], c2)) ch = 1;
          }
        }
        for (int k = lane + 128; k < nlist; k += 32) {
          uint32_t pr; int pos;
          ia_get(wid * capw + k, pr, pos);
          const int x = (int)(pr >> 16), ly = (int)(pr & 0xffffu);
          const unsigned long long dyb = dist[ly], dxb = dist[x];
          if (dyb == INF_BITS && dxb == INF_BITS) continue;
          const uint4 rc = __ldg(g.rec + pos);
          const double w = __hiloint2double((int)rc.w, (int)rc.z);
          if (dyb != INF_BITS) {
            const unsigned long long cand = (unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dyb), w));
            if (cand < dxb && cand < atomicMin(&dist[x], cand)) ch = 1;
          }
          if (dxb != INF_BITS) {
            const unsigned long long c2 = (unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dxb), w));
            if (c2 < dyb && c2 < atomicMin(&dist[ly], c2)) ch = 1;
          }
        }
        if (full) ch |= relax_rows(false);  // the flagged chunks, from their rows
        if (!__syncthreads_or(ch)) break;
      }
      TPROF(6);
#ifdef T1_PROFILE
      if (lane == 0) atomicAdd(&g_t1prof[15], (unsigned long long)cntw);
      if (tid == 0) { atomicAdd(&g_t1prof[17], (unsigned long long)nrounds_); if (full) atomicAdd(&g_t1prof[16], (unsigned long long)(clock64() - tlr0_)); }
      if (tid == 0) { atomicAdd(&g_t1prof[11], (unsigned long long)(full ? 1 : 0)); atomicAdd(&g_t1prof[12], 1ull); atomicAdd(&g_t1prof[13], (unsigned long long)nitems); atomicAdd(&g_t1prof[14], (unsigned long long)sh.dinv); }
#endif
      // ---- 3. tree rule for the invalid vertices: smallest local id y (= smallest row position) with fl(d[y] + w) == d[x] ----
      for (int kb = 0; kb * ngrp < nitems; kb += 8) {
        int mx = 0, ma = 0, mb = 0;
        { const int itl = (kb + l8) * ngrp + grp; if (itl < nitems) item_bounds(itl, mx, ma, mb, false); }
        for (int j = 0; j < 8; j++) {
        const int x = __shfl_sync(gm, mx, j, 8), a = __shfl_sync(gm, ma, j, 8);
        int b = __shfl_sync(gm, mb, j, 8);
        const unsigned long long dxb = b > a ? dist[x] : INF_BITS;
        if (dxb == INF_BITS) b = a;
        int hit = 0x7fffffff;
        for (int e0 = a; e0 < b; e0 += 32) {   // (uniform over the group: the exit test below is a group vote)
          uint4 rc[4];
#pragma unroll
          for (int q = 0; q < 4; q++) rc[q] = e0 + l8 + 8 * q < b ? __ldg(g.rec + e0 + l8 + 8 * q) : make_uint4(0xffffffffu, 0u, 0u, 0u);
#pragma unroll
          for (int q = 3; q >= 0; q--) {
            if (rc[q].x == 0xffffffffu) continue;
            const uint16_t ly = lid[rc[q].x];
            if (ly == 0xffff) continue;
            const unsigned long long dyb = dist[ly];
            if (dyb != INF_BITS && (unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dyb), __hiloint2double((int)rc[q].w, (int)rc[q].z))) == dxb)
              hit = e0 + l8 + 8 * q;
          }
          if (__ballot_sync(gm, hit != 0x7fffffff)) break;   // (the group's own vote: groups leave at different times)
        }
#pragma unroll
        for (int o = 4; o; o >>= 1) hit = min(hit, __shfl_xor_sync(gm, hit, o));
        if (l8 == 0 && hit != 0x7fffffff) atomicMin(&bpos[x], hit);
        }
      }
      __syncthreads();
      TPROF(7);
      // ---- 4. parents and outputs (phase "parents"): from here on the distances are not needed any more and every
      // vertex's 8-byte slot holds the weight of its tree edge instead, so that the walks below stay in shared memory.
      // A valid vertex's {Q, W} (one 16-byte load) gives that weight and its output, the table's path sum; four valid
      // vertices per thread with their loads in flight together.  An
      // invalid vertex takes its parent from the tree rule's row position, or is unreachable (nx.NetworkXNoPath:
      // disconnected vicinity, status 3 later).  The root and the unreachable vertices keep the hint -1.
      for (int x0 = tid; x0 < n; x0 += 4 * nt) {
        int32_t gx4[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const int x = x0 + k * nt;
          gx4[k] = x < n && x != root && cls[x] == VALID ? vert[x] : -1;
        }
        double2 e4[4];
#pragma unroll
        for (int k = 0; k < 4; k++) e4[k] = gx4[k] >= 0 ? QWrow[gx4[k]] : make_double2(0.0, 0.0);
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const int x = x0 + k * nt;
          if (x >= n) continue;
          unsigned long long wb = 0;
          if (x == root) out[x] = 0.0;
          else if (gx4[k] >= 0) {
            wb = (unsigned long long)__double_as_longlong(e4[k].y);
            out[x] = e4[k].x;
            hnt[x] = (int32_t)parl[x];
          } else {
            const int pos = bpos[x];
            if (dist[x] != INF_BITS && pos != 0x7fffffff) {
              const uint4 rc = __ldg(g.rec + pos);
              const uint16_t pl = lid[rc.x];
              parl[x] = pl;
              hnt[x] = (int32_t)pl;
              wb = ((unsigned long long)rc.w << 32) | rc.z;
            } else { cls[x] = UNREACH; out[x] = NO_PATH_DIST; }
          }
          dist[x] = wb;
        }
      }
      __syncthreads();
      TPROF(8);
      // ---- 5. path sums of the invalid vertices (phase "path_sums"): a walk in python order   :30,35 ----
      for (int i = tid; i < ninv; i += nt) {
        const int x = inv[i] & 0xffff;  // (without the rescan flag)
        if (cls[x] == UNREACH) continue;
        PySum ps{0.0, 0.0, 0};
        int y = x, guard = 0;
        while (y != root && guard++ <= n) {
          const int py = (int)parl[y];
          pysum_add(ps, __longlong_as_double((long long)dist[y]), plain);
          y = py;
        }
        out[x] = pysum_get(ps, plain);
      }
      __syncthreads();
      TPROF(9);
    }
    if (!two) for (int x = tid; x < n; x += nt) d2[x] = d1[x];
    __syncthreads();
    if (tid == 0) zero_roots(d1, d2, lu, lv);
  }
  __syncthreads();

  // ---- 6. descriptors + normalisation   riccidist2dgm.py:47-56 ; data_utils_NC.py:52-54 ----
  double mx = -1.0, sm = -1.0;
  for (int x = tid; x < n; x += nt) {
    const double a = d1[x], b = d2[x];
    mx = fmax(mx, fv_descriptor(TLC_DESC_MAX, node_mode, a, b));
    sm = fmax(sm, fv_descriptor(TLC_DESC_SUM, node_mode, a, b));
  }
  double smax = block_reduce_max(mx, sh.redd);
  double ssum = block_reduce_max(sm, sh.redd);
  const bool norm = (p.flags & TLC_F_NORM) != 0;
  if (norm && !fv_normalisers(p.flags, smax, ssum)) {
    if (tid == 0) c.tstatus[t] = TLC_ST_DEGENERATE;
    return;
  }
  for (int x = tid; x < n; x += nt) fval[x] = fv_value(p.descriptor, node_mode, norm, smax, ssum, d1[x], d2[x]);
  TPROF(10);
}

}  // namespace

// build the table rows of the targets' endpoints that do not exist yet (once per graph, hop and root); the ball cache
// must hold the ball of every root built
// targets == nullptr: every node of the graph (the eager build of the first call)
void launch_sssp_build(const GraphView& g, const Params& p, const int32_t* targets, int64_t E, const SsspTables& tb,
                       const uint32_t* ball_cache, const float* gminw, double* pw_scratch, int grid, cudaStream_t st) {
  if (!tb.D) return;
  cudaMemsetAsync(tb.count, 0, sizeof(int), st);
  if (targets) {
    if (E <= 0) return;
    const int mgrid = (int)std::min<int64_t>((2 * E + 255) / 256, 4096);
    sssp_mark_kernel<<<mgrid, 256, 0, st>>>(targets, E, p.mode == TLC_MODE_NODE ? 1 : 0, g, tb);
  } else {
    sssp_mark_all_kernel<<<(g.N + 255) / 256, 256, 0, st>>>(g, tb);
  }
  count_launch();
  const size_t bytes = sssp_build_smem(g.N);
  cudaFuncSetAttribute((const void*)sssp_build_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  cudaFuncSetAttribute((const void*)sssp_build_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  sssp_build_kernel<<<grid, 1024, bytes, st>>>(g, tb, ball_cache, gminw, pw_scratch, (p.flags & TLC_F_SUM_PLAIN) ? 1 : 0);
  count_launch();
}

// distances, parents, the root's ball bitmap, states (N = 16 384: 213 KB, 222 KB with the static BuildShared)
size_t sssp_build_smem(int N) { return (size_t)N * (8 + 4 + 1) + (size_t)(N + 31) / 32 * 4 + 16; }

void launch_filtration_table(const GraphView& g, const Params& p, const ChunkView& c, const VicinityScratch& vs,
                             const SsspTables& tb, int t0, int cnt, int block, int64_t n_max, cudaStream_t st) {
  const int W = (g.N + 31) / 32;
  const int cap = (int)((n_max + 7) / 8 * 8);
  const size_t bytes = (size_t)cap * 11 + (size_t)2 * W * 4 + ((size_t)g.N + 1) / 2 * 4 + 16;
  if (block < 128) block = 128;
  if (bytes + sizeof(TableShared) > 110 * 1024 && block >= 512) block = 1024;  // one resident CTA per SM: give it 32 warps
  if (const char* env = getenv("TLC_TABLE_BLOCK")) block = atoi(env);  // (tuning experiments)
  cudaFuncSetAttribute((const void*)filtration_table_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  cudaFuncSetAttribute((const void*)filtration_table_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
#ifdef T1_PROFILE
  if (getenv("T1_PROFILE_DUMP")) {  // ticks of thread 0 per phase, summed over the CTAs since the last dump
    unsigned long long h[24];
    cudaMemcpyFromSymbol(h, g_t1prof, sizeof h);
    static const char* nm[11] = {"prologue", "class_init", "class_rounds", "compaction", "chunks", "first_round", "later_rounds",
                                 "tree_rule", "parents", "path_sums", "descriptors"};
    unsigned long long tot = 0;
    for (int i = 0; i < 11; i++) tot += h[i];
    if (tot) {
      fprintf(stderr, "[1t profile]");
      for (int i = 0; i < 11; i++) fprintf(stderr, " %s %.1f%%", nm[i], 100.0 * (double)h[i] / (double)tot);
      fprintf(stderr, " | total %.1f Mticks | roots %llu, with flagged chunks %llu, items/root %.0f, records/root %.0f, list entries/root %.0f\n", (double)tot / 1e6,
              h[12], h[11], (double)h[13] / (double)(h[12] ? h[12] : 1), (double)h[14] / (double)(h[12] ? h[12] : 1), (double)h[15] / (double)(h[12] ? h[12] : 1));
      fprintf(stderr, "[1t profile] later rounds per root %.2f; ticks of the later rounds spent in roots with flagged chunks: %.1f Mticks\n", (double)h[17] / (double)(h[12] ? h[12] : 1), (double)h[16] / 1e6);
    }
    memset(h, 0, sizeof h);
    cudaMemcpyToSymbol(g_t1prof, h, sizeof h);
  }
#endif
  filtration_table_kernel<<<cnt, block, bytes, st>>>(p, c, t0, cap, g, vs.ball_cache, tb, W);
  count_launch();
}

// shared memory kernel 1t needs for a vicinity of n_max vertices (the host checks it against the 227 KB limit)
size_t filtration_table_smem(int N, int64_t n_max) {
  const int W = (N + 31) / 32;
  const int cap = (int)((n_max + 7) / 8 * 8);
  return (size_t)cap * 11 + (size_t)2 * W * 4 + ((size_t)N + 1) / 2 * 4 + 16 + sizeof(TableShared);
}

}  // namespace tlc
