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
  int32_t ninv;     // invalid (vertex, root) items of the pass
  int32_t nextra;   // further chunks of their long rows
  int32_t dinv;     // sum of their graph degrees
  int32_t nia;      // entries of the list of invalid-invalid adjacencies
  int32_t any;
  long long tprev;  // (-DT1_PROFILE: clock of thread 0 at the last phase tick)
};
#ifdef T1_PROFILE
__device__ unsigned long long g_t1prof[24];
#define TPROF(i) do { if (tid == 0) { const long long tnow_ = clock64(); atomicAdd(&g_t1prof[i], (unsigned long long)(tnow_ - sh.tprev)); sh.tprev = tnow_; } } while (0)
#else
#define TPROF(i) do { } while (0)
#endif

constexpr int UNKNOWN = 0, VALID = 1, INVALID = 2, UNREACH = 3;
constexpr int CLS_SHIFT = 14;          // per-(vertex, root) u16: class << 14 | parent local id (local ids are below 2^14)
constexpr int PAR_MASK = (1 << CLS_SHIFT) - 1;

// what the root passes of one target share
struct TableTarget {
  int n, lu, lv, u, v;
  int64_t vo;
  bool plain;
  const int32_t* vert;
  double *d1, *d2;
  int32_t *hint, *hint0;       // tree parent towards the last root (kernel 2v's "neighbour in an earlier block" hint), the first
  unsigned long long* dist;    // shared: per (vertex, root) distance, later the weight of its tree edge
  uint16_t* pcl;               // shared: per (vertex, root) class << 14 | parent local id
  const uint16_t* lid;         // shared: graph id -> local id (0xffff: not in S)
};

// The roots r0 .. r0 + NR - 1 of a target (0: u, 1: v) through phases 1 - 5, all of them in the same passes: the state of
// (vertex x, the rr-th root) is entry k = rr * n + x of dist / pcl, and every list item, list entry and walk carries k.
// NR = 2 gives every phase twice the independent work per thread and barrier (the phases are chains of dependent
// global round trips, about 4.5 vertices per thread and root on a median vicinity).
template <int NR>
__device__ __forceinline__ void root_passes(const TableTarget& T, int r0, const ChunkView& c, const GraphView& g,
                                            const SsspTables& tb, TableShared& sh) {
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  const int n = T.n, NN = NR * n, N = g.N;
  const int64_t vo = T.vo;
  const bool plain = T.plain;
  const int32_t* __restrict__ vert = T.vert;
  unsigned long long* dist = T.dist;
  uint16_t* pcl = T.pcl;
  const uint16_t* lid = T.lid;
  // the rr-th root of the pass: its state k, its table rows, its outputs
  auto R_of = [&](int rr) { return r0 + (NR == 2 ? rr : 0); };
  auto rootk = [&](int rr) { return (NR == 2 ? rr * n : 0) + (R_of(rr) == 0 ? T.lu : T.lv); };
  auto trow = [&](int rr) { return (size_t)(R_of(rr) == 0 ? T.u : T.v) * N; };
  auto out = [&](int rr) { return R_of(rr) == 0 ? T.d1 : T.d2; };
  auto hnt = [&](int rr) { return R_of(rr) == 0 ? T.hint0 : T.hint; };
  auto base_of = [&](int k) { return NR == 2 && k >= n ? n : 0; };  // k - base_of(k): the vertex's local id
  int32_t* inv0 = c.vs0 + vo;     // list of the invalid (vertex, root) items: 0 .. n - 1 ...
  int32_t* inv1 = c.vs2 + vo;     // ... n .. 2n - 1
  auto inv_at = [&](int i) -> int32_t& { return NR == 1 || i < n ? inv0[i] : inv1[i - n]; };
  int32_t* extra = c.vs1 + vo;    // further row chunks of the long invalid rows: k << 12 | chunk
  int32_t* bpos = reinterpret_cast<int32_t*>(c.v64b + vo);    // per k: smallest row position of a tree-parent candidate
  uint32_t* iap = reinterpret_cast<uint32_t*>(c.vord + vo);   // invalid-invalid adjacency: k << 16 | neighbour's k ...
  int32_t* iaq = c.vrank + vo;                                // ... and the row position of the entry; slots n .. 4n - 1:
  uint2* ia2 = reinterpret_cast<uint2*>(c.v64a + vo);
  uint2* ia3 = reinterpret_cast<uint2*>(c.v64c + vo);
  uint2* ia4 = reinterpret_cast<uint2*>(c.fval + vo);       // (the filtration values are written at the very end)

  if (tid == 0) { sh.ninv = 0; sh.nextra = 0; sh.dinv = 0; sh.nia = 0; }
  // ---- 1. classes: the branch of x stays in S <=> its table parent is in S and is valid itself ----
  // Four (vertex, root) states per thread with their loads in flight together: first the graph ids, then D and P of every
  // root, only then the local ids of the parents (each state alone would be two dependent global round trips)
  constexpr int VS = 4 / NR;
  for (int x0 = tid; x0 < n; x0 += VS * nt) {
    int32_t gx[VS];
#pragma unroll
    for (int s = 0; s < VS; s++) { const int x = x0 + s * nt; gx[s] = x < n ? vert[x] : -1; }
    double d[VS][NR];
    int32_t pp[VS][NR];
#pragma unroll
    for (int s = 0; s < VS; s++)
#pragma unroll
      for (int rr = 0; rr < NR; rr++) {
        d[s][rr] = gx[s] >= 0 ? tb.D[trow(rr) + gx[s]] : 0.0;
        pp[s][rr] = gx[s] >= 0 ? tb.P[trow(rr) + gx[s]] : -1;
      }
#pragma unroll
    for (int s = 0; s < VS; s++) {
      const int x = x0 + s * nt;
      if (x >= n) continue;
#pragma unroll
      for (int rr = 0; rr < NR; rr++) {
        const int k = rr * n + x;
        uint16_t e;
        if (k == rootk(rr)) e = (uint16_t)(VALID << CLS_SHIFT);
        else {
          const int32_t gp = pp[s][rr];
          const uint16_t pl = gp >= 0 ? lid[gp] : (uint16_t)0xffff;
          e = pl == 0xffff ? (uint16_t)(INVALID << CLS_SHIFT) : pl;  // (UNKNOWN << 14 | parent)
        }
        pcl[k] = e;
        dist[k] = (unsigned long long)__double_as_longlong(d[s][rr]);
      }
      if (r0 == 0) { T.hint[x] = -1; T.hint0[x] = -1; }
    }
  }
  __syncthreads();
  TPROF(1);
  for (int round = 0; round <= n; round++) {
    int ch = 0;
    for (int k = tid; k < NN; k += nt) {
      const uint16_t e = pcl[k];
      if ((e >> CLS_SHIFT) != UNKNOWN) continue;
      const int pc = pcl[base_of(k) + e] >> CLS_SHIFT;
      if (pc != UNKNOWN) pcl[k] = (uint16_t)(e | (pc << CLS_SHIFT));   // (a stale read only delays the state to the next round)
      ch = 1;
    }
    if (!__syncthreads_or(ch)) break;
  }
  TPROF(2);
  // ---- 2. the invalid states, their distances by pull relaxations over their own graph rows ----
  // Work items are row CHUNKS: item i < ninv is the first chunk of invalid state i, the further chunks of the long
  // rows (hubs) are listed once per state in extra[] -- a hub's row is then spread over many warps instead of stalling
  // one.  A chunk's best candidate goes into the state's distance with a shared-memory atomic min.
  for (int k0 = 0; k0 < NN; k0 += nt) {
    const int k = k0 + tid;
    const bool iv = k < NN && (pcl[k] >> CLS_SHIFT) == INVALID;
    const unsigned bal = __ballot_sync(0xffffffffu, iv);
    int base = 0;
    if (bal && lane == 0) base = atomicAdd(&sh.ninv, __popc(bal));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (iv) {
      const int32_t gx = vert[k - base_of(k)];
      inv_at(base + __popc(bal & lanemask_lt())) = k;
      dist[k] = INF_BITS; bpos[k] = 0x7fffffff;
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
    const int k = inv_at(i);
    const int32_t gx = vert[k - base_of(k)];
    const int cnt = (g.rowptr[gx + 1] - g.rowptr[gx] + chunk - 1) / chunk;
    if (cnt > 1) {
      const int at = atomicAdd(&sh.nextra, cnt - 1);
      for (int j = 1; j < cnt; j++) extra[at + j - 1] = (k << 12) | j;
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
  auto item_bounds = [&](int i, int& k, int& a, int& b, bool flagged_only) {
    const int raw = i < ninv ? inv_at(i) : extra[i - ninv];
    const int pk = i < ninv ? ((raw & 0xffff) << 12) : (raw & (ITEM_RESCAN - 1));
    k = pk >> 12;
    const int x = k - base_of(k);
    const int ra = c.astart[vo + x];
    a = ra + (pk & 4095) * chunk;
    b = min(ra + c.adeg[vo + x], a + chunk);
    if (flagged_only && !(raw & ITEM_RESCAN)) b = a;
  };
  // The FIRST round reads every invalid row once.  The valid neighbours' distances are final: their candidates never
  // need a second look.  The invalid neighbours go into a list of (state, neighbour's state, row position) entries -- the
  // graph among the invalid states, a few entries per state, every pair once (weights are symmetric, the later
  // rounds relax an entry both ways) -- and the following rounds run over that list only
  // (measured: 3 rounds, the second changes 2 - 5 % of the vertices, the third none).  A list that outgrows its 4n
  // slots (small vicinities that are mostly invalid) sends the chunks that did not fit back to rounds over the rows.
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
      // the group's next eight items, their bounds fetched lane-parallel (state -> row start, degree: a dependent chain)
      int mk = 0, ma = 0, mb = 0;
      { const int itl = (kb + l8) * ngrp + grp; if (itl < nitems) item_bounds(itl, mk, ma, mb, !first); }
      for (int j = 0; j < 8; j++) {
        const int k = __shfl_sync(gm, mk, j, 8), a = __shfl_sync(gm, ma, j, 8), b = __shfl_sync(gm, mb, j, 8);
        const int rb = base_of(k);
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
            const int ky = rb + (int)ly;
            if (first) {
              const bool need = ly != 0xffff && ky > k && (pcl[ky] >> CLS_SHIFT) == INVALID;  // (a pair is listed once, by its smaller end)
              const unsigned m = __ballot_sync(0xffffffffu, need);
              if (need) {
                const int slot = cntw + __popc(m & lanemask_lt());
                if (slot < capw) ia_put(wid * capw + slot, ((uint32_t)k << 16) | (uint32_t)ky, e0 + 8 * q);
              }
              cntw += __popc(m);
            }
            if (ly == 0xffff) continue;
            const double w = __hiloint2double((int)rc[q].w, (int)rc[q].z);
            const unsigned long long dyb = dist[ky];
            if (!first && (pcl[ky] >> CLS_SHIFT) == INVALID) {  // a reread chunk also pushes: the pairs it would have listed go both ways
              const unsigned long long dxb = dist[k];
              if (dxb != INF_BITS) {
                const unsigned long long c2 = (unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dxb), w));
                if (c2 < dyb && c2 < atomicMin(&dist[ky], c2)) ch = 1;
              }
            }
            if (dyb == INF_BITS) continue;
            const unsigned long long cand = (unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dyb), w));
            best = cand < best ? cand : best;
          }
        }
#pragma unroll
        for (int o = 4; o; o >>= 1) { const unsigned long long u2 = __shfl_xor_sync(gm, best, o); best = u2 < best ? u2 : best; }
        if (l8 == 0 && b > a && best < dist[k] && best < atomicMin(&dist[k], best)) ch = 1;
        if (first && cntw > capw && l8 == 0 && b > a) {  // the warp's region is full: this chunk stays on the row path
          const int itj = (kb + j) * ngrp + grp;
          if (itj < ninv) inv_at(itj) |= ITEM_RESCAN; else extra[itj - ninv] |= ITEM_RESCAN;
        }
      }
    }
    return ch;
  };
  relax_rows(true);
  const bool full = __syncthreads_or(cntw > capw ? 1 : 0) != 0;  // some chunks are flagged for rereading
  TPROF(5);
  const int nlist = min(cntw, capw);
  // the first 128 entries of the warp's region stay in registers over the rounds (state pair + edge weight): a round is
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
  if (tid == 0) { atomicAdd(&g_t1prof[11], (unsigned long long)(full ? 1 : 0)); atomicAdd(&g_t1prof[12], (unsigned long long)NR); atomicAdd(&g_t1prof[13], (unsigned long long)nitems); atomicAdd(&g_t1prof[14], (unsigned long long)sh.dinv); }
#endif
  // ---- 3. tree rule for the invalid states: smallest local id y (= smallest row position) with fl(d[y] + w) == d[x] ----
  for (int kb = 0; kb * ngrp < nitems; kb += 8) {
    int mk = 0, ma = 0, mb = 0;
    { const int itl = (kb + l8) * ngrp + grp; if (itl < nitems) item_bounds(itl, mk, ma, mb, false); }
    for (int j = 0; j < 8; j++) {
      const int k = __shfl_sync(gm, mk, j, 8), a = __shfl_sync(gm, ma, j, 8);
      int b = __shfl_sync(gm, mb, j, 8);
      const int rb = base_of(k);
      const unsigned long long dxb = b > a ? dist[k] : INF_BITS;
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
          const unsigned long long dyb = dist[rb + ly];
          if (dyb != INF_BITS && (unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dyb), __hiloint2double((int)rc[q].w, (int)rc[q].z))) == dxb)
            hit = e0 + l8 + 8 * q;
        }
        if (__ballot_sync(gm, hit != 0x7fffffff)) break;   // (the group's own vote: groups leave at different times)
      }
#pragma unroll
      for (int o = 4; o; o >>= 1) hit = min(hit, __shfl_xor_sync(gm, hit, o));
      if (l8 == 0 && hit != 0x7fffffff) atomicMin(&bpos[k], hit);
    }
  }
  __syncthreads();
  TPROF(7);
  // ---- 4. parents and outputs (phase "parents"): from here on the distances are not needed any more and every
  // state's 8-byte slot holds the weight of its tree edge instead, so that the walks below stay in shared memory.
  // A valid state's {Q, W} (one 16-byte load) gives that weight and its output, the table's path sum; four valid
  // states per thread with their loads in flight together, a vertex's graph id read once for all roots.  An
  // invalid state takes its parent from the tree rule's row position, or is unreachable (nx.NetworkXNoPath:
  // disconnected vicinity, status 3 later).  The root and the unreachable vertices keep the hint -1.
  for (int x0 = tid; x0 < n; x0 += VS * nt) {
    int32_t gx[VS];
    bool val[VS][NR];
#pragma unroll
    for (int s = 0; s < VS; s++) {
      const int x = x0 + s * nt;
      bool any = false;
#pragma unroll
      for (int rr = 0; rr < NR; rr++) {
        const int k = rr * n + x;
        val[s][rr] = x < n && k != rootk(rr) && (pcl[k] >> CLS_SHIFT) == VALID;
        any |= val[s][rr];
      }
      gx[s] = any ? vert[x] : -1;
    }
    double2 e[VS][NR];
#pragma unroll
    for (int s = 0; s < VS; s++)
#pragma unroll
      for (int rr = 0; rr < NR; rr++) e[s][rr] = val[s][rr] ? tb.QW[trow(rr) + gx[s]] : make_double2(0.0, 0.0);
#pragma unroll
    for (int s = 0; s < VS; s++) {
      const int x = x0 + s * nt;
      if (x >= n) continue;
#pragma unroll
      for (int rr = 0; rr < NR; rr++) {
        const int k = rr * n + x;
        unsigned long long wb = 0;
        if (k == rootk(rr)) out(rr)[x] = 0.0;
        else if (val[s][rr]) {
          wb = (unsigned long long)__double_as_longlong(e[s][rr].y);
          out(rr)[x] = e[s][rr].x;
          hnt(rr)[x] = (int32_t)(pcl[k] & PAR_MASK);
        } else {
          const int pos = bpos[k];
          if (dist[k] != INF_BITS && pos != 0x7fffffff) {
            const uint4 rc = __ldg(g.rec + pos);
            const uint16_t pl = lid[rc.x];
            pcl[k] = (uint16_t)((INVALID << CLS_SHIFT) | pl);
            hnt(rr)[x] = (int32_t)pl;
            wb = ((unsigned long long)rc.w << 32) | rc.z;
          } else { pcl[k] = (uint16_t)(UNREACH << CLS_SHIFT); out(rr)[x] = NO_PATH_DIST; }
        }
        dist[k] = wb;
      }
    }
  }
  __syncthreads();
  TPROF(8);
  // ---- 5. path sums of the invalid states (phase "path_sums"): a walk in python order   :30,35 ----
  for (int i = tid; i < ninv; i += nt) {
    const int k = inv_at(i) & 0xffff;  // (without the rescan flag)
    if ((pcl[k] >> CLS_SHIFT) == UNREACH) continue;
    const int rb = base_of(k), rr = rb ? 1 : 0, root = rootk(rr);
    PySum ps{0.0, 0.0, 0};
    int y = k, guard = 0;
    while (y != root && guard++ <= n) {
      const int py = rb + (pcl[y] & PAR_MASK);
      pysum_add(ps, __longlong_as_double((long long)dist[y]), plain);
      y = py;
    }
    out(rr)[k - rb] = pysum_get(ps, plain);
  }
  __syncthreads();
  TPROF(9);
}

// One CTA per target of the sub-range [t0, t0 + gridDim.x) whose vicinity size (n_of, the counting pass's) is at most
// two_max (TWO) or above it (!TWO); the other CTAs leave at once.  TWO: both roots' states in the same passes (a target
// with u == v runs them too and keeps the one-root outputs); !TWO: one root at a time, also in NODE mode.  The two are
// separate kernels so that each keeps its 64 registers without spilling.
template <bool TWO>
__global__ void __launch_bounds__(1024) filtration_table_kernel(Params p, ChunkView c, int t0, int slots,
                                                                const int32_t* __restrict__ n_of, int two_max, GraphView g,
                                                                const uint32_t* __restrict__ ball_cache, SsspTables tb, int W) {
  extern __shared__ __align__(16) unsigned long long dynt[];
  __shared__ TableShared sh;
  const int t = t0 + blockIdx.x;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  const bool node_mode = p.mode == TLC_MODE_NODE;
  const int64_t vo = c.voff[t];
  const int N = g.N;
  // dynamic shared memory: dist u64[slots] | class << 14 | parent local id u16[slots] | bitmap + ranks u32[2W] | local ids u16[N]
  unsigned long long* dist = dynt;
  uint16_t* pcl = reinterpret_cast<uint16_t*>(dynt + slots);
  uint32_t* bm = reinterpret_cast<uint32_t*>(reinterpret_cast<unsigned char*>(dynt) + (size_t)slots * 10);
  uint16_t* lid = reinterpret_cast<uint16_t*>(bm + 2 * W);

#ifdef T1_PROFILE
  if (tid == 0) sh.tprev = clock64();
#endif
  // ---- 0. the vicinity (as kernel 1b's graph-row prologue): nodes = set(nodes_u) & set(nodes_v), local ids = ranks   :311-316
  const int64_t ti = c.tidx[t];
  if ((n_of[ti] <= two_max) != TWO) return;
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

  double* d1 = c.d1 + vo;
  double* d2 = c.d2 + vo;
  double* fval = c.fval + vo;
  const bool roots_in = lu >= 0 && lv >= 0;
  const bool two = roots_in && !node_mode && lu != lv;

  if (!roots_in) {
    // nx.NodeNotFound for every vertex
    for (int x = tid; x < n; x += nt) { d1[x] = NO_PATH_DIST; d2[x] = NO_PATH_DIST; c.neg[vo + x] = -1; c.vcls[vo + x] = -1; }
  } else {
    const TableTarget T{n, lu, lv, u, v, vo, (p.flags & TLC_F_SUM_PLAIN) != 0, c.vert + vo, d1, d2, c.neg + vo, c.vcls + vo,
                        dist, pcl, lid};
    if constexpr (TWO) {
      root_passes<2>(T, 0, c, g, tb, sh);
      if (two) {
        if (tid == 0 && c.fb_counter) atomicAdd(&c.fb_counter[4], 1);
#ifdef T1_PROFILE
        if (tid == 0) atomicAdd(&g_t1prof[18], 1ull);
#endif
      } else {
        for (int x = tid; x < n; x += nt) T.hint[x] = -1;  // u == v: no second root
      }
    } else {
      for (int r = 0; r < (two ? 2 : 1); r++) root_passes<1>(T, r, c, g, tb, sh);
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

// dynamic shared memory of kernel 1t with room for `slots` (vertex, root) states: 10 B each (distance, class + parent),
// the bitmap with its ranks and the local-id table
static size_t table_smem_bytes(int N, int slots) {
  const int W = (N + 31) / 32;
  return (size_t)slots * 10 + (size_t)2 * W * 4 + ((size_t)N + 1) / 2 * 4 + 16;
}

// the largest vicinity whose two root states fit kernel 1t's shared memory (-1: every target one root at a time -- NODE
// mode, which has one root, or TLC_TABLE_ONE_ROOT=1 for tests and A/B runs in one build)
static int64_t filtration_table_two_max(int N, const Params& p) {
  const char* env = getenv("TLC_TABLE_ONE_ROOT");
  if (p.mode == TLC_MODE_NODE || (env && atoi(env) != 0)) return -1;
  return (int64_t)((226 * 1024 - sizeof(TableShared) - table_smem_bytes(N, 0)) / 20 / 8 * 8);
}

template <bool TWO>
static void launch_table_kernel(const GraphView& g, const Params& p, const ChunkView& c, const VicinityScratch& vs,
                                const SsspTables& tb, const int32_t* n_of, int64_t two_max, int t0, int cnt, int block,
                                int64_t states, int W, cudaStream_t st) {
  const int slots = (int)((states + 7) / 8 * 8);
  const size_t bytes = table_smem_bytes(g.N, slots);
  if (block < 128) block = 128;
  if (bytes + sizeof(TableShared) > 110 * 1024 && block >= 512) block = 1024;  // one resident CTA per SM: give it 32 warps
  if (const char* env = getenv("TLC_TABLE_BLOCK")) block = atoi(env);  // (tuning experiments)
  cudaFuncSetAttribute((const void*)filtration_table_kernel<TWO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  cudaFuncSetAttribute((const void*)filtration_table_kernel<TWO>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  filtration_table_kernel<TWO><<<cnt, block, bytes, st>>>(p, c, t0, slots, n_of, (int)two_max, g, vs.ball_cache, tb, W);
  count_launch();
}

// the sub-range's targets with n <= two_max by the two-root kernel, the others by the one-root kernel (each launch only
// when the sub-range has such targets: n_min, n_max)
void launch_filtration_table(const GraphView& g, const Params& p, const ChunkView& c, const VicinityScratch& vs,
                             const SsspTables& tb, const int32_t* n_of, int t0, int cnt, int block, int64_t n_min,
                             int64_t n_max, cudaStream_t st) {
  const int W = (g.N + 31) / 32;
  const int64_t two_max = filtration_table_two_max(g.N, p);
#ifdef T1_PROFILE
  if (getenv("T1_PROFILE_DUMP")) {  // ticks of thread 0 per phase, summed over the CTAs since the last dump (per target:
                                    // a target's two one-root passes add to the same phases)
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
      fprintf(stderr, "[1t profile] later rounds per root %.2f; ticks of the later rounds spent in roots with flagged chunks: %.1f Mticks; targets with both roots in the same passes %llu\n",
              (double)h[17] / (double)(h[12] ? h[12] : 1), (double)h[16] / 1e6, h[18]);
    }
    memset(h, 0, sizeof h);
    cudaMemcpyToSymbol(g_t1prof, h, sizeof h);
  }
#endif
  if (n_min <= two_max) launch_table_kernel<true>(g, p, c, vs, tb, n_of, two_max, t0, cnt, block, 2 * std::min(n_max, two_max), W, st);
  if (n_max > two_max) launch_table_kernel<false>(g, p, c, vs, tb, n_of, two_max, t0, cnt, block, n_max, W, st);
}


// shared memory kernel 1t needs for a vicinity of n_max vertices, one root at a time (the host checks it against the
// 227 KB limit)
size_t filtration_table_smem(int N, int64_t n_max) {
  return table_smem_bytes(N, (int)((n_max + 7) / 8 * 8)) + sizeof(TableShared);
}

}  // namespace tlc
