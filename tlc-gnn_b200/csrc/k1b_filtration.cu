// k1b_filtration.cu -- kernel 1b: the node filtration of every vicinity.
//
// Replaces filtration.build_fv(weight_graph=True, norm) (riccidist2dgm.py:20-61) and the KD copy
// (Knowledge_Distillation/data_utils_NC.py:34-55).  The reference runs one nx.dijkstra_path per
// (vertex, root) and sums kappa+1 along the returned path with python's sum(); here each root gets ONE
// shortest-path computation inside the vicinity, one CTA per vicinity, distances in shared memory:
//   1. distances: Dijkstra in parallel phases.  Each phase settles EVERY tentative vertex x with
//      d[x] <= fl(d_min + minw[x]), d_min the smallest tentative distance and minw[x] the smallest weight
//      incident to x (Crauser et al.'s IN criterion: whatever still reaches x comes from a vertex at
//      distance >= d_min over an edge >= minw[x]); fl(+) is monotone, so the test is exact in IEEE
//      arithmetic.  The settled vertices' rows are relaxed with a 64-bit atomicMin on the bit pattern of
//      the (non-negative) float64 distance in shared memory; every row is read once per root.  A warp
//      takes 32 settled vertices at a time and walks their concatenated rows (row found by a shuffle
//      bisection of the degree prefix), so all loads of a batch are independent;
//   2. shortest-path tree, in the same row read: parent[x] = smallest local id y with
//      fl(d[y] + w(y,x)) == d[x] (rows are ascending: the smallest matching row position) -- the same rule
//      as the oracle's fast mode.  All candidates y are final when x settles (d[y] <= d[x] - minw[x] <= d_min);
//   3. the path sum is re-accumulated from x towards the root in python-sum order (Neumaier
//      compensated as CPython >= 3.12 does, or plain with TLC_F_SUM_PLAIN)  -- SURVEY.md F5;
//   4. min / max / sum descriptors, block max-reduce, true division by the normaliser (:50-56).
// Precondition (as for networkx's Dijkstra): kappa + 1 > 0.
//
// Two instantiations.  <false>: rows come from the induced adjacency kernel 1's fill pass wrote to HBM.
// <true> (GRAPH-ROW route, dense vicinities): nothing is materialised -- the kernel builds the vicinity itself
// (AND of the two cached ball bitmaps, word-prefix ranks, vertex list, local roots, status: what the fill pass does
// except the adjacency) and walks the graph's own CSR rows, which stay L2-resident (<= 8 MB for every shape);
// an entry is kept iff its graph id is in the bitmap, its local id is the bitmap rank.  The settling margin is
// the smallest weight of the vertex's GRAPH row (<= the smallest induced weight: the criterion stays valid).
#include <cuda_fp16.h>

#include <cstdlib>

#include "tlc_common.cuh"

namespace tlc {
namespace {

#ifndef FILT_QCAP
#define FILT_QCAP 1024
#endif
#ifndef FILT_RU
#define FILT_RU 4
#endif
// Two variants of the relaxation loop that were built and MEASURED on B200 (round 2, Computers-shaped 2-hop, 4096 targets
// per step, kernel time of this kernel; DESIGN.md section 8) -- both issue fewer instructions per row entry and both are
// slower than the plain form, so they are off by default:
//   FILT_REC   = 1: one LDG.128 of an interleaved {id, 0, kappa + 1} row record instead of LDG.32 + LDG.64 + a float64 add
//                   (14.70 ms vs 14.59 ms: a third more bytes through the L2 for one instruction less)
//   FILT_SPLIT = 1: decide by d[y] > d[x] whether an entry is a relaxation or a parent candidate, one float64 add per entry
//                   instead of two (15.18 ms: the add can no longer issue before d[y] arrives -- the loop is latency-bound)
#ifndef FILT_REC
#define FILT_REC 0
#endif
#ifndef FILT_SPLIT
#define FILT_SPLIT 0
#endif
constexpr int QCAP = FILT_QCAP;  // vertices settled per phase at most
struct FiltShared {
  double redd[32];
  // the phase's settled vertices: id, first entry in the concatenated rows (exclusive degree prefix),
  // row start in the adjacency, smallest adjacency position of a tree-parent candidate
  int32_t qx[QCAP], qpre[QCAP + 1], qrs[QCAP], qbest[QCAP];
  int32_t wsum[33];
  // double-buffered by phase parity: vertices settled in the phase / smallest tentative distance for the next one
  int qn[2];
  unsigned long long nmin[2];
};

struct DirectArgs {
  GraphView g;
  const uint32_t* ball_cache;  // [N][W] closed k-hop balls (kernel 1's ball cache)
  const float* gminw;          // [N] smallest kappa + 1 of the node's graph row, rounded down
  int W;
  int lid_table;               // 1: shared memory also holds a graph id -> local id table (uint16[N], 0xffff = absent)
};

template <bool DIRECT, bool SMEM>
__global__ void __launch_bounds__(1024) filtration_kernel(Params p, ChunkView c, int t0, int cap, int bpv, DirectArgs da) {
  extern __shared__ unsigned long long dyn64[];
  __shared__ FiltShared sh;
  const int t = t0 + blockIdx.x;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  const bool node_mode = p.mode == TLC_MODE_NODE;
  const int64_t vo = c.voff[t];
  // graph-row route: vicinity bitmap [0, W) and word-prefix ranks [W, 2W), behind the per-vertex arrays
  uint32_t* bm = reinterpret_cast<uint32_t*>(reinterpret_cast<unsigned char*>(dyn64) + (size_t)cap * bpv);
  const int W = da.W;
  int n, lu, lv;
  if (DIRECT) {
    // ---- 0. the vicinity: nodes = set(nodes_u) & set(nodes_v), canonical local ids = ranks   riccidist2dgm.py:311-316
    const int64_t ti = c.tidx[t];
    const int32_t u = c.tgt[2 * ti], v = c.tgt[2 * ti + 1];
    const GraphView& g = da.g;
    if (unknown_target(g, u, v, node_mode)) {
      if (tid == 0) { c.tn[t] = 0; c.tnp[t] = 0; c.tnpos[t] = 0; c.tnneg[t] = 0; c.tlu[t] = -1; c.tlv[t] = -1;
                      c.tstatus[t] = TLC_ST_UNKNOWN_NODE; }
      return;
    }
    n = graph_row_bitmap(c, t, da.ball_cache, W, u, v, node_mode, bm, sh.wsum);
    for (int w = wid; w < W; w += nw) {  // a warp per bitmap word: vertex list, graph rows, settling margins
      const uint32_t bits = bm[w];
      if (!((bits >> lane) & 1u)) continue;
      const int lx = (int)bm[W + w] + __popc(bits & lanemask_lt());
      const int32_t x = w * 32 + lane;
      const int32_t ra = g.rowptr[x];
      c.vert[vo + lx] = x;
      c.astart[vo + lx] = ra;
      c.adeg[vo + lx] = g.rowptr[x + 1] - ra;
      c.aminw[vo + lx] = da.gminw[x];
    }
    if (da.lid_table) {  // graph id -> local id in ONE shared-memory read per row entry (instead of bitmap word + prefix + popcount)
      uint32_t* l32 = bm + 2 * W;
      for (int i = tid; i < (g.N + 1) / 2; i += nt) l32[i] = 0xffffffffu;
      __syncthreads();
      uint16_t* l16 = reinterpret_cast<uint16_t*>(l32);
      for (int w = wid; w < W; w += nw) {
        const uint32_t bits = bm[w];
        if ((bits >> lane) & 1u) l16[w * 32 + lane] = (uint16_t)((int)bm[W + w] + __popc(bits & lanemask_lt()));
      }
    }
    lu = bitmap_rank(bm, W, u);
    lv = node_mode ? lu : bitmap_rank(bm, W, v);
    uint8_t st0 = (lu >= 0 && lv >= 0) ? TLC_ST_OK : TLC_ST_TRIVIAL;
    // node mode: `return None, None` when the ball has no edge (data_utils_NC.py:103-104) <=> it is the lone centre
    if (n == 0 || (node_mode && n == 1)) st0 = TLC_ST_EMPTY;  // :318
    if (tid == 0) {
      c.tn[t] = n; c.tlu[t] = lu; c.tlv[t] = lv; c.tstatus[t] = st0;
      c.tnp[t] = 0; c.tnpos[t] = 0; c.tnneg[t] = 0; c.tncls[t] = 0;
    }
    __syncthreads();
    if (n == 0 || st0 > TLC_ST_TRIVIAL) return;
  } else {
    n = c.tn[t];
    if (n == 0) return;
    if (c.tstatus[t] > TLC_ST_TRIVIAL) return;
    lu = c.tlu[t]; lv = c.tlv[t];
  }
  const int64_t ao = DIRECT ? 0 : c.aoff[t];
  const int32_t* __restrict__ astart = c.astart + vo;
  const int32_t* __restrict__ adeg = c.adeg + vo;
  // rows: induced adjacency segment of the target, or (graph-row route) the graph's CSR itself
  const uint32_t* __restrict__ anb = DIRECT ? reinterpret_cast<const uint32_t*>(da.g.col) : c.anb + ao;
  const double* __restrict__ aw = DIRECT ? da.g.kappa : c.aw + ao;
#if FILT_REC
  const uint4* __restrict__ grec = da.g.rec;  // graph-row route: interleaved {id, 0, kappa + 1} row records
#endif
  double* d1 = c.d1 + vo;
  double* d2 = c.d2 + vo;
  double* fval = c.fval + vo;
  const bool roots_in = lu >= 0 && lv >= 0;
  const bool plain = (p.flags & TLC_F_SUM_PLAIN) != 0;
  const bool two = roots_in && !node_mode && lu != lv;

  // graph-row route, when the counting pass skipped the induced edges: every member entry read while relaxing for the
  // first root is counted (each reached vertex's row is read exactly once); rows the relaxation never reads (vertices
  // the first root does not reach, or no root in the vicinity at all) are counted separately below
  const bool count_m = DIRECT && c.count_m != 0;
  const bool use_lid = DIRECT && da.lid_table != 0;
  const uint16_t* slid = reinterpret_cast<const uint16_t*>(bm + 2 * W);
  int mcnt = 0;
  if (!roots_in) {
    // nx.NodeNotFound for every vertex
    for (int x = tid; x < n; x += nt) { d1[x] = NO_PATH_DIST; d2[x] = NO_PATH_DIST; c.neg[vo + x] = -1; c.vcls[vo + x] = -1; }
    if (count_m) {
      for (int x = wid; x < n; x += nw) {
        const int a = astart[x], dg = adeg[x];
        for (int j = lane; j < dg; j += 32) mcnt += bitmap_rank(bm, W, (int)anb[a + j]) >= 0 ? 1 : 0;
      }
    }
  } else {
    // SMEM: the launch sized shared memory for the sub-range's largest vicinity (n <= cap); otherwise the per-vertex
    // state lives in the arena.  A compile-time switch, so that the shared-memory accesses are LDS / ATOMS, not generic
    unsigned long long* dist = SMEM ? dyn64 : c.v64a + vo;
    // shared-memory state per vertex: dist (8 B), state (1 B) and -- unless the launch went LEAN to fit a very large
    // vicinity (bpv == 9) -- the settling margin as a half rounded down (2 B); lean launches read the float margin
    // from the arena instead (coalesced, once per tentative vertex and phase)
    const bool margins_in_smem = SMEM && bpv == 11;
    __half* smw = reinterpret_cast<__half*>(dyn64 + cap);
    uint8_t* state = SMEM ? (margins_in_smem ? reinterpret_cast<uint8_t*>(smw + cap) : reinterpret_cast<uint8_t*>(dyn64 + cap))
                          : reinterpret_cast<uint8_t*>(c.vs1 + vo);
    int32_t* tpar = c.vs2 + vo;                            // shortest-path tree: parent and weight of the parent edge
    // a true induced neighbour of every vertex that lies nearer to a root (its tree parent), or -1: kernel 2v tries it
    // first when it looks for "a neighbour in an earlier block" (c.neg is free until the edge-sorted kernels run)
    int32_t* hint = c.neg + vo;
    int32_t* hint0 = c.vcls + vo;  // ... and the parent towards the FIRST root (c.vcls: kernel 2's value classes come later)
    double* tpw = reinterpret_cast<double*>(c.v64b + vo);
    const float* __restrict__ aminw = c.aminw + vo;
    constexpr uint8_t FAR = 0, TENT = 1, DONE = 2;
    for (int r = 0; r < (two ? 2 : 1); r++) {
      const int root = r == 0 ? lu : lv;
      const int cnt_this_root = (count_m && r == 0) ? 1 : 0;
      double* out = r == 0 ? d1 : d2;
      for (int x = tid; x < n; x += nt) {
        dist[x] = INF_BITS; state[x] = FAR; tpar[x] = root; tpw[x] = 0.0;
        if (r == 0) { hint[x] = -1; hint0[x] = -1; }
        if (margins_in_smem && r == 0) smw[x] = __float2half_rd(fminf(aminw[x], 60000.f));  // rounded DOWN: the criterion stays valid
      }
      if (tid == 0) { sh.nmin[0] = 0ull; sh.nmin[1] = INF_BITS; sh.qn[0] = 0; sh.qn[1] = 0; }
      __syncthreads();
      if (tid == 0) { dist[root] = 0ull; state[root] = TENT; }
      __syncthreads();
      for (int phase = 0; phase < 2 * n + 2; phase++) {  // every phase settles at least one vertex
        const int cur = phase & 1;
        // smallest tentative distance: gathered by the previous phase (survivors of its settle scan, and every
        // value its relaxation wrote)
        const unsigned long long dminb = sh.nmin[cur];
        if (dminb == INF_BITS) break;  // nothing tentative left (the rest is unreachable)
        const double dmin = __longlong_as_double((long long)dminb);
        // ---- settle: d[x] <= fl(dmin + minw[x]); at most QCAP per phase (the others stay tentative) ----
        unsigned long long lmin = INF_BITS;
        for (int x0 = 0; x0 < n; x0 += nt) {
          const int x = x0 + tid;
          bool take = false;
          unsigned long long d = INF_BITS;
          if (x < n && state[x] == TENT) {
            d = dist[x];
            const double mw = margins_in_smem ? (double)__half2float(smw[x]) : (double)aminw[x];
            take = __longlong_as_double((long long)d) <= __dadd_rn(dmin, mw);
          }
          const unsigned bal = __ballot_sync(0xffffffffu, take);
          if (bal) {
            int base = 0;
            if (lane == 0) base = atomicAdd(&sh.qn[cur], __popc(bal));
            base = __shfl_sync(0xffffffffu, base, 0);
            const int pos = base + __popc(bal & lanemask_lt());
            if (take && pos < QCAP) {
              state[x] = DONE;
              sh.qx[pos] = x;
              sh.qpre[pos] = adeg[x];
              sh.qrs[pos] = astart[x];
              sh.qbest[pos] = 0x7fffffff;
              d = INF_BITS;
            }
          }
          lmin = d < lmin ? d : lmin;  // still tentative after this phase
        }
        lmin = warp_min_u64(lmin);
        if (lane == 0 && lmin != INF_BITS) atomicMin(&sh.nmin[cur ^ 1], lmin);
        __syncthreads();
        const int qn = min(sh.qn[cur], QCAP);
        if (tid == 0) { sh.nmin[cur] = INF_BITS; sh.qn[cur ^ 1] = 0; }  // (read by everyone before the barrier above)
        const int total = block_scan_shfl(sh.qpre, qn, sh.wsum);  // qpre[i] = first entry of row i in the phase's concatenation
        if (tid == 0) sh.qpre[qn] = total;
        __syncthreads();
        unsigned long long umin = INF_BITS;  // smallest distance this thread writes
        // ---- relax the settled rows, every warp an equal share of the concatenated entries (coalesced);
        //      the same read picks the tree parent of each settled vertex ----
        {
          const int span = ((total + nw - 1) / nw + 31) & ~31;
          const int e1 = min((wid + 1) * span, total);
          int e = wid * span + lane;
          if (e < e1) {
            int lo = 0, hi = qn;  // row i: largest i with qpre[i] <= e
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (sh.qpre[mid] <= e) lo = mid; else hi = mid; }
            int i = lo, nxt = sh.qpre[i + 1];
            while (e >= nxt) { i++; nxt = sh.qpre[i + 1]; }  // (rows of degree 0)
            int off = sh.qrs[i] - sh.qpre[i];
            unsigned long long dxb = dist[sh.qx[i]];
            // RU entries per lane and step: the row bookkeeping runs ahead in shared memory, then all loads of
            // the step are issued before the first use
            constexpr int RU = FILT_RU;
            for (; e < e1; e += 32 * RU) {
              int ai[RU], ri[RU];
              unsigned long long dx[RU];
#pragma unroll
              for (int k = 0; k < RU; k++) {
                const int ek = e + 32 * k;
                if (ek < e1) {
                  if (ek >= nxt) {
                    do { i++; nxt = sh.qpre[i + 1]; } while (ek >= nxt);
                    off = sh.qrs[i] - sh.qpre[i];
                    dxb = dist[sh.qx[i]];
                  }
                  ai[k] = off + ek; ri[k] = i; dx[k] = dxb;
                } else ai[k] = -1;
              }
              int yy[RU];
              double ww[RU];
#pragma unroll
              for (int k = 0; k < RU; k++) if (ai[k] >= 0) {
#if FILT_REC
                if (DIRECT) {  // {id, 0, kappa + 1}: ONE 128-bit load per row entry, the weight ready-made   riccidist2dgm.py:225
                  const uint4 r = __ldg(grec + ai[k]);
                  yy[k] = (int)r.x; ww[k] = __hiloint2double((int)r.w, (int)r.z);
                } else
#endif
                { yy[k] = (int)anb[ai[k]]; ww[k] = aw[ai[k]]; }
              }
#pragma unroll
              for (int k = 0; k < RU; k++) {
                if (ai[k] < 0) continue;
                int y = yy[k];
                if (DIRECT) {
                  if (use_lid) { const int l = (int)slid[y]; y = l == 0xffff ? -1 : l; }
                  else y = bitmap_rank(bm, W, y);
                  if (y < 0) continue;  // the neighbour is outside the vicinity
                  mcnt += cnt_this_root;
                }
#if FILT_REC
                const double w = ww[k];
#else
                const double w = DIRECT ? __dadd_rn(ww[k], 1.0) : ww[k];  // weight = kappa + 1   riccidist2dgm.py:225
#endif
                const unsigned long long dyb = dist[y];
#if FILT_SPLIT
                if (dyb > dx[k]) {
                  // y lies farther than x: relax.  (fl(d[y] + w) == d[x] is impossible here, w > 0)
                  const unsigned long long tb = (unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dx[k]), w));
                  if (tb < dyb) {
                    atomicMin(&dist[y], tb);
                    state[y] = TENT;  // (y is FAR or TENT: a settled vertex's distance is final and cannot be improved)
                    umin = tb < umin ? tb : umin;
                  }
                } else if ((unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dyb), w)) == dx[k]) {
                  // d[y] <= d[x]: fl(d[x] + w) >= d[x] >= d[y], nothing to relax; y is a parent of the row's vertex iff
                  // fl(d[y] + w) == d[x] (d[y] is final whenever this can hold)
                  atomicMin(&sh.qbest[ri[k]], ai[k]);
                }
#else
                const unsigned long long tb = (unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dx[k]), w));
                if (tb < dyb) {
                  atomicMin(&dist[y], tb);
                  state[y] = TENT;  // (y is FAR or TENT: a settled vertex's distance is final and cannot be improved)
                  umin = tb < umin ? tb : umin;
                } else if ((unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dyb), w)) == dx[k]) {
                  // (an unreached y carries +inf: inf + w never equals the finite d[x])
                  // y a parent of the row's vertex (d[y] is final whenever this can hold; it cannot when d[x] + w < d[y])
                  atomicMin(&sh.qbest[ri[k]], ai[k]);
                }
#endif
              }
            }
          }
        }
        umin = warp_min_u64(umin);
        if (lane == 0 && umin != INF_BITS) atomicMin(&sh.nmin[cur ^ 1], umin);
        __syncthreads();
        for (int i = tid; i < qn; i += nt) {
          const int x = sh.qx[i], a = sh.qbest[i];
          if (x != root && a != 0x7fffffff) {
            tpar[x] = DIRECT ? bitmap_rank(bm, W, (int)anb[a]) : (int)anb[a];
            (r == 0 ? hint0 : hint)[x] = tpar[x];
            tpw[x] = DIRECT ? __dadd_rn(aw[a], 1.0) : aw[a];  // (== the record's weight: the same IEEE add, done on the host)
          }
        }
        __syncthreads();  // the next phase overwrites the queue
      }
      __syncthreads();
      if (cnt_this_root) {  // rows of the vertices this root never reached (disconnected vicinity)
        for (int x = wid; x < n; x += nw) {
          if (state[x] == DONE) continue;
          const int a = astart[x], dg = adeg[x];
          for (int j = lane; j < dg; j += 32) mcnt += bitmap_rank(bm, W, (int)anb[a + j]) >= 0 ? 1 : 0;
        }
      }
      // ---- 3. python-order path sums ----
      for (int x = tid; x < n; x += nt) {
        double res;
        if (x == root) res = 0.0;
        else if (state[x] != DONE) res = NO_PATH_DIST;  // nx.NetworkXNoPath (disconnected vicinity; status 3 later)
        else {
          PySum ps{0.0, 0.0, 0};
          int y = x, guard = 0;
          while (y != root && guard++ <= n) {
            pysum_add(ps, tpw[y], plain);  // ricci_curv[(path[y], path[y+1])] + 1   :30
            y = tpar[y];
          }
          res = pysum_get(ps, plain);
        }
        out[x] = res;
      }
      __syncthreads();
    }
    if (!two) for (int x = tid; x < n; x += nt) d2[x] = d1[x];
    __syncthreads();
    if (tid == 0) zero_roots(d1, d2, lu, lv);
  }
  __syncthreads();

  if (count_m) {
    const int tot = block_reduce_sum(mcnt, sh.wsum);
    if (tid == 0) c.tm[t] = tot / 2;  // every induced edge was seen from both ends
  }
  // 4. descriptors + normalisation   riccidist2dgm.py:47-56 ; data_utils_NC.py:52-54
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
}

}  // namespace

// The PDGNN generators' structural filtrations (Knowledge_Distillation/data_utils_NC.py:118-128): induced degree, or
// networkx's degree centrality d * (1 / (n - 1)), divided by (max + 1e-10).  No roots, no shortest paths: one CTA per
// vicinity reads the induced degrees kernel 1's fill pass left in adeg[].
__global__ void __launch_bounds__(256) degree_filtration_kernel(Params p, ChunkView c) {
  __shared__ double redd[32];
  const int t = blockIdx.x;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int n = c.tn[t];
  if (n == 0 || c.tstatus[t] > TLC_ST_TRIVIAL) return;
  const int64_t vo = c.voff[t];
  const int32_t* __restrict__ adeg = c.adeg + vo;
  double* fval = c.fval + vo;
  const bool cen = (p.flags & TLC_F_FILT_CENTRALITY) != 0;
  const double sc = n > 1 ? __ddiv_rn(1.0, __dadd_rn((double)n, -1.0)) : 1.0;
  double mx = -1.0;
  for (int x = tid; x < n; x += nt) {
    double d = (double)adeg[x];
    if (cen) d = n > 1 ? __dmul_rn(d, sc) : 1.0;
    fval[x] = d;
    c.neg[vo + x] = -1; c.vcls[vo + x] = -1;  // (no shortest-path tree here: kernel 2v gets no neighbour hint)
    mx = fmax(mx, d);
  }
  const double m = __dadd_rn(block_reduce_max(mx, redd), 1e-10);
  for (int x = tid; x < n; x += nt) fval[x] = __ddiv_rn(fval[x], m);
}

// nx.clustering as a filtration (Knowledge_Distillation/data_utils_NC.py:122-125): c(v) = t / (d (d - 1)), t = sum over the
// neighbours w of |N(v) & N(w)| (twice the triangles through v), 0 when t == 0, then / (max + 1e-10).  One CTA per
// vicinity, a warp per vertex: for every neighbour w the lanes take the entries of w's (ascending) induced row and
// look each up in v's row by bisection.
__global__ void __launch_bounds__(256) clustering_filtration_kernel(Params p, ChunkView c) {
  __shared__ double redd[32];
  const int t = blockIdx.x;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  const int n = c.tn[t];
  if (n == 0 || c.tstatus[t] > TLC_ST_TRIVIAL) return;
  const int64_t vo = c.voff[t], ao = c.aoff[t];
  const int32_t* __restrict__ astart = c.astart + vo;
  const int32_t* __restrict__ adeg = c.adeg + vo;
  const uint32_t* __restrict__ anb = c.anb + ao;
  double* fval = c.fval + vo;
  double mx = -1.0;
  for (int x = wid; x < n; x += nw) {
    const int xa = astart[x], xd = adeg[x];
    long long tri = 0;
    for (int e = 0; e < xd; e++) {
      const int y = (int)anb[xa + e];
      const int ya = astart[y], yd = adeg[y];
      for (int j = lane; j < yd; j += 32) {
        const int z = (int)anb[ya + j];
        int lo = 0, hi = xd;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if ((int)anb[xa + mid] < z) lo = mid + 1; else hi = mid; }
        tri += (lo < xd && (int)anb[xa + lo] == z) ? 1 : 0;
      }
    }
    for (int o = 16; o; o >>= 1) tri += __shfl_xor_sync(0xffffffffu, tri, o);
    const long long d = xd;
    const double cv = tri == 0 ? 0.0 : __ddiv_rn((double)tri, (double)(d * (d - 1)));
    if (lane == 0) { fval[x] = cv; c.neg[vo + x] = -1; c.vcls[vo + x] = -1; }
    mx = fmax(mx, cv);
  }
  const double m = __dadd_rn(block_reduce_max(mx, redd), 1e-10);
  for (int x = tid; x < n; x += nt) fval[x] = __ddiv_rn(fval[x], m);
}

// Heat kernel signature as a filtration (Knowledge_Distillation/data_utils_NC.py:87-93, 115-117):
//   A = nx.adjacency_matrix(subgraph) (unweighted), L = csgraph.laplacian(A, normed=True), (lambda, phi) = eigh(L),
//   hks(x) = sum_k phi_k(x)^2 exp(-t lambda_k) = [exp(-t L)]_xx,   then / (max + 1e-10).
// With N = D^-1/2 A D^-1/2 (L = I - N on the vertices of positive degree; scipy puts 0 on the diagonal of an isolated
// vertex: hks = 1 there), exp(-t L) = e^-t exp(t N) and, N being symmetric, [exp(t N)]_xx = || exp((t/2) N) e_x ||^2.
// A WARP per source vertex x pushes e_x through the Taylor series z = sum_j ((t/2)^j / j!) N^j e_x (`terms` terms, the host
// chooses them so that the remainder is < 1e-18; ||N|| <= 1): its three vectors live in shared memory, a lane owns the rows
// a = lane, lane + 32, ... and walks each row in adjacency order (the sums do not depend on the launch geometry), and
// nothing but __syncwarp separates the terms.  The sources of one vicinity are dealt to gridDim.y CTAs of `wpc` warps, so
// that a hub's vicinity (n sources x terms x (n + 2m) operations) does not serialise on one SM.  hks_normalise_kernel
// then divides by the maximum.
__global__ void __launch_bounds__(256) hks_filtration_kernel(Params p, ChunkView c, double t, int terms, int cap, int wpc) {
  extern __shared__ __align__(16) double hsm[];
  const int tt = blockIdx.x;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5;
  const int n = c.tn[tt];
  if (n == 0 || c.tstatus[tt] > TLC_ST_TRIVIAL) return;
  const int64_t vo = c.voff[tt], ao = c.aoff[tt];
  const int32_t* __restrict__ astart = c.astart + vo;
  const int32_t* __restrict__ adeg = c.adeg + vo;
  const uint32_t* __restrict__ anb = c.anb + ao;
  double* fval = c.fval + vo;
  const bool in_smem = cap > 0;  // (the host sizes cap for the launch's largest vicinity, or 0: vectors in the arena, one warp)
  double* isd = in_smem ? hsm : c.d1 + vo;                                   // 1 / sqrt(degree), 0 for an isolated vertex
  const int per = (n + (int)gridDim.y - 1) / (int)gridDim.y;
  const int x_lo = (int)blockIdx.y * per, x_hi = min(n, x_lo + per);
  if (x_lo >= x_hi) return;
  for (int a = tid; a < n; a += nt) {
    const int dg = adeg[a];
    isd[a] = dg > 0 ? __ddiv_rn(1.0, sqrt((double)dg)) : 0.0;
    if (blockIdx.y == 0) { c.neg[vo + a] = -1; c.vcls[vo + a] = -1; }  // (no shortest-path tree here: kernel 2v gets no neighbour hint)
  }
  __syncthreads();
  if (wid >= wpc) return;
  double* y0 = in_smem ? hsm + (size_t)cap * (1 + 3 * wid) : reinterpret_cast<double*>(c.v64a + vo);
  double* y1 = in_smem ? y0 + cap : reinterpret_cast<double*>(c.v64b + vo);
  double* zz = in_smem ? y1 + cap : reinterpret_cast<double*>(c.v64c + vo);
  const double h = 0.5 * t;
  for (int x = x_lo + wid; x < x_hi; x += wpc) {
    if (adeg[x] == 0) { if (lane == 0) fval[x] = 1.0; continue; }   // (scipy: 0 on the diagonal of L -> exp(0) = 1)
    for (int a = lane; a < n; a += 32) { const double e = a == x ? 1.0 : 0.0; y0[a] = e; zz[a] = e; }
    __syncwarp();
    double cj = 1.0;
    double* src = y0;
    double* dst = y1;
    for (int j = 1; j <= terms; j++) {
      cj = cj * h / (double)j;
      for (int a = lane; a < n; a += 32) {
        const int s0 = astart[a], dg = adeg[a];
        double acc = 0.0;
        for (int q = 0; q < dg; q++) { const int b = (int)anb[s0 + q]; acc += isd[b] * src[b]; }
        const double v = isd[a] * acc;
        dst[a] = v;
        zz[a] += cj * v;
      }
      __syncwarp();
      double* tmp = src; src = dst; dst = tmp;
    }
    double part = 0.0;
    for (int a = lane; a < n; a += 32) part += zz[a] * zz[a];
    for (int o = 16; o; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) fval[x] = exp(-t) * part;
    __syncwarp();
  }
}

// filtration_val /= (max(filtration_val) + 1e-10)   data_utils_NC.py:117
__global__ void __launch_bounds__(256) hks_normalise_kernel(ChunkView c) {
  __shared__ double redd[32];
  const int tt = blockIdx.x;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int n = c.tn[tt];
  if (n == 0 || c.tstatus[tt] > TLC_ST_TRIVIAL) return;
  double* fval = c.fval + c.voff[tt];
  double mx = -1.0;
  for (int a = tid; a < n; a += nt) mx = fmax(mx, fval[a]);
  const double m = __dadd_rn(block_reduce_max(mx, redd), 1e-10);
  for (int a = tid; a < n; a += nt) fval[a] = __ddiv_rn(fval[a], m);
}

template <bool DIRECT>
static void launch_filtration_any(const Params& p, const ChunkView& c, int t0, int cnt, int block, int64_t n_max,
                                  const DirectArgs& da, cudaStream_t st) {
  // dist (8) + minw (2) + state (1) bytes per vertex in shared memory when the sub-range's largest vicinity fits;
  // graph-row route: + the vicinity bitmap and its word-prefix ranks
  size_t bmb = DIRECT ? (size_t)2 * da.W * 4 : 0;
  constexpr size_t BUDGET = 208 * 1024;  // dynamic shared memory next to the 17 KB of static queues (227 KB per CTA)
  int cap = (int)((n_max + 7) / 8 * 8);
  int bpv = 11;
  if ((size_t)cap * 11 + bmb > 190 * 1024) bpv = 9;            // very large vicinity: lean state (margins stay in the arena)
  if ((size_t)cap * bpv + bmb > BUDGET) cap = 0;               // larger still: per-vertex state in the arena
  DirectArgs da2 = da;
  if (DIRECT) {  // the graph id -> local id table, when it fits next to the per-vertex state
    const size_t lidb = ((size_t)da.g.N + 1) / 2 * 4;
    da2.lid_table = (n_max < 65535 && cap > 0 && (size_t)cap * bpv + bmb + lidb <= 190 * 1024) ? 1 : 0;
    if (getenv("TLC_NO_LID")) da2.lid_table = 0;  // (tuning experiments)
    if (da2.lid_table) bmb += lidb;
  }
  const size_t bytes = (size_t)cap * bpv + bmb;
  if (DIRECT && block < 128) block = 128;  // the prologue walks the bitmap a warp per word
  // one resident CTA per SM (large vicinities): give it 32 warps, the relaxation is latency-bound
  if (bytes + sizeof(FiltShared) > 110 * 1024 && block >= 512) block = 1024;
  if (const char* env = getenv("TLC_FILT_BLOCK")) block = atoi(env);  // (tuning experiments)
  auto go = [&](auto kern) {
    cudaFuncSetAttribute((const void*)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    cudaFuncSetAttribute((const void*)kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    kern<<<cnt, block, bytes, st>>>(p, c, t0, cap, bpv, da2);
  };
  if (cap > 0) go(filtration_kernel<DIRECT, true>);
  else go(filtration_kernel<DIRECT, false>);
  count_launch();
}

void launch_filtration(const Params& p, const ChunkView& c, int t0, int cnt, int block, int64_t n_max, cudaStream_t st) {
  launch_filtration_any<false>(p, c, t0, cnt, block, n_max, DirectArgs{}, st);
}

void launch_hks_filtration(const Params& p, const ChunkView& c, double t, int64_t n_max, cudaStream_t st) {
  // Taylor terms: (t/2)^j / j! below 1e-18 (and past the series' largest term)
  int terms = 1;
  double cj = 0.5 * t;
  while (terms < 400 && (cj > 1e-18 || terms < 0.5 * t)) { terms++; cj = cj * 0.5 * t / terms; }
  int cap = (int)((n_max + 1) / 2 * 2);
  constexpr size_t BUDGET = 200 * 1024;
  int wpc = (int)std::min<size_t>(8, (BUDGET / 8 / (size_t)std::max(cap, 1) - 1) / 3);  // warps whose three vectors fit next to isd[]
  int slices = (int)std::min<int64_t>(128, std::max<int64_t>(1, (n_max + 7) / 8));     // a source per warp of the largest vicinity's CTAs (measured: 32 slices 1.25 s, one CTA 2.58 s on 2048 PubMed-shaped node vicinities)
  if ((size_t)cap * 32 > BUDGET) { cap = 0; wpc = 1; slices = 1; }  // larger vicinities keep the (single set of) vectors in the arena
  const size_t bytes = (size_t)cap * 8 * (1 + 3 * wpc);
  cudaFuncSetAttribute((const void*)hks_filtration_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  hks_filtration_kernel<<<dim3((unsigned)c.T, (unsigned)slices), 256, bytes, st>>>(p, c, t, terms, cap, wpc);
  count_launch();
  hks_normalise_kernel<<<c.T, 256, 0, st>>>(c);
  count_launch();
}

void launch_degree_filtration(const Params& p, const ChunkView& c, cudaStream_t st) {
  if (p.flags & TLC_F_FILT_CLUSTERING) clustering_filtration_kernel<<<c.T, 256, 0, st>>>(p, c);
  else degree_filtration_kernel<<<c.T, 256, 0, st>>>(p, c);
  count_launch();
}

void launch_filtration_direct(const GraphView& g, const Params& p, const ChunkView& c, const VicinityScratch& vs,
                              const float* gminw, int t0, int cnt, int block, int64_t n_max, cudaStream_t st) {
  launch_filtration_any<true>(p, c, t0, cnt, block, n_max, DirectArgs{g, vs.ball_cache, gminw, (g.N + 31) / 32, 0}, st);
}

}  // namespace tlc
