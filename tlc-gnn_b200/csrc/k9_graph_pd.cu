// k9_graph_pd.cu -- kernel 9: persistence diagrams of a batch of caller-supplied graphs under a caller-supplied
// filtration (tlc_graph_batch_diagrams_dev), and the gradient of the pair values in that filtration
// (tlc_graph_batch_grad_dev).
//
// Graph t of a batch owns vertices noff[t] .. noff[t+1] and edges eoff[t] .. eoff[t+1] (batch-global vertex ids; the edge
// order is the sweeps' tie-break, as in tlc_union_find).  Its pairs are what the pipeline gives for a node-mode vicinity
// equal to that graph with filtration values f[noff[t] .. noff[t+1]].  Two routes, chosen per graph from its size:
//   fused  : graph_pd_kernel, a TEAM per graph with its whole state in shared memory -- a warp for n <= 64 / m <= 256,
//            a 128-thread CTA for n <= 256 / m <= 2048, a 256-thread CTA for n <= 1024 / m <= 4096 (kernel S's classes).
//            Stages 4-6 of kernel S (k0_small.cu) without the image: the perturbed float64 keys (accelerated_PD.py:18-21)
//            bitonic-sorted on (key, edge index), both union-find sweeps (:26-113), the loop pairing (:115-178)
//   staged : larger graphs, kernels 2 + 3 (+ 3b) over a ChunkView of the batch's own offsets (graph_fill_kernel writes the
//            local edge ids, fval and zeroed counters first, graph_export_kernel maps the pairs to batch-global ids)
// Both write a graph's pairs into the batch's staging area at soff[t] = noff[t] + eoff[t] + t (capacity n + m + 1) and its
// count into np[t]; kernel 7's scan / gather then compact them into the caller's arrays in graph order.  No atomics decide
// where anything lands, so the output is the same bits from call to call and whatever else the batch holds.
//
// Every pair has birth = f[bv] and death = f[dv] (copied, not computed), and the pairing is locally constant in f, so
// d birth / d f and d death / d f are indicator vectors: the gradient is a scatter of the point gradients onto the
// vertices that carry them.  graph_grad_kernel does it with a warp per graph, deterministically: the point references are
// counting-sorted by vertex in reference order (point k's birth term before its death term, k increasing), then every
// vertex sums its own list in that order.  No floating-point atomics.
#include <algorithm>
#include <cstdint>

#include "tlc_common.cuh"
#include "tlc_sort.cuh"

namespace tlc {
namespace {

constexpr unsigned FULLM = 0xffffffffu;

// per-team shared memory of the fused route: n <= NC vertices, m <= MC edges (MC a power of two >= 32)
template <int NC, int MC>
struct K9Mem {
  static constexpr size_t o_fv = 0;                          // f64[NC] filtration values
  static constexpr size_t o_key = o_fv + (size_t)NC * 8;     // u64[MC] sort keys
  static constexpr size_t o_pmx = o_key + (size_t)MC * 8;    // i32[NC] loops: (largest rank on the climb) << 10 | child end
  static constexpr size_t o_int = o_pmx + (size_t)NC * 4;    // i32[4]  team scalars
  static constexpr size_t o_sidx = o_int + 16;               // u16[MC] sorted edge indices; Pos edges after sweep 2
  static constexpr size_t o_elo = o_sidx + (size_t)MC * 2;   // u16[MC] local endpoints
  static constexpr size_t o_ehi = o_elo + (size_t)MC * 2;    // u16[MC]
  static constexpr size_t o_ark = o_ehi + (size_t)MC * 2;    // u16[MC] rank of every edge in the ascending sweep
  static constexpr size_t o_neg = o_ark + (size_t)MC * 2;    // u16[NC] Neg edges in sweep order
  static constexpr size_t o_par = o_neg + (size_t)NC * 2;    // u16[NC] union-find parents
  static constexpr size_t o_tpa = o_par + (size_t)NC * 2;    // u16[NC] loops: tree parents
  static constexpr size_t o_tpr = o_tpa + (size_t)NC * 2;    // u16[NC] loops: rank of the parent edge
  static constexpr size_t o_stp = o_tpr + (size_t)NC * 2;    // u16[NC] loops: visit stamp
  static constexpr size_t bytes = (o_stp + (size_t)NC * 2 + 15) / 16 * 16;
};

template <int NT>
__device__ __forceinline__ void team_sync() {
  if constexpr (NT == 32) __syncwarp(); else __syncthreads();
}
template <int NT>
__device__ __forceinline__ bool team_any(bool v) {
  if constexpr (NT == 32) return __any_sync(FULLM, v); else return __syncthreads_or(v ? 1 : 0) != 0;
}

template <int NT, int NC, int MC>
__global__ void __launch_bounds__(NT == 32 ? 128 : NT) graph_pd_kernel(GraphBatchView b, const int32_t* __restrict__ list,
                                                                      int cnt) {
  using M = K9Mem<NC, MC>;
  extern __shared__ __align__(16) unsigned char k9_dyn[];
  constexpr int TPB = NT == 32 ? 4 : 1;  // teams per CTA
  const int team = NT == 32 ? (int)(threadIdx.x >> 5) : 0;
  const int tid = NT == 32 ? (int)(threadIdx.x & 31) : (int)threadIdx.x;
  const int i = blockIdx.x * TPB + team;
  if (i >= cnt) return;  // (uniform over the team)
  unsigned char* base = k9_dyn + (size_t)team * M::bytes;
  double* fv = reinterpret_cast<double*>(base + M::o_fv);
  unsigned long long* skey = reinterpret_cast<unsigned long long*>(base + M::o_key);
  int32_t* pmx = reinterpret_cast<int32_t*>(base + M::o_pmx);
  int32_t* sint = reinterpret_cast<int32_t*>(base + M::o_int);
  uint16_t* sidx = reinterpret_cast<uint16_t*>(base + M::o_sidx);
  uint16_t* elo = reinterpret_cast<uint16_t*>(base + M::o_elo);
  uint16_t* ehi = reinterpret_cast<uint16_t*>(base + M::o_ehi);
  uint16_t* ark = reinterpret_cast<uint16_t*>(base + M::o_ark);
  uint16_t* negl = reinterpret_cast<uint16_t*>(base + M::o_neg);
  uint16_t* par = reinterpret_cast<uint16_t*>(base + M::o_par);
  uint16_t* tpa = reinterpret_cast<uint16_t*>(base + M::o_tpa);
  uint16_t* tpr = reinterpret_cast<uint16_t*>(base + M::o_tpr);
  uint16_t* stp = reinterpret_cast<uint16_t*>(base + M::o_stp);

  const int t = list[i];
  const int64_t v0 = b.noff[t], e0 = b.eoff[t];
  const int n = (int)(b.noff[t + 1] - v0), m = (int)(b.eoff[t + 1] - e0);
  const int64_t so = b.soff[t];
  const bool keep0 = (b.flags & TLC_F_KEEP_ZERO) != 0, ext = (b.flags & TLC_F_EXTENDED) != 0;
  const bool do_desc = (b.flags & TLC_F_ASC_ONLY) == 0;

  // ---------------- 1. load f and the edges ----------------
  bool bad = false;
  for (int x = tid; x < n; x += NT) { const double f = b.f[v0 + x]; fv[x] = f; bad |= !isfinite(f); }
  for (int k = tid; k < m; k += NT) { elo[k] = (uint16_t)(b.ea[e0 + k] - v0); ehi[k] = (uint16_t)(b.eb[e0 + k] - v0); }
  bad = team_any<NT>(bad);
  int status = n == 0 ? TLC_ST_EMPTY : (bad ? TLC_ST_NONFINITE : TLC_ST_OK);
  team_sync<NT>();

  int np = 0, nneg = 0, npos = 0;  // (meaningful on the team's first warp)
  if (status == TLC_ST_OK) {
    // min_value / max_value: first vertex (ascending id) attaining them   accelerated_PD.py:35-38
    int minv = 0, maxv = 0;
    if (tid < 32) {
      double lmx = -INFINITY, lmn = INFINITY;
      for (int x = tid; x < n; x += 32) { lmx = fmax(lmx, fv[x]); lmn = fmin(lmn, fv[x]); }
      for (int o = 16; o; o >>= 1) {
        lmx = fmax(lmx, __shfl_xor_sync(FULLM, lmx, o));
        lmn = fmin(lmn, __shfl_xor_sync(FULLM, lmn, o));
      }
      int imn = n, imx = n;
      for (int x = tid; x < n; x += 32) { if (fv[x] == lmn) imn = min(imn, x); if (fv[x] == lmx) imx = min(imx, x); }
      for (int o = 16; o; o >>= 1) {
        imn = min(imn, __shfl_xor_sync(FULLM, imn, o));
        imx = min(imx, __shfl_xor_sync(FULLM, imx, o));
      }
      minv = imn; maxv = imx;
    }
    int P2 = 32;
    while (P2 < m) P2 <<= 1;
    for (int sweep = 0; sweep < (do_desc ? 2 : 1); sweep++) {
      // ---------------- 2./3. keys asc = M + (mu + 1) * 1e-6, desc = mu - (101 - M) * 1e-6; sort on (key, index) ----
      for (int e = tid; e < P2; e += NT) {
        unsigned long long k = ~0ull;
        if (e < m) {
          const double fa = fv[elo[e]], fb = fv[ehi[e]];
          k = sweep == 0 ? f64_to_ordered(key_asc(fa, fb)) : ~f64_to_ordered(key_desc(fa, fb));
          if (k == ~0ull) k = ~0ull - 1;  // (keeps real edges ahead of the padding; unreachable for finite keys)
        }
        skey[e] = k;
        sidx[e] = (uint16_t)e;
      }
      team_sync<NT>();
      for (int kk = 2; kk <= P2; kk <<= 1) {
        for (int j = kk >> 1; j > 0; j >>= 1) {
          for (int q = tid; q < P2; q += NT) {
            const int l = q ^ j;
            if (l > q) {
              const unsigned long long kq = skey[q], kl = skey[l];
              const uint16_t xq = sidx[q], xl = sidx[l];
              const bool gt = kq > kl || (kq == kl && xq > xl);
              if (gt == ((q & kk) == 0)) { skey[q] = kl; skey[l] = kq; sidx[q] = xl; sidx[l] = xq; }
            }
          }
          team_sync<NT>();
        }
      }
      if (sweep == 0 && do_desc && ext) for (int k = tid; k < m; k += NT) ark[sidx[k]] = (uint16_t)k;
      for (int x = tid; x < n; x += NT) par[x] = (uint16_t)x;
      team_sync<NT>();
      // ---------------- 4. Kruskal over the sorted edges: 32 finds at a time, unions in sweep order ----------------
      if (tid < 32) {
        const int lane = tid;
        int merges = 0, wcur = 0;  // descending sweep: Pos edges compacted in place at the front of sidx[]
        for (int k0 = 0; k0 < m; k0 += 32) {
          const int k = k0 + lane;
          const bool valid = k < m;
          int e = 0, ea = 0, eb = 0, ra = 0, rb = 0;
          if (valid) { e = sidx[k]; ea = elo[e]; eb = ehi[e]; ra = uf_find(par, ea); rb = uf_find(par, eb); }
          __syncwarp();
          unsigned cm = __ballot_sync(FULLM, valid && ra != rb);
          unsigned negm = 0;
          while (cm) {
            const int l = __ffs(cm) - 1;
            cm &= cm - 1;
            const int Ar = __shfl_sync(FULLM, ra, l), Br = __shfl_sync(FULLM, rb, l);
            if (Ar == Br) continue;  // joined by an earlier union of this group: a cycle edge
            const int xa = __shfl_sync(FULLM, ea, l), xb = __shfl_sync(FULLM, eb, l);
            const int el = __shfl_sync(FULLM, e, l);
            const int small = fv[Ar] <= fv[Br] ? Ar : Br, large = Ar + Br - small;  // :61-63 / :100-102 (tie -> root of edge[0])
            const double fa = fv[xa], fb = fv[xb];
            if (sweep == 0) {
              const int max_node = fa > fb ? xa : xb;  // :64
              if (keep0 || fv[large] < fv[max_node]) {  // :65 (KD :68-69: always)
                if (lane == 0) {
                  const int64_t o = so + np;
                  b.stage.kind[o] = TLC_K_UP; b.stage.bv[o] = (int32_t)(v0 + large); b.stage.dv[o] = (int32_t)(v0 + max_node);
                  b.stage.birth[o] = fv[large]; b.stage.death[o] = fv[max_node];
                }
                np++;
              }
              if (lane == 0) par[large] = (uint16_t)small;  // :67
              if (ra == large) ra = small;
              if (rb == large) rb = small;
            } else {
              const int min_node = fa < fb ? xa : xb;  // :103-104
              if (keep0 || fv[small] > fv[min_node]) {  // :105 (KD :108-109: always)
                if (lane == 0) {
                  const int64_t o = so + np;
                  b.stage.kind[o] = TLC_K_DOWN; b.stage.bv[o] = (int32_t)(v0 + small); b.stage.dv[o] = (int32_t)(v0 + min_node);
                  b.stage.birth[o] = fv[small]; b.stage.death[o] = fv[min_node];
                }
                np++;
              }
              if (lane == 0) { par[small] = (uint16_t)large; negl[nneg] = (uint16_t)el; }  // :107, Neg_edges += [edge]  :99
              nneg++;
              negm |= 1u << l;
              if (ra == small) ra = large;
              if (rb == small) rb = large;
            }
            merges++;
            __syncwarp();
          }
          if (sweep == 1) {  // Pos_edges in sweep order   :109
            const unsigned posm = __ballot_sync(FULLM, valid) & ~negm;
            __syncwarp();
            if ((posm >> lane) & 1u) sidx[wcur + __popc(posm & lanemask_lt())] = (uint16_t)e;
            wcur += __popc(posm);
            __syncwarp();
          } else if (merges == n - 1) break;  // spanning tree complete: every later edge closes a cycle
        }
        if (sweep == 1) npos = wcur;
        // essential pair of the sweep   :110
        if (lane == 0) {
          const int bvx = sweep == 0 ? minv : maxv, dvx = sweep == 0 ? maxv : minv;
          const int64_t o = so + np;
          b.stage.kind[o] = sweep == 0 ? TLC_K_ESS : TLC_K_ESS_REV;
          b.stage.bv[o] = (int32_t)(v0 + bvx); b.stage.dv[o] = (int32_t)(v0 + dvx);
          b.stage.birth[o] = fv[bvx]; b.stage.death[o] = fv[dvx];
        }
        np++;
        // assert len(components) == 1   riccidist2dgm.py:318
        if (sweep == 0 && merges != n - 1) status = TLC_ST_DISCONNECTED;
        if (lane == 0) sint[0] = status;
      }
      team_sync<NT>();
      status = sint[0];
      team_sync<NT>();
      if (status != TLC_ST_OK) break;
    }

    // ---------------- 5. loops: Accelerate_PD   accelerated_PD.py:115-178 (the team's first warp) ----------------
    if (status == TLC_ST_OK && ext && tid < 32) {
      const int lane = tid;
      if (nneg == 0) status = TLC_ST_NO_TREE_EDGES;  // list(Nodes)[0] -> IndexError   :122 (single-vertex graph)
      else {
        for (int x = lane; x < n; x += 32) { tpa[x] = (uint16_t)x; stp[x] = 0xffff; tpr[x] = 0xffff; }
        __syncwarp();
        // root the tree of the Neg edges at the first endpoint of the first Neg edge   :119-125
        // (tpr == 0xffff marks "not reached yet"; the root is reached from the start)
        if (lane == 0) tpr[elo[negl[0]]] = 0xfffe;
        __syncwarp();
        for (int round = 0; round < n; round++) {
          bool ch = false;
          for (int q = lane; q < nneg; q += 32) {
            const int e = negl[q];
            const int xa = elo[e], xb = ehi[e];
            const bool ha = tpr[xa] != 0xffff, hb = tpr[xb] != 0xffff;
            if (ha && !hb) { tpa[xb] = (uint16_t)xa; tpr[xb] = ark[e]; ch = true; }
            else if (hb && !ha) { tpa[xa] = (uint16_t)xb; tpr[xa] = ark[e]; ch = true; }
          }
          __syncwarp();
          if (!__any_sync(FULLM, ch)) break;
        }
        // sequential sweep over the positive edges (sidx[0..npos) in sweep order) on the first lane
        if (lane == 0) {
          for (int k = 0; k < npos; k++) {
            const int pe = sidx[k];
            const int p0 = elo[pe], p1 = ehi[pe];
            int rc = ark[pe];
            // Loop = (p0 -> lca) + (p1 -> lca)   :131-151: the two climbs alternate, each stamping its own mark, until one
            // steps on the other's mark; every stamped vertex keeps the largest parent-edge rank met below it on its side
            const uint16_t mk0 = (uint16_t)(2 * k), mk1 = (uint16_t)(2 * k + 1);
            int best0 = -1, best1 = -1;
            {
              int x0 = p0, x1 = p1;
              stp[x0] = mk0; pmx[x0] = -1;
              stp[x1] = mk1; pmx[x1] = -1;  // (p0 != p1)
              for (;;) {
                const int q0 = (int)tpa[x0];
                if (q0 != x0) {
                  best0 = max(best0, ((int)tpr[x0] << 10) | x0);
                  if (stp[q0] == mk1) { best1 = pmx[q0]; break; }
                  stp[q0] = mk0; pmx[q0] = best0; x0 = q0;
                }
                const int q1 = (int)tpa[x1];
                if (q1 != x1) {
                  best1 = max(best1, ((int)tpr[x1] << 10) | x1);
                  if (stp[q1] == mk0) { best0 = pmx[q1]; break; }
                  stp[q1] = mk1; pmx[q1] = best1; x1 = q1;
                }
              }
            }
            const int in0 = best0 > best1 ? 1 : 0;       // (ranks are distinct)
            const int bc = (in0 ? best0 : best1) & 1023;  // child end of the cycle's largest edge
            const int by = (int)tpa[bc];                  // large_edge = (bc, by)   :155-159
            const int la = min(bc, by), lb = max(bc, by);
            const int lvv = fv[la] >= fv[lb] ? la : lb;   // large_value = max(old[large_edge])
            const int lov = fv[p0] <= fv[p1] ? p0 : p1;   // low_value   = min(old[pos_edge])
            if (keep0 || fv[lvv] > fv[lov]) {  // :160-165 (KD :169-170: always)
              const int64_t o = so + np;
              b.stage.kind[o] = TLC_K_ONE; b.stage.bv[o] = (int32_t)(v0 + lov); b.stage.dv[o] = (int32_t)(v0 + lvv);
              b.stage.birth[o] = fv[lov]; b.stage.death[o] = fv[lvv];
              np++;
            }
            // change the parent   :168-176
            int node = in0 ? p0 : p1, nodec = in0 ? p1 : p0;
            for (;;) {
              const int tp = (int)tpa[node], tr = tpr[node];
              tpa[node] = (uint16_t)nodec; tpr[node] = (uint16_t)rc;
              if (node == bc) break;
              nodec = node; rc = tr; node = tp;
            }
          }
        }
      }
    }
  }
  if (tid == 0) {
    b.np[t] = diag_pairs((uint8_t)status, np);
    b.status[t] = (uint8_t)status;
  }
}

// staged route, before kernels 2 / 3 / 3b: a warp per staged graph s (graph t = tidx[s]) writes its sizes, zeroed counters,
// status, fval and local edge ids into the chunk arena
__global__ void __launch_bounds__(256) graph_fill_kernel(GraphBatchView b, ChunkView c) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t s = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); s < c.T; s += nwarps) {
    const int64_t t = c.tidx[s];
    const int64_t v0 = b.noff[t], e0 = b.eoff[t];
    const int n = (int)(b.noff[t + 1] - v0), m = (int)(b.eoff[t + 1] - e0);
    double* fval = c.fval + c.voff[s];
    int32_t* elo = c.elo + c.eoff[s];
    int32_t* ehi = c.ehi + c.eoff[s];
    bool bad = false;
    for (int x = lane; x < n; x += 32) { const double f = b.f[v0 + x]; fval[x] = f; bad |= !isfinite(f); }
    for (int k = lane; k < m; k += 32) { elo[k] = (int32_t)(b.ea[e0 + k] - v0); ehi[k] = (int32_t)(b.eb[e0 + k] - v0); }
    bad = __any_sync(FULLM, bad);
    if (lane == 0) {
      c.tn[s] = n; c.tm[s] = m;
      c.tnp[s] = 0; c.tnpos[s] = 0; c.tnneg[s] = 0;
      c.tstatus[s] = n == 0 ? TLC_ST_EMPTY : (bad ? TLC_ST_NONFINITE : TLC_ST_OK);
    }
  }
}

// staged route, after kernels 2 / 3 / 3b: a warp per staged graph copies its pairs into the staging area at soff[t],
// vertex ids made batch-global, and records its count and status
__global__ void __launch_bounds__(256) graph_export_kernel(GraphBatchView b, ChunkView c) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t s = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); s < c.T; s += nwarps) {
    const int64_t t = c.tidx[s];
    const uint8_t st = c.tstatus[s];
    const int cnt = diag_pairs(st, c.tnp[s]);
    if (lane == 0) { b.np[t] = cnt; b.status[t] = st; }
    const int64_t po = c.poff((int)s), d = b.soff[t], v0 = b.noff[t];
    for (int i = lane; i < cnt; i += 32) {
      b.stage.kind[d + i] = c.pkind[po + i];
      b.stage.bv[d + i] = (int32_t)(v0 + c.pbv[po + i]);
      b.stage.dv[d + i] = (int32_t)(v0 + c.pdv[po + i]);
      b.stage.birth[d + i] = c.pbirth[po + i];
      b.stage.death[d + i] = c.pdeath[po + i];
    }
  }
}

// grad_f of every vertex of graph t, a warp per graph.  cnt[N] and lst[2 (N + M + D)] are the batch's scratch: graph t
// uses cnt[noff[t] ..] and lst[2 soff[t] ..] (its n + m + 1 points have 2 (n + m + 1) references)
__global__ void __launch_bounds__(256) graph_grad_kernel(GraphBatchView b, const int64_t* __restrict__ poff,
                                                         const int32_t* __restrict__ bv, const int32_t* __restrict__ dv,
                                                         const double* __restrict__ gb, const double* __restrict__ gd,
                                                         int32_t* __restrict__ cnt_all, int32_t* __restrict__ lst_all,
                                                         double* __restrict__ grad_f) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < b.D; t += nwarps) {
    const int64_t v0 = b.noff[t];
    const int n = (int)(b.noff[t + 1] - v0);
    const int64_t cap = (int64_t)n + (b.eoff[t + 1] - b.eoff[t]) + 1;
    const int64_t k0 = poff[t];
    const int64_t P = min(max(poff[t + 1] - k0, (int64_t)0), cap);
    const int R = (int)(2 * P);
    int32_t* cnt = cnt_all + v0;
    int32_t* lst = lst_all + 2 * b.soff[t];
    // vertex (local id) of reference r: point k0 + r / 2, its birth (r even) or death (r odd) vertex; -1 = no term
    auto ref_vertex = [&](int r) -> int {
      const int64_t k = k0 + (r >> 1);
      if ((r & 1) ? gd == nullptr : gb == nullptr) return -1;
      const int64_t v = ((r & 1) ? dv[k] : bv[k]) - v0;
      return v >= 0 && v < n ? (int)v : -1;  // (a point of another graph contributes nothing here)
    };
    for (int x = lane; x < n; x += 32) cnt[x] = 0;
    __syncwarp();
    for (int r = lane; r < R; r += 32) { const int v = ref_vertex(r); if (v >= 0) atomicAdd(&cnt[v], 1); }
    __syncwarp();
    int run = 0;  // exclusive scan: cnt[x] = first slot of x's list
    for (int x0 = 0; x0 < n; x0 += 32) {
      const int x = x0 + lane;
      const int c = x < n ? cnt[x] : 0;
      int inc = c;
      for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(FULLM, inc, o); if (lane >= o) inc += u; }
      if (x < n) cnt[x] = run + inc - c;
      run += __shfl_sync(FULLM, inc, 31);
    }
    __syncwarp();
    // stable placement, 32 references at a time in reference order; cnt[x] advances to the end of x's list
    for (int r0 = 0; r0 < R; r0 += 32) {
      const int r = r0 + lane;
      const int v = r < R ? ref_vertex(r) : -1;
      const unsigned peers = __match_any_sync(FULLM, v);
      if (v >= 0) lst[cnt[v] + __popc(peers & lanemask_lt())] = r;
      __syncwarp();
      if (v >= 0 && lane == 31 - __clz(peers)) cnt[v] += __popc(peers);
      __syncwarp();
    }
    for (int x = lane; x < n; x += 32) {
      const int s = x == 0 ? 0 : cnt[x - 1], e = cnt[x];
      double g = 0.0;
      for (int j = s; j < e; j++) {
        const int r = lst[j];
        const int64_t k = k0 + (r >> 1);
        g += (r & 1) ? gd[k] : gb[k];
      }
      grad_f[v0 + x] = g;
    }
  }
}

int warp_grid(int64_t warps, int sm_count) {
  return (int)std::max<int64_t>(1, std::min<int64_t>((warps + 7) / 8, (int64_t)sm_count * 16));
}

template <int NT, int NC, int MC>
void launch_class(const GraphBatchView& b, const int32_t* list, int cnt, cudaStream_t st) {
  if (cnt <= 0) return;
  constexpr int TPB = NT == 32 ? 4 : 1;
  const size_t bytes = K9Mem<NC, MC>::bytes * TPB;
  if (bytes > 48 * 1024)
    cudaFuncSetAttribute((const void*)graph_pd_kernel<NT, NC, MC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  graph_pd_kernel<NT, NC, MC><<<(cnt + TPB - 1) / TPB, NT * TPB, bytes, st>>>(b, list, cnt);
  count_launch();
}

}  // namespace

void launch_graph_pd_small(const GraphBatchView& b, const int32_t* const lists[3], const int counts[3], cudaStream_t st) {
  launch_class<32, GRAPH_A_N, GRAPH_A_M>(b, lists[0], counts[0], st);
  launch_class<128, GRAPH_B_N, GRAPH_B_M>(b, lists[1], counts[1], st);
  launch_class<256, GRAPH_C_N, GRAPH_C_M>(b, lists[2], counts[2], st);
}

void launch_graph_fill(const GraphBatchView& b, const ChunkView& c, int sm_count, cudaStream_t st) {
  if (c.T <= 0) return;
  graph_fill_kernel<<<warp_grid(c.T, sm_count), 256, 0, st>>>(b, c);
  count_launch();
}

void launch_graph_export(const GraphBatchView& b, const ChunkView& c, int sm_count, cudaStream_t st) {
  if (c.T <= 0) return;
  graph_export_kernel<<<warp_grid(c.T, sm_count), 256, 0, st>>>(b, c);
  count_launch();
}

void launch_graph_grad(const GraphBatchView& b, const int64_t* poff, const int32_t* bv, const int32_t* dv, const double* gb,
                       const double* gd, int32_t* cnt, int32_t* lst, double* grad_f, int sm_count, cudaStream_t st) {
  if (b.D <= 0) return;
  graph_grad_kernel<<<warp_grid(b.D, sm_count), 256, 0, st>>>(b, poff, bv, dv, gb, gd, cnt, lst, grad_f);
  count_launch();
}

}  // namespace tlc
