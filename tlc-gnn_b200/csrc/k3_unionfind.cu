// k3_unionfind.cu -- kernel 3: batched union-find persistence, both sweeps, one CTA per vicinity.
//
// Replaces Union_find (accelerated_PD.py:26-113; KD copy Knowledge_Distillation/accelerated_PD.py:25-118):
//   ascending sweep  -> PD_up   pairs [old[large], old[max_node]]            (:43-67)
//   descending sweep -> PD_down pairs [old[small], old[min_node]], Neg (tree) / Pos (cycle) edges (:79-109)
//   essential pairs [min,max] and [max,min]                                  (:110)
// and the connectivity assertion of riccidist2dgm.py:318 (tree edges == n-1).
//
// The sweep is sequential only in its UNIONS (n-1 per sweep); the 2m FINDS are not.  Each step takes
// blockDim consecutive edges of the sorted order: every thread finds both roots (path halving on the
// shared-memory parent array; concurrent halving only ever re-points a vertex to one of its own
// ancestors, and no union runs meanwhile), edges whose roots already coincide are cycle edges for
// good, the rest are compacted in order (ballot + warp prefix) and resolved by warp 0 in groups of 32:
// roots are re-found, each union is applied by the warp in sweep order and broadcast so that the
// other lanes patch their stale roots in registers.  Value comparisons use the dense value classes
// of kernel 2 (same order and same ties as the float64 values); birth/death values are gathered at
// the end.  parent/class arrays live in shared memory when 8*n bytes fit, else in the HBM arena.
#include "tlc_common.cuh"

namespace tlc {
namespace {

struct UfShared {
  int32_t cl_k[1024], cl_a[1024], cl_b[1024];
  int32_t wcnt[33];
  int32_t total, nmerge, npairs, nneg, minv, maxv;
};

__global__ void union_find_kernel(Params p, ChunkView c, int smem_ints, int build_lists, int sweep_mask, int fb_only) {
  extern __shared__ int32_t dyn[];
  __shared__ UfShared sh;
  const int t = blockIdx.x;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  const int n = c.tn[t], m = c.tm[t];
  if (n == 0 || c.tstatus[t] > TLC_ST_TRIVIAL) return;
  if (fb_only && !c.tfb[t]) sweep_mask &= ~1;  // kernel 3v already produced PD_up and [min,max] of this target
  if (!sweep_mask) return;
  const bool do_asc = (sweep_mask & 1) != 0, do_desc = (sweep_mask & 2) != 0;
  const int64_t vo = c.voff[t], eo = c.eoff[t], po = c.poff(t);
  const int32_t* __restrict__ elo = c.elo + eo;
  const int32_t* __restrict__ ehi = c.ehi + eo;
  const bool in_smem = 2 * n <= smem_ints;
  int32_t* parent = in_smem ? dyn : c.vs0 + vo;
  int32_t* cls = in_smem ? dyn + n : c.vcls + vo;
  const bool keep0 = (p.flags & TLC_F_KEEP_ZERO) != 0;
  uint8_t* pkind = c.pkind + po;
  int32_t* pbv = c.pbv + po;
  int32_t* pdv = c.pdv + po;
  int32_t* neg = c.neg + vo;
  uint8_t* isneg = c.isneg + eo;
  const int ncls = c.tncls[t];

  if (in_smem) for (int x = tid; x < n; x += nt) cls[x] = c.vcls[vo + x];
  if (tid == 0) { sh.npairs = do_asc ? 0 : c.tnp[t]; sh.minv = n; sh.maxv = n; sh.nneg = 0; sh.nmerge = 0; }
  __syncthreads();
  // min_value / max_value: first vertex (ascending id) attaining them   accelerated_PD.py:35-38
  for (int x = tid; x < n; x += nt) {
    const int cx = cls[x];
    if (cx == 0) atomicMin(&sh.minv, x);
    if (cx == ncls - 1) atomicMin(&sh.maxv, x);
  }

  for (int sweep = 0; sweep < 2; sweep++) {
    if (!((sweep_mask >> sweep) & 1)) continue;
    const uint32_t* __restrict__ ord = (sweep == 0 ? c.ord_asc : c.ord_desc) + eo;
    for (int x = tid; x < n; x += nt) parent[x] = x;
    if (sweep == 1) for (int k = tid; k < m; k += nt) isneg[k] = 0;
    if (tid == 0) sh.nmerge = 0;
    __syncthreads();
    for (int base = 0; base < m; base += nt) {
      const int k = base + tid;
      int ra = 0, rb = 0;
      bool cand = false;
      if (k < m) {
        const uint32_t e = ord[k];
        ra = uf_find(parent, elo[e]);
        rb = uf_find(parent, ehi[e]);
        cand = ra != rb;
      }
      const unsigned bal = __ballot_sync(0xffffffffu, cand);
      if (lane == 0) sh.wcnt[wid] = __popc(bal);
      __syncthreads();
      int pre = 0, tot = 0;
      for (int w = 0; w < nw; w++) { const int cw = sh.wcnt[w]; if (w < wid) pre += cw; tot += cw; }
      if (cand) {
        const int j = pre + __popc(bal & lanemask_lt());
        sh.cl_k[j] = k; sh.cl_a[j] = ra; sh.cl_b[j] = rb;
      }
      __syncthreads();
      if (wid == 0 && tot > 0) {
        int np = sh.npairs, nmerge = sh.nmerge, nneg = sh.nneg;
        for (int s = 0; s < tot; s += 32) {
          const int j = s + lane;
          const bool valid = j < tot;
          int kk = 0, a = 0, b = 0;
          uint32_t e = 0;
          ra = rb = 0;
          if (valid) {
            kk = sh.cl_k[j];
            e = ord[kk];
            a = elo[e]; b = ehi[e];
            ra = uf_find(parent, sh.cl_a[j]);  // re-find from the (possibly stale) roots
            rb = uf_find(parent, sh.cl_b[j]);
          }
          __syncwarp();
          unsigned cm = __ballot_sync(0xffffffffu, valid && ra != rb);
          while (cm) {  // uniform over the warp: unions in sweep order
            const int l = __ffs(cm) - 1;
            cm &= cm - 1;
            const int A = __shfl_sync(0xffffffffu, ra, l), B = __shfl_sync(0xffffffffu, rb, l);
            const int ea = __shfl_sync(0xffffffffu, a, l), eb = __shfl_sync(0xffffffffu, b, l);
            const int kl = __shfl_sync(0xffffffffu, kk, l);
            const uint32_t el = __shfl_sync(0xffffffffu, e, l);
            if (A == B) continue;  // joined by an earlier union of this group: a cycle edge
            const int cA = cls[A], cB = cls[B];
            const int small = (cA <= cB) ? A : B, large = A + B - small;  // :61-63 / :100-102 (tie -> root of edge[0])
            const int ca = cls[ea], cb2 = cls[eb];
            if (sweep == 0) {
              const int max_node = ca > cb2 ? ea : eb;                     // :64
              if (keep0 || max(cA, cB) < cls[max_node]) {                  // :65 (KD :68-69: always)
                if (lane == 0) { pkind[np] = TLC_K_UP; pbv[np] = large; pdv[np] = max_node; }
                np++;
              }
              if (lane == 0) parent[large] = small;                        // :67
              if (ra == large) ra = small;
              if (rb == large) rb = small;
            } else {
              const int min_node = ca < cb2 ? ea : eb;                     // :103-104
              if (keep0 || min(cA, cB) > cls[min_node]) {                  // :105 (KD :108-109: always)
                if (lane == 0) { pkind[np] = TLC_K_DOWN; pbv[np] = small; pdv[np] = min_node; }
                np++;
              }
              if (lane == 0) {
                parent[small] = large;                                     // :107
                neg[nneg] = (int32_t)el;                                   // Neg_edges += [edge]  :99
                isneg[kl] = 1;
              }
              nneg++;
              if (ra == small) ra = large;
              if (rb == small) rb = large;
            }
            nmerge++;
            __syncwarp();
          }
        }
        if (lane == 0) { sh.npairs = np; sh.nmerge = nmerge; sh.nneg = nneg; }
      }
      __syncthreads();
      if (sh.nmerge == n - 1) break;  // spanning tree complete: every later edge closes a cycle
    }
    __syncthreads();
    if (tid == 0) {
      const int np = sh.npairs;
      pkind[np] = sweep == 0 ? TLC_K_ESS : TLC_K_ESS_REV;                  // :110
      pbv[np] = sweep == 0 ? sh.minv : sh.maxv;
      pdv[np] = sweep == 0 ? sh.maxv : sh.minv;
      sh.npairs = np + 1;
    }
    __syncthreads();
  }

  // Pos_edges in sweep order (accelerated_PD.py:109): ordered compaction of the non-tree flags
  const int nneg = sh.nneg;
  const int last_merges = sh.nmerge;
  if (build_lists && do_desc) {
    const uint32_t* __restrict__ ord = c.ord_desc + eo;
    int32_t* pos = c.pos + eo;
    int cursor = 0;
    for (int base = 0; base < m; base += nt) {
      const int k = base + tid;
      const bool f = k < m && !isneg[k];
      const unsigned bal = __ballot_sync(0xffffffffu, f);
      __syncthreads();
      if (lane == 0) sh.wcnt[wid] = __popc(bal);
      __syncthreads();
      int pre = 0, tot = 0;
      for (int w = 0; w < nw; w++) { const int cw = sh.wcnt[w]; if (w < wid) pre += cw; tot += cw; }
      if (f) pos[cursor + pre + __popc(bal & lanemask_lt())] = (int32_t)ord[k];
      cursor += tot;
    }
  }
  // birth / death values of the 0-dim pairs
  const int np = sh.npairs;
  const double* __restrict__ fval = c.fval + vo;
  for (int i = tid; i < np; i += nt) {
    c.pbirth[po + i] = fval[pbv[i]];
    c.pdeath[po + i] = fval[pdv[i]];
  }
  if (tid == 0) {
    c.tnp[t] = np;
    if (do_desc) { c.tnneg[t] = nneg; c.tnpos[t] = m - nneg; }
    else { c.tnneg[t] = 0; c.tnpos[t] = 0; }
    // assert len(components) == 1 (riccidist2dgm.py:318): a spanning tree has n-1 merges in either sweep
    if (last_merges != n - 1) c.tstatus[t] = TLC_ST_DISCONNECTED;
  }
}

}  // namespace

void launch_union_find(const Params& p, const ChunkView& c, int block, int smem_ints, int build_lists, int sweep_mask,
                       int fb_only, cudaStream_t st) {
  const size_t bytes = (size_t)smem_ints * 4;
  if (bytes > 48 * 1024)
    cudaFuncSetAttribute((const void*)union_find_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  union_find_kernel<<<c.T, block, bytes, st>>>(p, c, smem_ints, build_lists, sweep_mask, fb_only);
  count_launch();
}

}  // namespace tlc
