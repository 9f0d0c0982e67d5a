// k3v_sweep.cu -- kernel 3v: the ascending union-find sweep in VERTEX order, one warp per vicinity.
//
// Replaces the ascending half of Union_find (accelerated_PD.py:27-68; KD copy :25-70) and produces the
// identical pair sequence [old[large], old[max_node]] (same values, same vertex ids, same order) as
// Kruskal over the reference's (perturbed key, canonical index) edge order -- without ever sorting the
// m edges.  Kernel 2v cut the (value, id) vertex order into blocks whose owned edges are totally
// ordered block against block; here a warp walks the blocks in order:
//
//   trivial block (the overwhelmingly common case): all vertices of the block carry the same value,
//     every one of them has a neighbour in an earlier block, and all those neighbours sit in ONE
//     component R.  Each vertex then joins R through its first edge as a singleton whose value equals
//     the edge's max value: the reference's `if old[large] < old[max_node]` (:65) is false, no pair is
//     emitted, whatever the order of the block's edges.  parent[x] = R, done -- one ballot.
//   general block: every owned edge (x, y) can only merge if it is the first, in (key, index) order,
//     among the block's edges joining the same pair of components-at-block-start.  The warp keeps that
//     first edge per (x, component) ("representative"), sorts the handful of representatives by
//     (key, lo, hi) and runs the reference's union rule on them in order (:53-67).
//
// A target whose block needs more than REP_CAP representatives is flagged in tfb[] and redone by the
// edge-sorted kernels 2 + 3 (same results, different cost).  The union-find parents are ranks in shared
// memory (16-bit when n < 65536).  Connectivity (riccidist2dgm.py:318) falls out as merges == n - 1.
#include "tlc_common.cuh"
#include "tlc_sort.cuh"

namespace tlc {
namespace {

constexpr int REP_CAP = 128;
constexpr int SWEEP_WARPS = 1;  // one warp per CTA: the shared-memory footprint (parents of ONE vicinity) sets the residency

struct RepBuf {
  unsigned long long key[REP_CAP];
  int32_t lo[REP_CAP], hi[REP_CAP];  // local ids, lo < hi (canonical orientation: edge[0] = lo)
  int32_t root[REP_CAP];             // component (rank of its root) of the earlier endpoint at block start
  int32_t perm[REP_CAP];
};

__device__ __forceinline__ bool rep_less(unsigned long long ka, int la, int ha, unsigned long long kb, int lb, int hb) {
  if (ka != kb) return ka < kb;
  if (la != lb) return la < lb;  // canonical edge index order == lexicographic (lo, hi)
  return ha < hb;
}

template <typename PT>
__global__ void __launch_bounds__(SWEEP_WARPS * 32) sweep_kernel(Params p, ChunkView c, int t0, int tend, int cap) {
  extern __shared__ unsigned char dyn_raw[];
  __shared__ RepBuf reps_all[SWEEP_WARPS];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int t = t0 + blockIdx.x * SWEEP_WARPS + wid;
  if (t >= tend) return;
  const int n = c.tn[t];
  if (n == 0 || c.tstatus[t] > TLC_ST_TRIVIAL) return;
  const int64_t vo = c.voff[t], po = c.poff(t);
  const int32_t* __restrict__ vord = c.vord + vo;
  const int32_t* __restrict__ vrank = c.vrank + vo;
  const int32_t* __restrict__ bfirst = c.bfirst + vo + t;
  const int32_t* __restrict__ astart = c.astart + vo;
  const int32_t* __restrict__ adeg = c.adeg + vo;
  // rows: the induced adjacency (local neighbour ids), or on the graph-row route the graph's CSR row of vert[x]
  // mapped through the vicinity bitmap (-1: the neighbour is outside the vicinity)
  const bool direct = c.dbm != nullptr;
  const uint32_t* __restrict__ anb = direct ? reinterpret_cast<const uint32_t*>(c.gcol) : c.anb + c.aoff[t];
  const uint32_t* __restrict__ bm = direct ? c.dbm + (size_t)t * 2 * c.W : nullptr;
  const int32_t* __restrict__ vert = c.vert + vo;
  const int bW = c.W;
  auto nbr = [&](int pos) -> int { return direct ? bitmap_rank(bm, bW, (int)anb[pos]) : (int)anb[pos]; };
  const double* __restrict__ fval = c.fval + vo;
  PT* parent = n <= cap ? reinterpret_cast<PT*>(dyn_raw) + (size_t)wid * cap : reinterpret_cast<PT*>(c.vs2 + vo);
  RepBuf& rb = reps_all[wid];
  const bool keep0 = (p.flags & TLC_F_KEEP_ZERO) != 0;
  const int nb = c.tnb[t];
  if (nb < 0) return;  // kernel 2v proved that the diagram is the essential pair alone and wrote it
  const unsigned FULL = 0xffffffffu;

  for (int r = lane; r < n; r += 32) parent[r] = (PT)r;
  __syncwarp();

  int np = 0, nmerge = 0;
  int ncomp = 0;  // components among the vertices of the blocks processed so far
  int ngeneral = 0, nrowcheck = 0;  // statistics: blocks through the general path / through the row check
  bool bail = false;
  int s = 0;
  // block table, 32 blocks per coalesced load, the next group already in flight
  int cur_first = 0, nxt_first = 0;
  if (lane <= nb) nxt_first = bfirst[lane];
  int carry = 0;  // bfirst[b] of the current block (flags), handed over from the previous iteration
  bool one_block = false;
  if (nb == 1 && !keep0) {
    // ONE block: every vertex carries the same value (e.g. both roots outside the vicinity: all distances 100).  No merge
    // can emit a pair (`old[large] < old[max_node]` never holds, accelerated_PD.py:65), so only connectivity matters
    // (riccidist2dgm.py:318): a warp-parallel breadth-first search from rank 0 instead of m sequential unions.
    // parent[r] == 0 marks "reached" (rank 0 itself included).
    one_block = true;
    int32_t* queue = c.vs0 + vo;  // (kernel 2v's sort payload: free by now)
    if (lane == 0) queue[0] = 0;
    __syncwarp();
    int head = 0, tail = 1;
    while (head < tail) {
      const int lx = vord[queue[head++]];
      const int a = astart[lx], dg = adeg[lx];
      for (int j0 = 0; j0 < dg; j0 += 32) {
        const int j = j0 + lane;
        int ry = -1;
        if (j < dg) {
          const int ly = nbr(a + j);
          if (ly >= 0) { ry = vrank[ly]; if (parent[ry] == 0) ry = -1; }
        }
        const unsigned bal = __ballot_sync(FULL, ry >= 0);
        if (ry >= 0) { parent[ry] = (PT)0; queue[tail + __popc(bal & lanemask_lt())] = ry; }
        tail += __popc(bal);
        __syncwarp();
      }
    }
    nmerge = tail - 1;
  }
  for (int b = 0; b < nb && !bail && !one_block; b++) {
    if ((b & 31) == 0) {
      cur_first = nxt_first;
      const int i = b + 32 + lane;
      if (i <= nb) nxt_first = bfirst[i];
      carry = __shfl_sync(FULL, cur_first, 0);
      // a whole group of trivial blocks above a connected prefix: every vertex of the group joins the one root
      if (ncomp == 1 && !keep0) {
        const int nbk = min(32, nb - b);
        const bool triv = lane >= nbk || ((cur_first >> 30) & 3) == 1;  // bit 30 set, bit 31 clear
        if (__all_sync(FULL, triv)) {
          const int ge = (nbk < 32 ? __shfl_sync(FULL, cur_first, nbk) : __shfl_sync(FULL, nxt_first, 0)) & 0x3fffffff;
          const int R = uf_find(parent, 0);
          __syncwarp();
          for (int x = s + lane; x < ge; x += 32) parent[x] = (PT)R;
          __syncwarp();
          nmerge += ge - s;
          s = ge;
          b += nbk - 1;
          continue;
        }
      }
    }
    const int wb = carry;
    // bfirst[b + 1]: lane (b+1)&31 of the current group, or lane 0 of the next one
    const int wn = ((b + 1) & 31) ? __shfl_sync(FULL, cur_first, (b + 1) & 31) : __shfl_sync(FULL, nxt_first, 0);
    carry = wn;
    const int e = wn & 0x3fffffff;
    const bool distinct = wb < 0;
    const bool all_out = ((wb >> 30) & 1) != 0;  // every vertex of the block has a neighbour in an earlier block

    // ---------------- trivial block test ----------------
    bool done = false;
    if (!distinct && !keep0 && all_out) {
      int R = -1;
      bool ok = true;
      if (ncomp == 1) {
        // the processed prefix is ONE component: every earlier-block neighbour is in it, no row needs reading
        R = uf_find(parent, 0);
      } else {
        nrowcheck++;
        // several components below: all earlier-block neighbours of the block must share one root
        for (int x = s; x < e && ok; x++) {
          const int lx = vord[x];
          const int a = astart[lx], dg = adeg[lx];
          for (int j0 = 0; j0 < dg && ok; j0 += 32) {
            const int j = j0 + lane;
            const int ly = j < dg ? nbr(a + j) : -1;
            const int ry = ly >= 0 ? vrank[ly] : e;  // e: "not in an earlier block", ignored
            const bool out = ry < s;
            const int rt = out ? uf_find(parent, ry) : -1;
            const unsigned bo = __ballot_sync(FULL, out);
            if (bo) {
              if (R < 0) R = __shfl_sync(FULL, rt, __ffs(bo) - 1);
              ok = __all_sync(FULL, !out || rt == R);
            }
          }
        }
      }
      if (ok) {
        __syncwarp();
        for (int x = s + lane; x < e; x += 32) parent[x] = (PT)R;
        __syncwarp();
        nmerge += e - s;
        done = true;  // ncomp unchanged: the block's vertices joined an existing component
      }
    }

    // ---------------- general block ----------------
    if (!done) {
      ngeneral++;
      const int merges_before = nmerge;
      int nrep = 0;
      // A block of EQUAL values is swept in two stages.  Its edges into earlier blocks carry keys fl(M + fl((mu+1)e-6))
      // with mu < M, its in-block edges the one key fl(M + fl((M+1)e-6)): stage 1 = representatives of the edges into
      // earlier blocks (sorted, applied in order); stage 2 = the in-block edges, whose order is then purely the canonical
      // (lo, hi) index order -- block vertices ascending, each row ascending -- and needs no buffering at all.  (A clique
      // of k tied vertices would otherwise need k(k-1)/2 representatives.)  The strict key separation is verified below.
      const bool staged = !distinct;
      const int ylim0 = staged ? s : e;  // stage 1 looks at neighbours of rank < min(x, ylim0)
      for (int x = s; x < e && !bail; x++) {
        const int xrep0 = nrep;
        const int lx = vord[x];
        const double fx = fval[lx];
        const int xa = astart[lx], xdg = adeg[lx];
        // owned edges of x = its neighbours of smaller rank.  Few earlier vertices (the first ranks, typically the
        // two roots with their huge rows): probe each of them in x's ascending row instead of scanning the row
        const bool probe = x <= 32;
        for (int j0 = 0; j0 < (probe ? 1 : xdg) && !bail; j0 += 32) {
          const int j = j0 + lane;
          int y = 0, ly = 0, ry = -1, lo = 0, hi = 0;
          unsigned long long K = 0;
          bool valid = false;
          if (probe) {
            if (lane < min(x, ylim0)) {
              y = lane;
              ly = vord[y];
              const int key = direct ? vert[ly] : ly;  // rows ascend in graph id and in local id alike
              int l0 = 0, h0 = xdg;  // lower bound of ly in the row
              while (l0 < h0) { const int mid = (l0 + h0) >> 1; if ((int)anb[xa + mid] < key) l0 = mid + 1; else h0 = mid; }
              valid = l0 < xdg && (int)anb[xa + l0] == key;
            }
          } else if (j < xdg) {
            ly = nbr(xa + j);
            if (ly >= 0) {
              y = vrank[ly];
              valid = y < min(x, ylim0);  // the edge is owned by its later endpoint
            }
          }
          if (valid) {
            ry = uf_find(parent, y);  // no union has happened in this block yet: component at block start
            K = f64_to_ordered(key_asc(fx, fval[ly]));
            lo = min(lx, ly); hi = max(lx, ly);
          }
          if (!__any_sync(FULL, valid)) continue;  // no owned edge among these 32 entries
          // first edge, in (key, lo, hi) order, per component within this chunk
          bool is_min = valid;
          for (int i = 0; i < 32; i++) {
            const int ri = __shfl_sync(FULL, ry, i);
            const unsigned long long Ki = __shfl_sync(FULL, K, i);
            const int loi = __shfl_sync(FULL, lo, i), hii = __shfl_sync(FULL, hi, i);
            if (is_min && i != lane && ri == ry && ri >= 0 && rep_less(Ki, loi, hii, K, lo, hi)) is_min = false;
          }
          // merge with the representatives x already has (earlier chunks of the same vertex)
          bool append = false;
          if (is_min) {
            int found = -1;
            for (int q = xrep0; q < nrep; q++) if (rb.root[q] == ry) found = q;
            if (found >= 0) {
              if (rep_less(K, lo, hi, rb.key[found], rb.lo[found], rb.hi[found])) { rb.key[found] = K; rb.lo[found] = lo; rb.hi[found] = hi; }
            } else append = true;
          }
          const unsigned ba = __ballot_sync(FULL, append);
          const int add = __popc(ba);
          if (nrep + add > REP_CAP) { bail = true; break; }
          if (append) {
            const int q = nrep + __popc(ba & lanemask_lt());
            rb.key[q] = K; rb.lo[q] = lo; rb.hi[q] = hi; rb.root[q] = ry;
          }
          nrep += add;
          __syncwarp();
        }
      }
      if (!bail) {
        // order the representatives: perm[rank] = q
        for (int q = lane; q < nrep; q += 32) {
          const unsigned long long K = rb.key[q];
          const int lo = rb.lo[q], hi = rb.hi[q];
          int rk = 0;
          for (int i = 0; i < nrep; i++) rk += rep_less(rb.key[i], rb.lo[i], rb.hi[i], K, lo, hi) ? 1 : 0;
          rb.perm[rk] = q;
        }
        __syncwarp();
        // the reference's union step for edge [a, b], a < b (local ids); lane 0 only
        auto apply_edge = [&](int a, int bb) {
          const int A = uf_find(parent, vrank[a]), B = uf_find(parent, vrank[bb]);
          if (A == B) return;
          const int la = vord[A], lb = vord[B];  // local ids of the two roots
          const double fA = fval[la], fB = fval[lb];
          const bool a_small = fA <= fB;         // small = pu if new[pu] <= new[pv]   :61-63
          const int small = a_small ? A : B, large = a_small ? B : A;
          const int llarge = a_small ? lb : la;
          const double flarge = a_small ? fB : fA;
          const double fa = fval[a], fb = fval[bb];
          const int max_node = fa > fb ? a : bb;  // :64
          const double fmaxn = fa > fb ? fa : fb;
          if (keep0 || flarge < fmaxn) {          // :65 (KD :68-69: always)
            c.pkind[po + np] = TLC_K_UP;
            c.pbv[po + np] = llarge; c.pdv[po + np] = max_node;
            c.pbirth[po + np] = flarge; c.pdeath[po + np] = fmaxn;
            np++;
          }
          parent[large] = (PT)small;            // :67
          nmerge++;
        };
        if (lane == 0) {
          for (int i = 0; i < nrep; i++) {
            const int q = rb.perm[i];
            apply_edge(rb.lo[q], rb.hi[q]);
          }
        }
        if (staged) {
          // every stage-1 key must lie strictly below the in-block key (true whenever the smallest value is 0, i.e. a
          // root is in the vicinity; verified rather than assumed)
          const double M = fval[vord[s]];
          const unsigned long long kin = f64_to_ordered(key_asc(M, M));
          bool ok = true;
          for (int q = lane; q < nrep; q += 32) ok = ok && rb.key[q] < kin;
          if (!__all_sync(FULL, ok)) bail = true;
          __syncwarp();
          // stage 2: in-block edges in canonical order
          int stage2_edges = 0;
          for (int x = s; x < e && !bail; x++) {
            const int lx = vord[x];
            const int xa = astart[lx], xdg = adeg[lx];
            // small block (typically the two roots with their huge rows): probe the <= 32 later block vertices in x's
            // ascending row instead of scanning the row
            const bool probe2 = e - s <= 33;
            for (int j0 = 0; j0 < (probe2 ? 1 : xdg); j0 += 32) {
              const int j = j0 + lane;
              int ly = -1;
              if (probe2) {
                const int y = x + 1 + lane;
                if (y < e) {
                  const int cand = vord[y];
                  const int key = direct ? vert[cand] : cand;
                  int l0 = 0, h0 = xdg;
                  while (l0 < h0) { const int mid = (l0 + h0) >> 1; if ((int)anb[xa + mid] < key) l0 = mid + 1; else h0 = mid; }
                  if (l0 < xdg && (int)anb[xa + l0] == key) ly = cand;
                }
              } else if (j < xdg) {
                ly = nbr(xa + j);
                if (ly >= 0) { const int y = vrank[ly]; if (!(y > x && y < e)) ly = -1; }
              }
              unsigned mk = __ballot_sync(FULL, ly >= 0);
              // the in-block unions run on one lane: a block with thousands of them goes to the edge-sorted kernels instead
              stage2_edges += __popc(mk);
              if (stage2_edges > 4096) { bail = true; break; }
              while (mk) {
                const int i = __ffs(mk) - 1;
                mk &= mk - 1;
                const int lyi = __shfl_sync(FULL, ly, i);
                if (lane == 0) apply_edge(lx, lyi);  // (equal values: rank order == id order, so lx < lyi)
              }
              __syncwarp();
            }
          }
        }
        np = __shfl_sync(FULL, np, 0);
        nmerge = __shfl_sync(FULL, nmerge, 0);
        __syncwarp();
        ncomp += (e - s) - (nmerge - merges_before);
      }
    }
    s = e;
  }

  if (lane == 0 && c.fb_counter) { atomicAdd(c.fb_counter + 1, ngeneral); atomicAdd(c.fb_counter + 2, nrowcheck); atomicAdd(c.fb_counter + 3, nb); }
  if (lane == 0) {
    if (bail) {
      c.tfb[t] = 1;
      if (c.fb_counter) atomicAdd(c.fb_counter, 1);
    } else {
      const int lmin = c.tminv[t], lmax = c.tmaxv[t];
      c.pkind[po + np] = TLC_K_ESS;               // [min_value, max_value]   accelerated_PD.py:110
      c.pbv[po + np] = lmin; c.pdv[po + np] = lmax;
      c.pbirth[po + np] = fval[lmin]; c.pdeath[po + np] = fval[lmax];
      c.tnp[t] = np + 1;
      c.tnneg[t] = 0; c.tnpos[t] = 0;
      if (nmerge != n - 1) c.tstatus[t] = TLC_ST_DISCONNECTED;  // assert len(components) == 1   riccidist2dgm.py:318
    }
  }
}

}  // namespace

void launch_sweep(const Params& p, const ChunkView& c, int t0, int cnt, int64_t n_max, cudaStream_t st) {
  // parents in shared memory when SWEEP_WARPS vicinities of the chunk's largest size fit
  const bool narrow = n_max < 65536;
  const size_t esz = narrow ? 2 : 4;
  const size_t budget = 220 * 1024;
  int cap = (int)((n_max + 7) / 8 * 8);
  if ((size_t)cap * esz * SWEEP_WARPS > budget) cap = 0;
  const size_t bytes = (size_t)cap * esz * SWEEP_WARPS;
  const int grid = (cnt + SWEEP_WARPS - 1) / SWEEP_WARPS;
  if (narrow) {
    cudaFuncSetAttribute((const void*)sweep_kernel<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    cudaFuncSetAttribute((const void*)sweep_kernel<uint16_t>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    sweep_kernel<uint16_t><<<grid, SWEEP_WARPS * 32, bytes, st>>>(p, c, t0, t0 + cnt, cap);
  } else {
    cudaFuncSetAttribute((const void*)sweep_kernel<int32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    sweep_kernel<int32_t><<<grid, SWEEP_WARPS * 32, bytes, st>>>(p, c, t0, t0 + cnt, cap);
  }
  count_launch();
}

}  // namespace tlc
