// k0_small.cu -- kernel S: the WHOLE per-target path for small vicinities in one launch, state in shared memory.
//
// For vicinities of a few dozen vertices (the reference's own settings: 2 hops on Cora / PubMed-like graphs,
// 1 hop on Computers / Photo, baselines/TLCGNN.py:102) the staged pipeline of tlc_api.cu is bound by its host round trip
// (counting pass -> plan -> five launches) and by one CTA per vicinity per stage.  Here one TEAM -- a warp for
// n <= 64, a 128-thread CTA for n <= 256 -- takes a target from its two ids to the finished image row:
//   1. vicinity   : AND of the two cached k-hop ball bitmaps, members in ascending graph id = canonical local ids
//                   (riccidist2dgm.py:311-316; node mode: Knowledge_Distillation/data_utils_NC.py:97-100)
//   2. adjacency  : ONE ordered compaction over the members' concatenated CSR rows (membership = bisection of the
//                   sorted member list), weights kappa + 1 (:225); the canonical (lo, hi) edge list falls out of it
//   3. filtration : build_fv (:20-61).  Distances are the least fixpoint of d[y] = min_x fl(d[x] + w(x, y)) -- exactly
//                   what Dijkstra returns, fl(+) being monotone -- reached by entry-parallel relaxation rounds; tree
//                   parent = smallest local id y with fl(d[y] + w) == d[x]; path re-summed x -> root in CPython order
//   4. edge orders: the reference's perturbed float64 keys (accelerated_PD.py:18-21), bitonic sort on (key, index)
//   5. sweeps     : Union_find (accelerated_PD.py:40-109): finds of 32 sorted edges in parallel, unions in order
//   6. loops      : Accelerate_PD (:115-178), the tree walk of kernel 3b on the team's first lane
//   7. image      : PersistenceImager.transform (PersistenceImager.pyx:352-388), separable form of kernel 4
// A target that does not fit the team's capacity is appended to a device-side list for the next larger class (and,
// after the largest, for the staged pipeline).  Results are bit-identical to the staged kernels: same canonical order,
// same IEEE operation order (tests/test_gpu_small.py compares pairs and images with the oracle).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <type_traits>

#include "tlc_common.cuh"
#include "tlc_sort.cuh"

namespace tlc {
namespace {

constexpr unsigned FULLM = 0xffffffffu;
constexpr int PBUF = 32;  // pairs buffered before the team rasterises them

// ---- team primitives: NT == 32 -> a warp (several teams per CTA), NT > 32 -> the whole CTA ----
template <int NT>
struct Team {
  int tid;          // thread within the team
  int32_t* xchg;    // NT > 32: 40 ints of CTA-shared scratch
  __device__ __forceinline__ void sync() const {
    if constexpr (NT == 32) __syncwarp(); else __syncthreads();
  }
  __device__ __forceinline__ bool any(bool v) const {
    if constexpr (NT == 32) return __any_sync(FULLM, v); else return __syncthreads_or(v ? 1 : 0) != 0;
  }
  // exclusive prefix sum over the team in thread order; total returned through `tot`
  __device__ __forceinline__ int exscan(int v, int& tot) const {
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(FULLM, inc, o); if ((tid & 31) >= o) inc += u; }
    if constexpr (NT == 32) {
      tot = __shfl_sync(FULLM, inc, 31);
      return inc - v;
    } else {
      const int w = tid >> 5;
      __syncthreads();
      if ((tid & 31) == 31) xchg[w] = inc;
      __syncthreads();
      int base = 0, t = 0;
#pragma unroll
      for (int i = 0; i < NT / 32; i++) { const int c = xchg[i]; if (i < w) base += c; t += c; }
      tot = t;
      return base + inc - v;
    }
  }
  // values of the team's first thread to everyone
  __device__ __forceinline__ void bcast4(int& a0, int& a1, int& a2, int& a3) const {
    if constexpr (NT == 32) {
      a0 = __shfl_sync(FULLM, a0, 0); a1 = __shfl_sync(FULLM, a1, 0); a2 = __shfl_sync(FULLM, a2, 0); a3 = __shfl_sync(FULLM, a3, 0);
    } else {
      __syncthreads();
      if (tid == 0) { xchg[32] = a0; xchg[33] = a1; xchg[34] = a2; xchg[35] = a3; }
      __syncthreads();
      a0 = xchg[32]; a1 = xchg[33]; a2 = xchg[34]; a3 = xchg[35];
      __syncthreads();
    }
  }
  __device__ __forceinline__ double maxd(double v) const {
#pragma unroll
    for (int o = 16; o; o >>= 1) v = fmax(v, __shfl_xor_sync(FULLM, v, o));
    if constexpr (NT == 32) return v;
    else {
      double* xd = reinterpret_cast<double*>(xchg + 8);
      __syncthreads();
      if ((tid & 31) == 0) xd[tid >> 5] = v;
      __syncthreads();
      double t = xd[0];
#pragma unroll
      for (int i = 1; i < NT / 32; i++) t = fmax(t, xd[i]);
      return t;
    }
  }
};

#ifdef SMALL_PROFILE
#define SPROF(slot) do { if (tid == 0 && a.prof) { const long long now_ = clock64(); atomicAdd(&a.prof[a.cls * 16 + (slot)], (unsigned long long)(now_ - tprof)); tprof = now_; } } while (0)
#else
#define SPROF(slot) do { } while (0)
#endif

struct SmallArgs {
  GraphView g;
  Params p;
  const int32_t* targets;   // [E][2] graph ids
  const int32_t* list;      // nullptr: targets 0..E-1; else the rows to process
  const int* list_count;    // device count of `list`
  int64_t E;
  const uint32_t* ball_cache;  // [N][W] closed k-hop balls
  int W;
  double* out_pi;           // [E][25]
  float* out_pi32;          // [E][25] or nullptr
  uint8_t* out_status;      // [E] or nullptr
  int32_t* defer_list;      // rows that do not fit this class
  int* defer_count;
  int32_t* big_list;        // class A: rows with more than big_thresh vertices (no class takes them), or nullptr
  int* big_count;
  int big_thresh;
  int32_t *out_n, *out_m;   // optional [E]: vicinity sizes of the handled targets
  // optional diagram output (tlc_small_diagrams): pairs of row t at poff[t]
  const int64_t* poff;
  int32_t* dnp;
  uint8_t* dkind;
  int32_t *dbv, *ddv;
  double *dbirth, *ddeath;
  int want_desc;            // run the descending sweep although no loops are wanted (diagram output)
  int graph_ids;            // diagram output: vertices as graph ids (vert[lid]) instead of local ids
  SmallStats* stats;        // device accumulators (handled rows, sum n, sum m, algorithmic bytes) or nullptr
  const unsigned long long* ball_acc;  // [N][2] per ball: expanded degree sum, rowptr pairs read (byte accounting)
  int cls;                  // 0: class A, 1: class B, 2: class C
  unsigned long long* prof; // -DSMALL_PROFILE builds: clock64 ticks per class and stage [3][16]
};

template <int NC, int AC>
struct SmallMem {
  using LID = typename std::conditional<(NC <= 256), uint8_t, uint16_t>::type;
  static constexpr int MC = AC / 2;
  // 8-byte arrays first, then 4-, 2- and 1-byte ones
  static constexpr size_t o_aw = 0;                                  // f64[AC]; later: sort keys u64[MC] + index u16[MC]
  static constexpr size_t o_d1 = o_aw + (size_t)AC * 8;              // u64[NC]
  static constexpr size_t o_d2 = o_d1 + (size_t)NC * 8;              // u64[NC]
  static constexpr size_t o_fv = o_d2 + (size_t)NC * 8;              // f64[NC]
  static constexpr size_t o_pb = o_fv + (size_t)NC * 8;              // f64[2 * PBUF] buffered (birth, death)
  static constexpr size_t o_img = o_pb + (size_t)PBUF * 16;          // f64[26]
  static constexpr size_t o_vert = o_img + 26 * 8;                   // i32[NC]
  static constexpr size_t o_ast = o_vert + (size_t)NC * 4;           // i32[NC + 1]  adjacency row starts
  static constexpr size_t o_gra = o_ast + (size_t)(NC + 1) * 4;      // i32[NC]      graph row starts      | later tpe (parent entry)
  static constexpr size_t o_gpre = o_gra + (size_t)NC * 4;           // i32[NC + 1]  prefix of graph degrees
  static constexpr size_t o_pm = o_gpre + (size_t)(NC + 1) * 4;      // i32[NC]      loops: (largest rank below the vertex on its climb) << 10 | child end
  static constexpr size_t o_ark = o_pm + (size_t)NC * 4;             // u16[MC]      rank of every edge in the ascending sweep
  static constexpr size_t o_neg = o_ark + (size_t)MC * 2;            // u16[NC]      Neg edges in sweep order
  static constexpr size_t o_tpr = o_neg + (size_t)NC * 2;            // u16[NC]      loops: rank of the parent edge
  static constexpr size_t o_stp = o_tpr + (size_t)NC * 2;            // u16[NC]      loops: visit stamp
  static constexpr size_t o_anb = o_stp + (size_t)NC * 2;            // LID[AC]
  static constexpr size_t o_src = o_anb + (size_t)AC * sizeof(LID);  // LID[AC]
  static constexpr size_t o_elo = o_src + (size_t)AC * sizeof(LID);  // LID[MC]
  static constexpr size_t o_ehi = o_elo + (size_t)MC * sizeof(LID);  // LID[MC]
  static constexpr size_t o_par = o_ehi + (size_t)MC * sizeof(LID);  // LID[NC]  union-find parents
  static constexpr size_t o_tpa = o_par + (size_t)NC * sizeof(LID);  // LID[NC]  loops: tree parents
  static constexpr size_t bytes = (o_tpa + (size_t)NC * sizeof(LID) + 15) / 16 * 16;
};

// rasterise the buffered pairs: a thread per pair, 25 partial sums reduced over the warp, one atomic per pixel and warp
template <int NT>
__device__ __forceinline__ void flush_pairs(const Team<NT>& tm, const double* pb, int cnt, double* img) {
  const double step = ((1.0 + 1.0 / 5) - 0.0) / (5 + 1);  // np.linspace(0, 1 + pixel, res + 1, endpoint=False)  PersistenceImager.pyx:311-314
  for (int k0 = 0; k0 < cnt; k0 += NT) {
    const int k = k0 + tm.tid;
    const bool act = k < cnt;
    if (!__any_sync(FULLM, act)) continue;
    double acc[25];
#pragma unroll
    for (int i = 0; i < 25; i++) acc[i] = 0.0;
    if (act) {
      const double birth = pb[2 * k], death = pb[2 * k + 1];
      const double pers = death - birth;  // skew :366
      const double w = ramp_weight(pers);
      double gb[5], gp[5];
      cdf_diffs(5, step, birth, pers, gb, gp);
#pragma unroll
      for (int i = 0; i < 5; i++) {
        const double wb = w * gb[i];
#pragma unroll
        for (int j = 0; j < 5; j++) acc[i * 5 + j] = wb * gp[j];
      }
    }
#pragma unroll
    for (int i = 0; i < 25; i++) {
      double v = acc[i];
#pragma unroll
      for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULLM, v, o);
      if ((tm.tid & 31) == 0) {
        if constexpr (NT == 32) img[i] += v; else atomicAdd(&img[i], v);
      }
    }
  }
  tm.sync();
}

template <int NT, int NC, int AC>
__global__ void __launch_bounds__(NT == 32 ? 128 : NT) small_kernel(SmallArgs a) {
  using M = SmallMem<NC, AC>;
  using LID = typename M::LID;
  constexpr int MC = M::MC;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(16) int32_t xchg_all[48];
  constexpr int TEAMS = NT == 32 ? 4 : 1;  // teams per CTA
  const int team_in_cta = NT == 32 ? (threadIdx.x >> 5) : 0;
  Team<NT> tm{NT == 32 ? (int)(threadIdx.x & 31) : (int)threadIdx.x, xchg_all};
  const int tid = tm.tid;
  unsigned char* base = smem_raw + (size_t)team_in_cta * M::bytes;
  double* aw = reinterpret_cast<double*>(base + M::o_aw);
  unsigned long long* skey = reinterpret_cast<unsigned long long*>(base + M::o_aw);           // (after the filtration)
  uint16_t* sidx = reinterpret_cast<uint16_t*>(base + M::o_aw + (size_t)MC * 8);
  unsigned long long* d1 = reinterpret_cast<unsigned long long*>(base + M::o_d1);
  unsigned long long* d2 = reinterpret_cast<unsigned long long*>(base + M::o_d2);
  double* fv = reinterpret_cast<double*>(base + M::o_fv);
  double* pb = reinterpret_cast<double*>(base + M::o_pb);
  double* img = reinterpret_cast<double*>(base + M::o_img);
  int32_t* vert = reinterpret_cast<int32_t*>(base + M::o_vert);
  int32_t* ast = reinterpret_cast<int32_t*>(base + M::o_ast);
  int32_t* gra = reinterpret_cast<int32_t*>(base + M::o_gra);
  int32_t* tpe = gra;  // (graph row starts are dead once the adjacency exists)
  int32_t* gpre = reinterpret_cast<int32_t*>(base + M::o_gpre);
  int32_t* pmx = reinterpret_cast<int32_t*>(base + M::o_pm);
  uint16_t* ark = reinterpret_cast<uint16_t*>(base + M::o_ark);
  uint16_t* negl = reinterpret_cast<uint16_t*>(base + M::o_neg);
  uint16_t* tpr = reinterpret_cast<uint16_t*>(base + M::o_tpr);
  uint16_t* stp = reinterpret_cast<uint16_t*>(base + M::o_stp);
  LID* anb = reinterpret_cast<LID*>(base + M::o_anb);
  LID* esrc = reinterpret_cast<LID*>(base + M::o_src);
  LID* elo = reinterpret_cast<LID*>(base + M::o_elo);
  LID* ehi = reinterpret_cast<LID*>(base + M::o_ehi);
  LID* par = reinterpret_cast<LID*>(base + M::o_par);
  LID* tpa = reinterpret_cast<LID*>(base + M::o_tpa);

  const GraphView& g = a.g;
  const Params& p = a.p;
  const bool node_mode = p.mode == TLC_MODE_NODE, forced = p.mode == TLC_MODE_EDGE_FORCED;
  const bool plain = (p.flags & TLC_F_SUM_PLAIN) != 0, keep0 = (p.flags & TLC_F_KEEP_ZERO) != 0;
  const bool ext = (p.flags & TLC_F_EXTENDED) != 0;
  const bool norm = (p.flags & TLC_F_NORM) != 0;
  const bool do_desc = ext || a.want_desc != 0;
  auto vid = [&](int x) { return a.graph_ids ? vert[x] : x; };  // diagram output: local -> graph id
  const int W = a.W;
  const int64_t count = a.list ? (int64_t)*a.list_count : a.E;
  const int64_t nteams = (int64_t)gridDim.x * TEAMS;

  for (int64_t it = (int64_t)blockIdx.x * TEAMS + team_in_cta; it < count; it += nteams) {
    tm.sync();  // (the previous target's last readers are done)
    const int64_t row = a.list ? (int64_t)a.list[it] : it;
    const int32_t u = a.targets[2 * row], v = a.targets[2 * row + 1];
    double* out = a.out_pi + row * 25;
    float* out32 = a.out_pi32 ? a.out_pi32 + row * 25 : nullptr;
    uint8_t status = TLC_ST_OK;
#ifdef SMALL_PROFILE
    long long tprof = clock64();
#endif
    int n = 0, m = 0, np = 0;
    int gpre_total = 0;  // sum of the members' graph degrees (D_S)
    const int64_t dpo = a.poff ? a.poff[row] : 0;
    bool deferred = false;

    // unknown_target, written out: calling it changes this kernel's register allocation
    bool bad = u < 0 || u >= g.N || (!node_mode && (v < 0 || v >= g.N));
    if (!bad) bad = g.rowptr[u + 1] == g.rowptr[u] || (!node_mode && g.rowptr[v + 1] == g.rowptr[v]);
    if (bad) status = TLC_ST_UNKNOWN_NODE;

    if (status == TLC_ST_OK) {
      // ---------------- 1. vicinity ----------------
      const uint32_t* __restrict__ bu = a.ball_cache + (size_t)u * W;
      const uint32_t* __restrict__ bv = a.ball_cache + (size_t)(node_mode ? u : v) * W;
      for (int w0 = 0; w0 < W; w0 += NT) {
        const int w = w0 + tid;
        uint32_t bits = 0;
        if (w < W) bits = combine_balls(p.mode, bu[w], bv[w], w, u, v);
        int tot;
        const int pre = tm.exscan(__popc(bits), tot);
        if (n + tot <= NC) {
          int k = n + pre;
          while (bits) { const int b = __ffs(bits) - 1; bits &= bits - 1; vert[k++] = w * 32 + b; }
        }
        n += tot;
      }
      if (n > NC) deferred = true;
    }
    if (deferred) {
      // too many vertices for this class: on to the next one -- or, beyond every class (class A sees that at once from
      // the popcount), straight to the staged pipeline's list, so that it can start while classes B / C still run
      if (tid == 0) {
        if (a.big_list && n > a.big_thresh) a.big_list[atomicAdd(a.big_count, 1)] = (int32_t)row;
        else a.defer_list[atomicAdd(a.defer_count, 1)] = (int32_t)row;
      }
      continue;
    }
    SPROF(0);
    int lu = -1, lv = -1;
    if (status == TLC_ST_OK) {
      tm.sync();
      if (n == 0) status = TLC_ST_EMPTY;  // assert len(components) == 1 with no component   :318
    }
    if (status == TLC_ST_OK) {
      // ---------------- 2. induced adjacency (both directions, rows ascending) + canonical edge list ----------------
      for (int i = tid; i < n; i += NT) {
        const int32_t x = vert[i];
        const int32_t r0 = g.rowptr[x];
        gra[i] = r0;
        gpre[i + 1] = g.rowptr[x + 1] - r0;  // degree, scanned below
        ast[i + 1] = 0;                      // kept entries per row, scanned below
      }
      if (tid == 0) { gpre[0] = 0; ast[0] = 0; }
      tm.sync();
      {  // inclusive scan of the degrees in gpre[1..n]
        int run = 0;
        for (int b0 = 1; b0 <= n; b0 += NT) {
          const int i = b0 + tid;
          const int vdeg = i <= n ? gpre[i] : 0;
          int tot;
          const int ex = tm.exscan(vdeg, tot);
          if (i <= n) gpre[i] = run + ex + vdeg;
          run += tot;
        }
      }
      tm.sync();
      const int D = gpre[n];
      gpre_total = D;
      int acur = 0, ecur = 0;
      int r = 0;
      bool overflow = false;
      for (int e0 = 0; e0 < D; e0 += NT) {
        const int e = e0 + tid;
        int lid = -1, gpos = 0;
        if (e < D) {
          while (e >= gpre[r + 1]) r++;
          gpos = gra[r] + (e - gpre[r]);
          const int32_t y = g.col[gpos];
          int lo = 0, hi = n;
          while (lo < hi) { const int mid = (lo + hi) >> 1; if (vert[mid] < y) lo = mid + 1; else hi = mid; }
          if (lo < n && vert[lo] == y) lid = lo;
        }
        const bool keep = lid >= 0, up = keep && lid > r;
        int tot;
        const int pre = tm.exscan((keep ? 1 : 0) | (up ? 0x10000 : 0), tot);
        const int tk = tot & 0xffff, tu = tot >> 16;
        if (acur + tk > AC || ecur + tu > MC) { overflow = true; break; }
        if (keep) {
          const int o = acur + (pre & 0xffff);
          anb[o] = (LID)lid; esrc[o] = (LID)r;
          aw[o] = __dadd_rn(g.kappa[gpos], 1.0);  // graph[a][b]['weight'] = kappa + 1   riccidist2dgm.py:225
          atomicAdd(&ast[r + 1], 1);
          if (up) { const int q = ecur + (pre >> 16); elo[q] = (LID)r; ehi[q] = (LID)lid; }
        }
        acur += tk; ecur += tu;
      }
      if (overflow) {  // (uniform over the team)
        if (tid == 0) a.defer_list[atomicAdd(a.defer_count, 1)] = (int32_t)row;
        continue;
      }
      m = ecur;
      tm.sync();
      {  // inclusive scan of the kept entries per row in ast[1..n]
        int run = 0;
        for (int b0 = 1; b0 <= n; b0 += NT) {
          const int i = b0 + tid;
          const int vdeg = i <= n ? ast[i] : 0;
          int tot;
          const int ex = tm.exscan(vdeg, tot);
          if (i <= n) ast[i] = run + ex + vdeg;
          run += tot;
        }
      }
      // local roots
      {
        int lo = 0, hi = n;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (vert[mid] < u) lo = mid + 1; else hi = mid; }
        lu = (lo < n && vert[lo] == u) ? lo : -1;
        if (node_mode) lv = lu;
        else {
          lo = 0; hi = n;
          while (lo < hi) { const int mid = (lo + hi) >> 1; if (vert[mid] < v) lo = mid + 1; else hi = mid; }
          lv = (lo < n && vert[lo] == v) ? lo : -1;
        }
      }
      tm.sync();
      if ((node_mode || forced) && m == 0) status = TLC_ST_EMPTY;  // `return None, None`  data_utils_NC.py:103-104, data_utils_LP.py:117-118
    }
    SPROF(1);
    const bool live0 = status == TLC_ST_OK;  // the staged pipeline's "live" targets: a valid, non-empty vicinity (byte accounting)
    const int A2 = status == TLC_ST_OK ? ast[n] : 0;  // directed entries = 2m
    const bool roots_in = lu >= 0 && lv >= 0;

    if (status == TLC_ST_OK) {
      // ---------------- 3. filtration: build_fv(weight_graph=True, norm)   riccidist2dgm.py:20-61 ----------------
      if (!roots_in) {
        // nx.NodeNotFound for every vertex
        for (int x = tid; x < n; x += NT) { d1[x] = (unsigned long long)__double_as_longlong(NO_PATH_DIST); d2[x] = d1[x]; }
      } else {
        const bool two = !node_mode && lu != lv;
        for (int rr = 0; rr < (two ? 2 : 1); rr++) {
          const int root = rr == 0 ? lu : lv;
          unsigned long long* dist = rr == 0 ? d1 : d2;
          for (int x = tid; x < n; x += NT) { dist[x] = x == root ? 0ull : INF_BITS; tpe[x] = 0x7fffffff; }
          tm.sync();
          // least fixpoint of d[y] = min_x fl(d[x] + w(x, y)): relaxation rounds over all directed entries
          for (int round = 0; round <= n; round++) {
            bool ch = false;
            for (int e = tid; e < A2; e += NT) {
              const unsigned long long dxb = dist[esrc[e]];
              if (dxb == INF_BITS) continue;
              const unsigned long long tb = (unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dxb), aw[e]));
              const int y = (int)anb[e];
              if (tb < dist[y]) { atomicMin(&dist[y], tb); ch = true; }
            }
            tm.sync();
            if (!tm.any(ch)) break;
          }
          // tree parent of x: the smallest local id y (= smallest row position) with fl(d[y] + w(y, x)) == d[x]
          for (int e = tid; e < A2; e += NT) {
            const int x = (int)esrc[e];
            const unsigned long long dxb = dist[x], dyb = dist[anb[e]];
            if (x == root || dxb == INF_BITS || dyb == INF_BITS) continue;
            if ((unsigned long long)__double_as_longlong(__dadd_rn(__longlong_as_double((long long)dyb), aw[e])) == dxb) atomicMin(&tpe[x], e);
          }
          tm.sync();
          // path sums in python order, x -> root   :30,35
          double res_x[(NC + NT - 1) / NT];
#pragma unroll
          for (int j = 0; j < (NC + NT - 1) / NT; j++) {
            const int x = tid + j * NT;
            double res = 0.0;
            if (x < n) {
              if (x == root) res = 0.0;
              else if (dist[x] == INF_BITS) res = NO_PATH_DIST;  // nx.NetworkXNoPath (disconnected vicinity: status 3 from the sweep)
              else {
                PySum ps{0.0, 0.0, 0};
                int y = x, guard = 0;
                while (y != root && guard++ <= n) { const int e = tpe[y]; pysum_add(ps, aw[e], plain); y = (int)anb[e]; }
                res = pysum_get(ps, plain);
              }
            }
            res_x[j] = res;
          }
          tm.sync();
#pragma unroll
          for (int j = 0; j < (NC + NT - 1) / NT; j++) {
            const int x = tid + j * NT;
            if (x < n) dist[x] = (unsigned long long)__double_as_longlong(res_x[j]);
          }
          tm.sync();
        }
        if (!two) for (int x = tid; x < n; x += NT) d2[x] = d1[x];
        tm.sync();
        if (tid == 0) zero_roots(d1, d2, lu, lv);
        tm.sync();
      }
      // descriptors + normalisation
      double mx = -1.0, sm = -1.0;
      for (int x = tid; x < n; x += NT) {
        const double da = __longlong_as_double((long long)d1[x]), db = __longlong_as_double((long long)d2[x]);
        mx = fmax(mx, fv_descriptor(TLC_DESC_MAX, node_mode, da, db));
        sm = fmax(sm, fv_descriptor(TLC_DESC_SUM, node_mode, da, db));
      }
      double smax = tm.maxd(mx), ssum = tm.maxd(sm);
      if (norm) {  // fv_normalisers, written out for the same reason
        if (p.flags & TLC_F_NORM_EPS) { smax = __dadd_rn(smax, 1e-10); ssum = __dadd_rn(ssum, 1e-10); }
        else if (smax == 0.0 || ssum == 0.0) {
          // ZeroDivisionError -> zeros (:54-56,356-357); every vertex is a root here, so n <= 2 and the connectivity
          // assertion (:318, which the reference checks first) fails iff the two roots are not adjacent
          status = (m == n - 1) ? TLC_ST_DEGENERATE : TLC_ST_DISCONNECTED;
        }
      }
      if (status == TLC_ST_OK) {
        for (int x = tid; x < n; x += NT) {
          const double da = __longlong_as_double((long long)d1[x]), db = __longlong_as_double((long long)d2[x]);
          fv[x] = fv_value(p.descriptor, node_mode, norm, smax, ssum, da, db);
        }
      }
      tm.sync();
    }

    SPROF(2);
    int npb = 0;  // pairs waiting in the buffer
    if (tid < 25) img[tid] = 0.0;
    tm.sync();

    if (status == TLC_ST_OK) {
      // ---------------- 4./5. edge orders and sweeps   accelerated_PD.py:6-23, 26-113 ----------------
      // min_value / max_value: first vertex (ascending id) attaining them   :35-38
      int minv = 0, maxv = 0;
      {
        double lmx = -1e300, lmn = -1e300;  // (min through max of the negated values)
        for (int x = tid; x < n; x += NT) { const double f = fv[x]; lmx = fmax(lmx, f); lmn = fmax(lmn, -f); }
        const double fmx = tm.maxd(lmx), fmn = -tm.maxd(lmn);
        if (tid == 0) { ast[0] = 0x7fffffff; gpre[0] = 0x7fffffff; }  // (both arrays are dead by now)
        tm.sync();
        for (int x = tid; x < n; x += NT) { const double f = fv[x]; if (f == fmn) atomicMin(&ast[0], x); if (f == fmx) atomicMin(&gpre[0], x); }
        tm.sync();
        minv = ast[0]; maxv = gpre[0];
        tm.sync();
      }
      int P2 = 32;
      while (P2 < m) P2 <<= 1;
      int nneg = 0, npos = 0;
      int merges_asc = 0;
      for (int sweep = 0; sweep < (do_desc ? 2 : 1); sweep++) {
        // keys: asc = M + (mu + 1) * 1e-6, desc = mu - (101 - M) * 1e-6, ties by canonical edge index   :18-21,40-41,76-77
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
        tm.sync();
        for (int kk = 2; kk <= P2; kk <<= 1) {
          for (int j = kk >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < P2; i += NT) {
              const int l = i ^ j;
              if (l > i) {
                const unsigned long long ki = skey[i], kl = skey[l];
                const uint16_t xi = sidx[i], xl = sidx[l];
                const bool gt = ki > kl || (ki == kl && xi > xl);
                const bool upw = (i & kk) == 0;
                if (gt == upw) { skey[i] = kl; skey[l] = ki; sidx[i] = xl; sidx[l] = xi; }
              }
            }
            tm.sync();
          }
        }
        SPROF(3 + 2 * sweep);
        if (sweep == 0 && do_desc && ext) { for (int k = tid; k < m; k += NT) ark[sidx[k]] = (uint16_t)k; }
        for (int x = tid; x < n; x += NT) par[x] = (LID)x;
        tm.sync();
        // Kruskal over the sorted edges: 32 finds at a time, unions in sweep order (first warp of the team)
        int merges = 0;
        if (tid < 32) {
          const int lane = tid;
          int wcur = 0;  // descending sweep: Pos edges compacted in place at the front of sidx[]
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
              const double fA = fv[Ar], fB = fv[Br];
              const int small = fA <= fB ? Ar : Br, large = Ar + Br - small;  // :61-63 / :100-102 (tie -> root of edge[0])
              const double fa = fv[xa], fb = fv[xb];
              if (sweep == 0) {
                const int max_node = fa > fb ? xa : xb;  // :64
                if (keep0 || fv[large] < fv[max_node]) {  // :65 (KD :68-69: always)
                  if (lane == 0) {
                    if (a.poff) { const int64_t o = dpo + np; a.dkind[o] = TLC_K_UP; a.dbv[o] = vid(large); a.ddv[o] = vid(max_node); a.dbirth[o] = fv[large]; a.ddeath[o] = fv[max_node]; }
                    if (((p.img_mask >> TLC_K_UP) & 1u) && fv[max_node] > fv[large]) { pb[2 * npb] = fv[large]; pb[2 * npb + 1] = fv[max_node]; }
                  }
                  if (((p.img_mask >> TLC_K_UP) & 1u) && fv[max_node] > fv[large]) npb++;
                  np++;
                }
                if (lane == 0) par[large] = (LID)small;  // :67
                if (ra == large) ra = small;
                if (rb == large) rb = small;
              } else {
                const int min_node = fa < fb ? xa : xb;  // :103-104
                if (keep0 || fv[small] > fv[min_node]) {  // :105 (KD :108-109: always)
                  if (lane == 0 && a.poff) { const int64_t o = dpo + np; a.dkind[o] = TLC_K_DOWN; a.dbv[o] = vid(small); a.ddv[o] = vid(min_node); a.dbirth[o] = fv[small]; a.ddeath[o] = fv[min_node]; }
                  np++;  // (PD_down has death <= birth: weight 0 in the image, SURVEY.md F6)
                }
                if (lane == 0) { par[small] = (LID)large; negl[nneg] = (uint16_t)el; }  // :107, Neg_edges += [edge]  :99
                nneg++;
                negm |= 1u << l;
                if (ra == small) ra = large;
                if (rb == small) rb = large;
              }
              merges++;
              __syncwarp();
              if (npb == PBUF) { flush_pairs<32>(Team<32>{lane, nullptr}, pb, npb, img); npb = 0; }
            }
            if (sweep == 1) {  // Pos_edges in sweep order   :109
              const unsigned vm = __ballot_sync(FULLM, valid);
              const unsigned posm = vm & ~negm;
              __syncwarp();
              if ((posm >> lane) & 1u) sidx[wcur + __popc(posm & lanemask_lt())] = (uint16_t)e;
              wcur += __popc(posm);
              __syncwarp();
            } else if (merges == n - 1) break;  // spanning tree complete: every later edge closes a cycle
          }
          if (sweep == 1) npos = wcur;
        }
        if constexpr (NT > 32) {  // hand the warp's counters to the rest of the team
          __syncthreads();
          if (tid == 0) { xchg_all[40] = np; xchg_all[41] = npb; xchg_all[42] = merges; xchg_all[43] = nneg; xchg_all[44] = npos; }
          __syncthreads();
          np = xchg_all[40]; npb = xchg_all[41]; merges = xchg_all[42]; nneg = xchg_all[43]; npos = xchg_all[44];
          __syncthreads();
        }
        SPROF(4 + 2 * sweep);
        if (sweep == 0) merges_asc = merges;
        // essential pair of the sweep   :110
        if (tid == 0) {
          const int bvx = sweep == 0 ? minv : maxv, dvx = sweep == 0 ? maxv : minv;
          if (a.poff) { const int64_t o = dpo + np; a.dkind[o] = sweep == 0 ? TLC_K_ESS : TLC_K_ESS_REV; a.dbv[o] = vid(bvx); a.ddv[o] = vid(dvx); a.dbirth[o] = fv[bvx]; a.ddeath[o] = fv[dvx]; }
          if (sweep == 0 && ((p.img_mask >> TLC_K_ESS) & 1u) && fv[dvx] > fv[bvx]) { pb[2 * npb] = fv[bvx]; pb[2 * npb + 1] = fv[dvx]; }
        }
        if (sweep == 0 && ((p.img_mask >> TLC_K_ESS) & 1u) && fv[maxv] > fv[minv]) npb++;
        np++;
        tm.sync();
        if (npb == PBUF) { flush_pairs<NT>(tm, pb, npb, img); npb = 0; }
        if (sweep == 0 && merges_asc != n - 1) { status = TLC_ST_DISCONNECTED; break; }  // assert len(components) == 1   riccidist2dgm.py:318
      }

      // ---------------- 6. loops: Accelerate_PD   accelerated_PD.py:115-178 ----------------
      if (status == TLC_ST_OK && ext) {
        if (nneg == 0) status = TLC_ST_NO_TREE_EDGES;  // list(Nodes)[0] -> IndexError   :122 (single-vertex vicinity)
        else {
          for (int x = tid; x < n; x += NT) { tpa[x] = (LID)x; stp[x] = 0xffff; tpr[x] = 0xffff; }
          tm.sync();
          // root the tree of the Neg edges at the first endpoint of the first Neg edge   :119-125
          const int root = (int)elo[negl[0]];
          // (tpr == 0xffff marks "not reached yet"; the root is reached from the start)
          if (tid == 0) tpr[root] = 0xfffe;
          tm.sync();
          for (int round = 0; round < n; round++) {
            bool ch = false;
            for (int i = tid; i < nneg; i += NT) {
              const int e = negl[i];
              const int xa = elo[e], xb = ehi[e];
              const bool ha = tpr[xa] != 0xffff, hb = tpr[xb] != 0xffff;
              if (ha && !hb) { tpa[xb] = (LID)xa; tpr[xb] = ark[e]; ch = true; }
              else if (hb && !ha) { tpa[xa] = (LID)xb; tpr[xa] = ark[e]; ch = true; }
            }
            tm.sync();
            if (!tm.any(ch)) break;
          }
          SPROF(7);
          // sequential sweep over the positive edges (sidx[0..npos) in sweep order) on the team's first lane; whenever the
          // pair buffer fills, the lane stops, the whole team rasterises the buffer, and the sweep resumes
          int k = 0, st_i = status;
          for (;;) {
            if (tid == 0) {
              while (k < npos && npb < PBUF) {
                const int pe = sidx[k];
                const int p0 = elo[pe], p1 = ehi[pe];
                int rc = ark[pe];
                // Loop = path_0 (p0 -> root) xor path_1 (p1 -> root) = (p0 -> lca) + (p1 -> lca)   :131-151.  The two climbs
                // alternate, each stamping its own mark, until one steps on the other's mark: ~2 x the cycle length
                // instead of the whole root path (the Neg trees of sparse vicinities are deep)
                const uint16_t mk0 = (uint16_t)(2 * k), mk1 = (uint16_t)(2 * k + 1);
                // every stamped vertex also keeps the largest parent-edge rank met below it on its side's climb (packed with
                // that edge's child end), so the cycle's maximum is known the moment the climbs meet -- no second walk
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
                const int by = (int)tpa[bc];  // large_edge = (bc, by)   :155-159
                const int la = min(bc, by), lb = max(bc, by);
                const int lvv = fv[la] >= fv[lb] ? la : lb;   // large_value = max(old[large_edge])
                const int lov = fv[p0] <= fv[p1] ? p0 : p1;   // low_value   = min(old[pos_edge])
                if (keep0 || fv[lvv] > fv[lov]) {  // :160-165 (KD :169-170: always)
                  if (a.poff) { const int64_t o = dpo + np; a.dkind[o] = TLC_K_ONE; a.dbv[o] = vid(lov); a.ddv[o] = vid(lvv); a.dbirth[o] = fv[lov]; a.ddeath[o] = fv[lvv]; }
                  np++;
                  if (((p.img_mask >> TLC_K_ONE) & 1u) && fv[lvv] > fv[lov]) { pb[2 * npb] = fv[lov]; pb[2 * npb + 1] = fv[lvv]; npb++; }
                }
                // change the parent   :168-176
                int node = in0 ? p0 : p1, nodec = in0 ? p1 : p0;
                for (;;) {
                  const int tp = (int)tpa[node], tr = tpr[node];
                  tpa[node] = (LID)nodec; tpr[node] = (uint16_t)rc;
                  if (node == bc) break;
                  nodec = node; rc = tr; node = tp;
                }
                k++;
              }
            }
            tm.bcast4(k, np, npb, st_i);
            if (npb == PBUF) { flush_pairs<NT>(tm, pb, npb, img); npb = 0; }
            if (k >= npos) break;
          }
        }
      }
    }
    tm.sync();
    SPROF(8);

    // ---------------- 7. image + outputs ----------------
    // (status, np, npb are uniform over the team here: every single-lane section ends with a broadcast)
    if (status <= TLC_ST_TRIVIAL && npb > 0) flush_pairs<NT>(tm, pb, npb, img);
    tm.sync();
    if (status == TLC_ST_OK && !roots_in) status = TLC_ST_TRIVIAL;
    if (tid < 25) {
      const double val = status <= TLC_ST_TRIVIAL ? img[tid] : 0.0;  // except BaseException: zeros   riccidist2dgm.py:356-357
      out[tid] = val;
      if (out32) out32[tid] = (float)val;
    }
    SPROF(9);
    if (tid == 0) {
      if (a.out_status) a.out_status[row] = status;
      if (a.out_n) a.out_n[row] = n;
      if (a.out_m) a.out_m[row] = m;
      if (a.dnp) a.dnp[row] = status <= TLC_ST_TRIVIAL || status == TLC_ST_NO_TREE_EDGES ? np : 0;
      if (a.stats) {
        atomicAdd(&a.stats->handled[a.cls], 1ull);
        if (live0) {
          // compulsory bytes B_e (SURVEY.md 8d): neighbour reads of both ball expansions and of the induced scan, rowptr
          // pairs, one f64 weight per induced directed edge, the fp32 image row
          const unsigned long long du = a.ball_acc ? a.ball_acc[2 * (size_t)u] + (node_mode ? 0ull : a.ball_acc[2 * (size_t)v]) : 0ull;
          const unsigned long long xu = a.ball_acc ? a.ball_acc[2 * (size_t)u + 1] + (node_mode ? 0ull : a.ball_acc[2 * (size_t)v + 1]) : 0ull;
          const double be = 4.0 * (double)(du + (unsigned long long)gpre_total) + 8.0 * (double)(xu + (unsigned long long)n) + 16.0 * (double)m + 100.0;
          atomicAdd(&a.stats->live, 1ull);
          atomicAdd(&a.stats->sum_n, (unsigned long long)n);
          atomicAdd(&a.stats->sum_m, (unsigned long long)m);
          atomicAdd(&a.stats->bytes, be);
        }
      }
    }
  }
}

// Rows class A deferred (64 < n <= 1024): count the induced adjacency entries and route each row to the class that can
// hold it -- B (n <= 256, <= 4096 entries), C (n <= 1024, <= 8192 entries) -- or to the staged pipeline's list.  With the
// sizes known up front the three run side by side (run_small) instead of B, then C, then the staged leftovers.
__global__ void __launch_bounds__(256) small_classify_kernel(SmallArgs a, int32_t* list_b2, int* count_b2, int32_t* list_c,
                                                             int* count_c) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(16) int32_t xchg_all[48];
  __shared__ int32_t vert[1024];
  __shared__ int s_entries;
  uint32_t* bm = reinterpret_cast<uint32_t*>(smem_raw);
  Team<256> tm{(int)threadIdx.x, xchg_all};
  const int tid = tm.tid, lane = tid & 31, wid = tid >> 5;
  const bool node_mode = a.p.mode == TLC_MODE_NODE;
  const int W = a.W;
  const int count = *a.list_count;
  for (int it = blockIdx.x; it < count; it += gridDim.x) {
    __syncthreads();
    const int32_t row = a.list[it];
    const int32_t u = a.targets[2 * (int64_t)row], v = a.targets[2 * (int64_t)row + 1];
    const uint32_t* __restrict__ bu = a.ball_cache + (size_t)u * W;
    const uint32_t* __restrict__ bv = a.ball_cache + (size_t)(node_mode ? u : v) * W;
    if (tid == 0) s_entries = 0;
    int n = 0;
    for (int w0 = 0; w0 < W; w0 += 256) {
      const int w = w0 + tid;
      uint32_t bits = 0;
      if (w < W) { bits = combine_balls(a.p.mode, bu[w], bv[w], w, u, v); bm[w] = bits; }
      int tot;
      const int pre = tm.exscan(__popc(bits), tot);
      if (n + tot <= 1024) {
        int k = n + pre;
        while (bits) { const int b = __ffs(bits) - 1; bits &= bits - 1; vert[k++] = w * 32 + b; }
      }
      n += tot;
    }
    __syncthreads();
    int cnt = 0;
    if (n <= 1024) {
      for (int i = wid; i < n; i += 8) {
        const int32_t x = vert[i];
        const int ra = a.g.rowptr[x], rb = a.g.rowptr[x + 1];
        for (int e = ra + lane; e < rb; e += 32) {
          const int32_t y = a.g.col[e];
          cnt += (bm[y >> 5] >> (y & 31)) & 1u;
        }
      }
      for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(FULLM, cnt, o);
      if (lane == 0 && cnt) atomicAdd(&s_entries, cnt);
    }
    __syncthreads();
    if (tid == 0) {
      const int d2 = s_entries;
      if (n <= 256 && d2 <= 4096) list_b2[atomicAdd(count_b2, 1)] = row;
      else if (n <= 1024 && d2 <= 8192) list_c[atomicAdd(count_c, 1)] = row;
      else a.big_list[atomicAdd(a.big_count, 1)] = row;
    }
  }
}

template <int NT, int NC, int AC>
static void launch_class(const SmallArgs& a, int grid, cudaStream_t st) {
  using M = SmallMem<NC, AC>;
  constexpr int TEAMS = NT == 32 ? 4 : 1;
  const size_t bytes = M::bytes * TEAMS;
  cudaFuncSetAttribute((const void*)small_kernel<NT, NC, AC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  cudaFuncSetAttribute((const void*)small_kernel<NT, NC, AC>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  small_kernel<NT, NC, AC><<<grid, NT == 32 ? 128 : NT, bytes, st>>>(a);
  count_launch();
}

}  // namespace

// class A: a warp per target (n <= 64, <= 256 induced edges); class B: a 128-thread CTA per target (n <= 256, <= 2048 edges);
// class C: a 256-thread CTA per target (n <= 1024, <= 4096 edges).
// counters[0] / [1] / [2]: rows deferred from A to B (list_b) / from B to C (list_c) / from C to the staged pipeline (list_b
// again: class B has consumed it by then); counters[3]: rows class A sends straight to the staged pipeline (list_big: more
// than 1024 vertices); counters[4]: rows of list_b2.  phases: 1 = class A (zeroes the counters), 2 = classes B then C.
void launch_small(const GraphView& g, const Params& p, const int32_t* targets, int64_t E, const VicinityScratch& vs,
                  double* out_pi, float* out_pi32, uint8_t* out_status, int32_t* list_b, int32_t* list_c, int32_t* list_big,
                  int* counters, int32_t* out_n, int32_t* out_m, const SmallDiag* diag, SmallStats* stats, int sm_count,
                  int phases, cudaStream_t st, int32_t* list_b2) {
  SmallArgs a{};
  a.stats = stats; a.ball_acc = vs.ball_acc;
#ifdef SMALL_PROFILE
  static unsigned long long* d_prof = nullptr;
  if (!d_prof) { cudaMalloc((void**)&d_prof, 48 * 8); cudaMemset(d_prof, 0, 48 * 8); }
  a.prof = d_prof;
  if (getenv("SMALL_PROFILE_DUMP") && (phases & 1)) {
    unsigned long long h[48];
    cudaMemcpy(h, d_prof, sizeof h, cudaMemcpyDeviceToHost);
    static const char* nm[10] = {"vicinity", "adjacency", "filtration", "sort_asc", "sweep_asc", "sort_desc", "sweep_desc", "tree_root", "loops", "image"};
    for (int c = 0; c < 3; c++) { fprintf(stderr, "[small profile] class %c:", 'A' + c); for (int i = 0; i < 10; i++) fprintf(stderr, " %s %.1fM", nm[i], h[c * 16 + i] / 1e6); fprintf(stderr, "\n"); }
    cudaMemset(d_prof, 0, 48 * 8);
  }
#endif
  a.g = g; a.p = p; a.targets = targets; a.E = E;
  a.ball_cache = vs.ball_cache; a.W = (g.N + 31) / 32;
  a.out_pi = out_pi; a.out_pi32 = out_pi32; a.out_status = out_status;
  a.out_n = out_n; a.out_m = out_m;
  if (diag) {
    a.poff = diag->poff; a.dnp = diag->np; a.dkind = diag->kind; a.dbv = diag->bv; a.ddv = diag->dv;
    a.dbirth = diag->birth; a.ddeath = diag->death; a.want_desc = diag->want_desc; a.graph_ids = diag->graph_ids;
  }
  if (phases & 1) {
    cudaMemsetAsync(counters, 0, 8 * sizeof(int), st);
    if (stats) cudaMemsetAsync(stats, 0, sizeof(SmallStats), st);
    // class A over every target
    a.cls = 0;
    a.list = nullptr; a.list_count = nullptr; a.defer_list = list_b; a.defer_count = counters;
    a.big_list = list_big; a.big_count = counters + 3; a.big_thresh = 1024;
    const int64_t want = (E + 3) / 4;
    const int grid = (int)std::min<int64_t>(want, (int64_t)sm_count * 16);
    launch_class<32, 64, 512>(a, std::max(grid, 1), st);
  }
  if (phases & 2) {
    a.big_list = nullptr; a.big_count = nullptr; a.big_thresh = 0;
    // class B over the rows class A deferred
    a.cls = 1;
    a.list = list_b; a.list_count = counters; a.defer_list = list_c; a.defer_count = counters + 1;
    {
      const int grid = (int)std::min<int64_t>(E, (int64_t)sm_count * 3);
      launch_class<128, 256, 4096>(a, std::max(grid, 1), st);
    }
    // class C over the rows class B deferred; what it cannot take either goes back into list_b for the staged pipeline
    a.cls = 2;
    a.list = list_c; a.list_count = counters + 1; a.defer_list = list_b; a.defer_count = counters + 2;
    {
      const int grid = (int)std::min<int64_t>(E, (int64_t)sm_count);
      launch_class<256, 1024, 8192>(a, std::max(grid, 1), st);
    }
  }
  // The side-by-side flow of run_small: 4 = route class A's deferred rows by their exact sizes (list_b -> list_b2 / list_c /
  // list_big), 8 = class B over list_b2, 16 = class C over list_c; what either still cannot take goes into list_b.
  if (phases & 4) {
    a.list = list_b; a.list_count = counters;
    a.big_list = list_big; a.big_count = counters + 3;
    const size_t bytes = (size_t)a.W * 4 + 16;
    cudaFuncSetAttribute((const void*)small_classify_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    const int grid = (int)std::min<int64_t>(E, (int64_t)sm_count * 4);
    small_classify_kernel<<<std::max(grid, 1), 256, bytes, st>>>(a, list_b2, counters + 4, list_c, counters + 1);
    count_launch();
  }
  if (phases & 8) {
    a.big_list = nullptr; a.big_count = nullptr; a.big_thresh = 0;
    a.cls = 1;
    a.list = list_b2; a.list_count = counters + 4; a.defer_list = list_b; a.defer_count = counters + 2;
    const int grid = (int)std::min<int64_t>(E, (int64_t)sm_count * 3);
    launch_class<128, 256, 4096>(a, std::max(grid, 1), st);
  }
  if (phases & 16) {
    a.big_list = nullptr; a.big_count = nullptr; a.big_thresh = 0;
    a.cls = 2;
    a.list = list_c; a.list_count = counters + 1; a.defer_list = list_b; a.defer_count = counters + 2;
    const int grid = (int)std::min<int64_t>(E, (int64_t)sm_count);
    launch_class<256, 1024, 8192>(a, std::max(grid, 1), st);
  }
}

}  // namespace tlc
