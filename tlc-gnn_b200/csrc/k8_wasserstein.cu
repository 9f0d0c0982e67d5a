// k8_wasserstein.cu -- kernel 8: exact Wasserstein distances between pairs of device-resident persistence diagrams, and
// their gradient.
//
// Pair t compares X = points poff_x[t] .. poff_x[t+1] with Y = points poff_y[t] .. poff_y[t+1] (selected by kind, as
// the batch imager selects them).  The distance is gudhi's wasserstein_distance(X, Y, order=q, internal_p=p), the loss
// of Knowledge_Distillation/wasserstein.py (:93, :198): the minimum over partial matchings of
//     W = (sum c)^(1/q),  c = ||x - y||_p^q for a matched pair,  c = delta(x)^q for a point matched to the diagonal,
// delta(x) = |d - b| * 2^(1/p - 1).  gudhi states it as an (n+1) x (m+1) transport problem; the same optimum is the
// square assignment problem of size N = n' + m' solved here (n', m': the selected points with b != d):
//   rows    = the n' X points, then m' diagonal slots;
//   columns = the m' Y points, then n' diagonal slots;
//   cost(x, y) = ||x - y||_p^q,  cost(x, slot) = delta(x)^q,  cost(slot, y) = delta(y)^q,  cost(slot, slot) = 0.
// Points with b == d are matched to the diagonal without entering the problem: delta(x) = 0 there and
// delta(y) <= ||x - y||_p for any y, so some optimum matches them so.  Costs are computed from the two points when
// needed; no cost matrix is stored.
//
// Solver: one CTA per pair runs the shortest-augmenting-path algorithm with dual potentials (Jonker-Volgenant; the
// form of scipy.optimize.linear_sum_assignment, Crouse 2016).  Row r = 0 .. N-1 is added in turn by a Dijkstra search
// over reduced costs; each search step scans one column, so a search takes at most N steps, and the augmentation walks
// back at most N columns.  Every loop's trip count is bounded by N alone: N augmentations of at most N steps of O(N)
// work each, O(N^3) in the worst case.  A step is one pass over the unscanned columns (thread j % THREADS owns column
// j and is the only thread that reads or writes its search state) and one block reduction to the minimum label.
// Ties go to a free column, then to the lowest column index (scipy prefers free columns as well), so the matching and
// the distance -- the matched costs summed by row -- are the same bits from call to call and whatever the batch.
// A pair with a selected non-finite coordinate, a search that meets no finite label (costs that overflow), or a
// workspace slice outside the workspace is not solved: its distance is NaN and all its matches are -1.
//
// Gradient: a thread per point.  With S = W^q and G = grad_out[t], a point's gradient is
//   G (1/q) S^(1/q - 1) dc/d(b, d) = G (n / W)^(q-1) dn/d(b, d)   (n = ||x - y||_p, or delta for the diagonal),
// with torch's conventions for torch.linalg.vector_norm: dn/de = 0 at n = 0, sgn(0) = 0, and for p = inf the
// gradient is split evenly among the coordinates that tie for the max.  W = 0 gives 0; an unsolved pair gives NaN.
#include <math_constants.h>

#include "tlc_common.cuh"

namespace tlc {
namespace {

constexpr int WS_THREADS = 256;  // forward CTA: one per pair
constexpr int WS_WARPS = WS_THREADS / 32;
constexpr int WG_THREADS = 128;  // backward CTA: one per pair, one thread per point

// p and q with their cheap special cases decided once per call (uniform across the grid: no divergence)
struct Metric {
  double p, q, kappa;  // kappa = 2^(1/p - 1): delta(x) = |d - b| * kappa
  int pk, qk;          // pk: 0 inf, 1 one, 2 two, 3 other; qk: 1 one, 2 two, 3 other
};

__device__ __forceinline__ double ground(const Metric& M, double eb, double ed) {
  const double a = fabs(eb), b = fabs(ed);
  switch (M.pk) {
    case 0: return fmax(a, b);
    case 1: return a + b;
    case 2: return sqrt(a * a + b * b);
    default: return pow(pow(a, M.p) + pow(b, M.p), 1.0 / M.p);
  }
}

__device__ __forceinline__ double powq(const Metric& M, double n) {
  return M.qk == 1 ? n : M.qk == 2 ? n * n : pow(n, M.q);
}

__device__ __forceinline__ double diag_cost(const Metric& M, double2 x) { return powq(M, fabs(x.y - x.x) * M.kappa); }

__device__ __forceinline__ bool selected(const uint8_t* kind, uint32_t mask, int64_t k) {
  return !kind || (kind[k] < 32 && ((mask >> kind[k]) & 1u));
}

// The pair's slice of the workspace: n = nx, m = ny raw segment lengths (bounds on n', m'), N = n + m.
// 62 N bytes of the 64 N reserved per point; every array is naturally aligned.
struct Slice {
  double2 *xp, *yp;  // compacted (birth, death) of the selected nonzero-persistence points
  int64_t *xi, *yi;  // their global indices
  double *u, *v, *spc;
  int *col4row, *row4col, *path;
  uint8_t *sr, *sc;  // row scanned, column scanned
  __device__ Slice(unsigned char* w, int64_t n, int64_t m) {
    const int64_t N = n + m;
    xp = (double2*)w;
    yp = (double2*)(w + 16 * n);
    xi = (int64_t*)(w + 16 * N);
    yi = (int64_t*)(w + 16 * N + 8 * n);
    u = (double*)(w + 24 * N);
    v = (double*)(w + 32 * N);
    spc = (double*)(w + 40 * N);
    col4row = (int*)(w + 48 * N);
    row4col = (int*)(w + 52 * N);
    path = (int*)(w + 56 * N);
    sr = w + 60 * N;
    sc = w + 61 * N;
  }
};

// Order-preserving compaction of one side's selected nonzero-persistence points into (pts, idx); writes the match of
// every other point (-2 masked out, -1 zero persistence).  Returns the count; *bad |= a selected non-finite point.
__device__ int compact_side(const double* birth, const double* death, const uint8_t* kind, uint32_t mask, int64_t lo,
                            int64_t hi, double2* pts, int64_t* idx, int64_t* match, int* s_cnt, int* bad) {
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  int total = 0, nonfinite = 0;
  for (int64_t c = lo; c < hi; c += WS_THREADS) {
    const int64_t k = c + tid;
    bool keep = false;
    double2 x = make_double2(0.0, 0.0);
    if (k < hi) {
      if (!selected(kind, mask, k)) {
        if (match) match[k] = -2;
      } else {
        x = make_double2(birth[k], death[k]);
        if (!isfinite(x.x) || !isfinite(x.y)) nonfinite = 1;
        keep = x.x != x.y;
        if (!keep && match) match[k] = -1;
      }
    }
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) s_cnt[wid] = __popc(bal);
    __syncthreads();
    int base = total;
    for (int w = 0; w < wid; w++) base += s_cnt[w];
    for (int w = 0; w < WS_WARPS; w++) total += s_cnt[w];
    if (keep) {
      const int at = base + __popc(bal & ((1u << lane) - 1u));
      pts[at] = x;
      idx[at] = k;
    }
    __syncthreads();
  }
  if (__syncthreads_or(nonfinite)) *bad = 1;
  return total;
}

__global__ void __launch_bounds__(WS_THREADS) wasserstein_kernel(
    const int64_t* poff_x, const double* bx, const double* dx, const uint8_t* kx, const int64_t* poff_y,
    const double* by, const double* dy, const uint8_t* ky, uint32_t mask, Metric M, unsigned char* ws,
    uint64_t ws_bytes, double* dist, int64_t* match_x, int64_t* match_y) {
  __shared__ double s_val[2][WS_WARPS];
  __shared__ int s_key[2][WS_WARPS];
  __shared__ int s_cnt[WS_WARPS];
  __shared__ int s_bad;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int64_t t = blockIdx.x;
  const int64_t lo_x = poff_x[t], hi_x = max(poff_x[t + 1], lo_x), lo_y = poff_y[t], hi_y = max(poff_y[t + 1], lo_y);
  const int64_t n = hi_x - lo_x, m = hi_y - lo_y, rel_x = lo_x - poff_x[0], rel_y = lo_y - poff_y[0];
  if (tid == 0) s_bad = 0;
  __syncthreads();
  // the slice must lie in the workspace (it does whenever poff is non-decreasing and the size is the query's)
  const bool fits = rel_x >= 0 && rel_y >= 0 && n + m < ((int64_t)1 << 30) &&
                    (uint64_t)(64 * (rel_x + rel_y + n + m)) <= ws_bytes;
  int nx = 0, ny = 0;
  Slice S(ws + (fits ? 64 * (rel_x + rel_y) : 0), fits ? n : 0, fits ? m : 0);
  if (fits) {
    nx = compact_side(bx, dx, kx, mask, lo_x, hi_x, S.xp, S.xi, match_x, s_cnt, &s_bad);
    ny = compact_side(by, dy, ky, mask, lo_y, hi_y, S.yp, S.yi, match_y, s_cnt, &s_bad);
  }
  const int N = nx + ny;
  __syncthreads();
  bool ok = fits && !s_bad;
  if (ok) {
    for (int i = tid; i < N; i += WS_THREADS) {
      S.u[i] = 0.0; S.v[i] = 0.0;
      S.col4row[i] = -1; S.row4col[i] = -1;
    }
    __syncthreads();
    // N augmentations; row r enters the matching in the r-th
    for (int r = 0; r < N && ok; r++) {
      for (int j = tid; j < N; j += WS_THREADS) { S.spc[j] = CUDART_INF; S.sc[j] = 0; S.sr[j] = 0; }
      __syncthreads();
      double minv = 0.0;
      int i = r, sink = -1;
      // at most N steps: each scans a new column
      for (int step = 0; step < N; step++) {
        if (tid == 0) S.sr[i] = 1;
        const double ui = S.u[i];
        const bool xrow = i < nx;
        const double2 x = xrow ? S.xp[i] : make_double2(0.0, 0.0);
        const double cx = xrow ? diag_cost(M, x) : 0.0;  // to any diagonal slot
        double best = CUDART_INF;
        int bkey = 0x7fffffff;
        for (int j = tid; j < N; j += WS_THREADS) {
          if (S.sc[j]) continue;
          double c;
          if (j < ny) {
            const double2 y = S.yp[j];
            c = xrow ? powq(M, ground(M, x.x - y.x, x.y - y.y)) : diag_cost(M, y);
          } else {
            c = cx;
          }
          const double rc = minv + c - ui - S.v[j];
          double lab = S.spc[j];
          if (rc < lab) { lab = rc; S.spc[j] = rc; S.path[j] = i; }
          const int key = (S.row4col[j] >= 0 ? 0x40000000 : 0) | j;  // free columns first, then the lowest index
          if (lab < best || (lab == best && key < bkey)) { best = lab; bkey = key; }
        }
        for (int o = 16; o; o >>= 1) {
          const double ob = __shfl_xor_sync(0xffffffffu, best, o);
          const int ok2 = __shfl_xor_sync(0xffffffffu, bkey, o);
          if (ob < best || (ob == best && ok2 < bkey)) { best = ob; bkey = ok2; }
        }
        const int buf = step & 1;  // double-buffered: one barrier per step
        if (lane == 0) { s_val[buf][wid] = best; s_key[buf][wid] = bkey; }
        __syncthreads();
        best = s_val[buf][0]; bkey = s_key[buf][0];
        for (int w = 1; w < WS_WARPS; w++) {
          const double ob = s_val[buf][w];
          const int ok2 = s_key[buf][w];
          if (ob < best || (ob == best && ok2 < bkey)) { best = ob; bkey = ok2; }
        }
        if (!(best < CUDART_INF)) break;  // no finite label: the costs overflowed
        minv = best;
        const int j = bkey & 0x3fffffff;
        if (j % WS_THREADS == tid) S.sc[j] = 1;
        if (!(bkey & 0x40000000)) { sink = j; break; }
        i = S.row4col[j];
      }
      __syncthreads();
      if (sink < 0) { ok = false; break; }  // uniform: every thread saw the same reductions
      // dual update of the scanned rows and columns, then the augmentation along path[]
      for (int k = tid; k < N; k += WS_THREADS) {
        if (S.sr[k]) S.u[k] += k == r ? minv : minv - S.spc[S.col4row[k]];
        if (S.sc[k]) S.v[k] -= minv - S.spc[k];
      }
      __syncthreads();
      if (tid == 0) {
        int j = sink;
        for (int s = 0; s < N; s++) {  // at most N columns on the path
          const int pi = S.path[j];
          S.row4col[j] = pi;
          const int nj = S.col4row[pi];
          S.col4row[pi] = j;
          j = nj;
          if (pi == r) break;
        }
      }
      __syncthreads();
    }
  }
  if (!ok) {
    if (tid == 0) dist[t] = CUDART_NAN;
    for (int64_t k = lo_x + tid; k < hi_x && match_x; k += WS_THREADS) match_x[k] = -1;
    for (int64_t k = lo_y + tid; k < hi_y && match_y; k += WS_THREADS) match_y[k] = -1;
    return;
  }
  if (match_x)
    for (int i = tid; i < nx; i += WS_THREADS) {
      const int j = S.col4row[i];
      match_x[S.xi[i]] = j < ny ? S.yi[j] : -1;
    }
  if (match_y)
    for (int j = tid; j < ny; j += WS_THREADS) {
      const int i = S.row4col[j];
      match_y[S.yi[j]] = i < nx ? S.xi[i] : -1;
    }
  if (tid == 0) {  // the matched costs in row order
    double s = 0.0;
    for (int i = 0; i < N; i++) {
      const int j = S.col4row[i];
      if (i < nx) {
        const double2 x = S.xp[i];
        if (j < ny) {
          const double2 y = S.yp[j];
          s += powq(M, ground(M, x.x - y.x, x.y - y.y));
        } else {
          s += diag_cost(M, x);
        }
      } else if (j < ny) {
        s += diag_cost(M, S.yp[j]);
      }
    }
    dist[t] = M.qk == 1 ? s : pow(s, 1.0 / M.q);
  }
}

// dn/d(e_b, e_d) of n = ||e||_p with torch's vector_norm conventions (0 at n = 0, sgn(0) = 0, p = inf ties split evenly)
__device__ void ground_grad(const Metric& M, double eb, double ed, double n, double* gb, double* gd) {
  const double sb = (eb > 0.0) - (eb < 0.0), sd = (ed > 0.0) - (ed < 0.0);
  if (M.pk == 1) { *gb = sb; *gd = sd; return; }
  if (n == 0.0) { *gb = 0.0; *gd = 0.0; return; }
  const double a = fabs(eb), b = fabs(ed);
  switch (M.pk) {
    case 0: {
      const double wa = a == n ? 1.0 : 0.0, wb = b == n ? 1.0 : 0.0, cnt = wa + wb;
      *gb = sb * wa / cnt; *gd = sd * wb / cnt;
      return;
    }
    case 2: *gb = eb / n; *gd = ed / n; return;
    default: {
      const double den = pow(n, M.p - 1.0);
      *gb = sb * pow(a, M.p - 1.0) / den; *gd = sd * pow(b, M.p - 1.0) / den;
    }
  }
}

// One side's gradient: the points of [lo, hi) of (birth, death), matched through `match` to the other side's points.
// `sign` is +1 for X (e = x - y) and -1 for Y (e = x - y differentiated in y).
__device__ void side_grad(const Metric& M, double G, double W, const double* birth, const double* death,
                          const uint8_t* kind, uint32_t mask, int64_t lo, int64_t hi, const int64_t* match,
                          const double* ob, const double* od, double sign, double* grad_birth, double* grad_death) {
  for (int64_t k = lo + threadIdx.x; k < hi; k += WG_THREADS) {
    double gb = 0.0, gd = 0.0;
    if (selected(kind, mask, k)) {
      if (W != W) {
        gb = gd = CUDART_NAN;
      } else if (W != 0.0) {
        const double b = birth[k], d = death[k];
        const int64_t o = match[k];
        double n, db, dd;
        if (o < 0) {  // the diagonal: n = |d - b| kappa
          const double s = (d > b) - (d < b);
          n = fabs(d - b) * M.kappa;
          db = -s * M.kappa;
          dd = s * M.kappa;
        } else {
          const double eb = sign * (b - ob[o]), ed = sign * (d - od[o]);
          n = ground(M, eb, ed);
          ground_grad(M, eb, ed, n, &db, &dd);
          db *= sign;
          dd *= sign;
        }
        const double f = M.qk == 1 ? G : G * pow(n / W, M.q - 1.0);  // G (n / W)^(q-1)
        gb = f * db;
        gd = f * dd;
      }
    }
    if (grad_birth) grad_birth[k] = gb;
    if (grad_death) grad_death[k] = gd;
  }
}

__global__ void __launch_bounds__(WG_THREADS) wasserstein_grad_kernel(
    const int64_t* poff_x, const double* bx, const double* dx, const uint8_t* kx, const int64_t* poff_y,
    const double* by, const double* dy, const uint8_t* ky, uint32_t mask, Metric M, const double* dist,
    const int64_t* match_x, const int64_t* match_y, const double* grad_out, double* gbx, double* gdx, double* gby,
    double* gdy) {
  const int64_t t = blockIdx.x;
  const int64_t lo_x = poff_x[t], hi_x = max(poff_x[t + 1], lo_x), lo_y = poff_y[t], hi_y = max(poff_y[t + 1], lo_y);
  const double G = grad_out[t], W = dist[t];
  if (gbx || gdx) side_grad(M, G, W, bx, dx, kx, mask, lo_x, hi_x, match_x, by, dy, 1.0, gbx, gdx);
  if (gby || gdy) side_grad(M, G, W, by, dy, ky, mask, lo_y, hi_y, match_y, bx, dx, -1.0, gby, gdy);
}

Metric make_metric(double order, double internal_p) {
  Metric M;
  M.p = internal_p;
  M.q = order;
  M.pk = isinf(internal_p) ? 0 : internal_p == 1.0 ? 1 : internal_p == 2.0 ? 2 : 3;
  M.qk = order == 1.0 ? 1 : order == 2.0 ? 2 : 3;
  M.kappa = M.pk == 0 ? 0.5 : std::exp2(1.0 / internal_p - 1.0);
  return M;
}

}  // namespace

uint64_t wasserstein_workspace_bytes(int64_t D, int64_t Px, int64_t Py) {
  (void)D;
  return 64ull * (uint64_t)(Px + Py);
}

void launch_wasserstein(const int64_t* poff_x, const double* bx, const double* dx, const uint8_t* kx,
                        const int64_t* poff_y, const double* by, const double* dy, const uint8_t* ky, uint32_t mask,
                        double order, double internal_p, int64_t D, void* ws, uint64_t ws_bytes, double* dist,
                        int64_t* match_x, int64_t* match_y, cudaStream_t st) {
  wasserstein_kernel<<<(unsigned)D, WS_THREADS, 0, st>>>(poff_x, bx, dx, kx, poff_y, by, dy, ky, mask,
                                                         make_metric(order, internal_p), (unsigned char*)ws, ws_bytes,
                                                         dist, match_x, match_y);
  count_launch();
}

void launch_wasserstein_grad(const int64_t* poff_x, const double* bx, const double* dx, const uint8_t* kx,
                             const int64_t* poff_y, const double* by, const double* dy, const uint8_t* ky,
                             uint32_t mask, double order, double internal_p, int64_t D, const double* dist,
                             const int64_t* match_x, const int64_t* match_y, const double* grad_out, double* gbx,
                             double* gdx, double* gby, double* gdy, cudaStream_t st) {
  wasserstein_grad_kernel<<<(unsigned)D, WG_THREADS, 0, st>>>(poff_x, bx, dx, kx, poff_y, by, dy, ky, mask,
                                                              make_metric(order, internal_p), dist, match_x, match_y,
                                                              grad_out, gbx, gdx, gby, gdy);
  count_launch();
}

}  // namespace tlc
