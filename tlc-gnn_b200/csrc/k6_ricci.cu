// k6_ricci.cu -- kernel 6: Ollivier-Ricci curvature of every edge, the step BEFORE the path (SURVEY.md row N4).
//
// Replaces compute_ricci_curvature (loaddatas.py:105-123):
//     OllivierRicci(Gd, alpha=0.5, method="Sinkhorn").compute_ricci_curvature()
// on the unweighted graph the reference builds (every edge weight 1).  The arithmetic of that call lives in two
// third-party packages (GraphRicciCurvature, POT) that are not part of the reference tree; their published algorithm is
// restated here and in oracle/ricci_oracle.py (PARITY UNPINNED, see that file):
//   * measure of a node x: (1 - alpha) / k on each of its k = min(deg, 3000) kept neighbours (equal weights e^-1,
//     normalised by their running sum), alpha on x itself; a heap of 3000 keeps the largest (weight, id): the largest ids;
//   * cost = hop distance between the two supports, 0..3 for the supports of an edge: 0 same node, 1 adjacent, 2 inside
//     each other's closed 2-hop ball, else 3 -- two bit tests against cached 1-hop / 2-hop ball bitmaps;
//   * Sinkhorn-Knopp on K = exp(cost / -0.1): v = b / (K^T u), u = 1 / ((K / a) v), marginal error every 10th iteration,
//     stop at 1e-9 or 1000 iterations, loss = sum(u K v * cost);  curvature = 1 - loss.
// One CTA per edge.  The cost matrix is kept as 2-bit-worth codes (one byte each) in shared memory when the two supports
// are small, in a per-CTA slab of HBM otherwise (a 3001 x 3001 matrix of two hubs is 9 MB); the four Gibbs factors come
// from the host's exp().  float64 throughout: K spans 14 orders of magnitude.
#include <algorithm>
#include <cmath>
#include <vector>

#include "tlc_common.cuh"

namespace tlc {
namespace {

struct RicciArgs {
  const int32_t* rowptr;
  const int32_t* col;
  const uint32_t* ball1;   // [N][W] closed 1-hop balls
  const uint32_t* ball2;   // [N][W] closed 2-hop balls
  int W;
  const int64_t* epos;     // [E] CSR position of the entry (x -> y), x < y
  const int64_t* emir;     // [E] position of the mirror entry (y -> x)
  const int32_t* esrc;     // [E] x
  int64_t E;
  double alpha;
  double kval[4];          // exp(d / -reg), d = 0 .. 3
  const double* wsum;      // [topk + 1] running sums of the neighbour weight e^-1 (python's sum(), left to right)
  double wnb;              // e^-1
  int topk, max_iter;
  double stop_thr;
  int cap;                 // support capacity of this launch (vectors in shared memory)
  int codes_smem;          // 1: the cap x cap code matrix is in shared memory too
  uint8_t* slab;           // per-CTA code matrix in HBM (codes_smem == 0)
  size_t slab_stride;
  double* out;             // [nnz]
  int32_t* iters;          // [nnz] or nullptr: Sinkhorn iterations spent
};

__device__ inline double block_sum(double v, double* red) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[w] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < nw; i++) t += red[i];
  __syncthreads();
  return t;
}

__global__ void __launch_bounds__(256) ricci_kernel(RicciArgs a) {
  extern __shared__ __align__(16) unsigned char rsm[];
  __shared__ double red[32];
  __shared__ int sflag;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  const int cap = a.cap;
  double* u = reinterpret_cast<double*>(rsm);       // [cap] each
  double* v = u + cap;
  double* up = v + cap;
  double* vp = up + cap;
  double* ma = vp + cap;                            // masses of the source support
  double* mb = ma + cap;                            // ... of the target support
  int32_t* su = reinterpret_cast<int32_t*>(mb + cap);  // support node ids
  int32_t* sv = su + cap;
  uint8_t* codes = a.codes_smem ? reinterpret_cast<uint8_t*>(sv + cap) : a.slab + (size_t)blockIdx.x * a.slab_stride;

  for (int64_t ei = blockIdx.x; ei < a.E; ei += gridDim.x) {
    __syncthreads();
    const int x = a.esrc[ei];
    const int64_t e = a.epos[ei];
    const int y = a.col[e];
    const int ax = a.rowptr[x], dx = a.rowptr[x + 1] - ax;
    const int ay = a.rowptr[y], dy = a.rowptr[y + 1] - ay;
    const int kx = min(dx, a.topk), ky = min(dy, a.topk);
    const int na = kx + 1, nb = ky + 1;
    // supports and masses: (1 - alpha) * w / sum(w) on the kept neighbours (largest ids), alpha on the node itself
    for (int i = tid; i < na; i += nt) {
      su[i] = i < kx ? a.col[ax + (dx - kx) + i] : x;
      ma[i] = i < kx ? (1.0 - a.alpha) * a.wnb / a.wsum[kx] : a.alpha;
      u[i] = 1.0 / (double)na;
    }
    for (int j = tid; j < nb; j += nt) {
      sv[j] = j < ky ? a.col[ay + (dy - ky) + j] : y;
      mb[j] = j < ky ? (1.0 - a.alpha) * a.wnb / a.wsum[ky] : a.alpha;
      v[j] = 1.0 / (double)nb;
    }
    __syncthreads();
    // hop costs between the supports: 0 same node, 1 adjacent, 2 within two hops, else 3
    for (int i = wid; i < na; i += nw) {
      const int an = su[i];
      const uint32_t* b1 = a.ball1 + (size_t)an * a.W;
      const uint32_t* b2 = a.ball2 + (size_t)an * a.W;
      for (int j = lane; j < nb; j += 32) {
        const int bn = sv[j];
        codes[(size_t)i * nb + j] = bn == an ? 0 : (test_bit(b1, bn) ? 1 : (test_bit(b2, bn) ? 2 : 3));
      }
    }
    __syncthreads();
    // Sinkhorn-Knopp (POT sinkhorn_knopp): K = exp(M / -reg), Kp = K / a
    int cpt = 0;
    double err = 1.0;
    while (err > a.stop_thr && cpt < a.max_iter) {
      if (tid == 0) sflag = 0;
      for (int i = tid; i < na; i += nt) up[i] = u[i];
      for (int j = tid; j < nb; j += nt) vp[j] = v[j];
      __syncthreads();
      // v = b / (K^T u)
      int bad = 0;
      for (int j = tid; j < nb; j += nt) {
        double s = 0.0;
        for (int i = 0; i < na; i++) s += a.kval[codes[(size_t)i * nb + j]] * up[i];
        if (s == 0.0) bad = 1;
        const double q = mb[j] / s;
        if (isnan(q) || isinf(q)) bad = 1;
        v[j] = q;
      }
      __syncthreads();
      // u = 1 / (Kp v)
      for (int i = wid; i < na; i += nw) {
        const double ia = 1.0 / ma[i];
        double s = 0.0;
        for (int j = lane; j < nb; j += 32) s += ia * a.kval[codes[(size_t)i * nb + j]] * v[j];
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) {
          const double q = 1.0 / s;
          if (isnan(q) || isinf(q)) bad = 1;
          u[i] = q;
        }
      }
      if (bad) sflag = 1;
      __syncthreads();
      if (sflag) {  // numerical errors: come back to the previous solution and quit the loop
        for (int i = tid; i < na; i += nt) u[i] = up[i];
        for (int j = tid; j < nb; j += nt) v[j] = vp[j];
        __syncthreads();
        break;
      }
      if (cpt % 10 == 0) {  // violation of the right marginal, every 10th iteration
        double part = 0.0;
        for (int j = tid; j < nb; j += nt) {
          double s = 0.0;
          for (int i = 0; i < na; i++) s += u[i] * a.kval[codes[(size_t)i * nb + j]];
          const double t2 = s * v[j] - mb[j];
          part += t2 * t2;
        }
        err = sqrt(block_sum(part, red));
      }
      cpt++;
    }
    // loss = sum(u K v * M)
    double part = 0.0;
    for (int i = wid; i < na; i += nw) {
      const double ui = u[i];
      for (int j = lane; j < nb; j += 32) {
        const int cde = codes[(size_t)i * nb + j];
        part += ui * a.kval[cde] * v[j] * (double)cde;
      }
    }
    const double loss = block_sum(part, red);
    if (tid == 0) {
      const double kappa = 1.0 - loss / 1.0;  // result = 1 - (m / weight(source, target))
      a.out[e] = kappa;
      a.out[a.emir[ei]] = kappa;
      if (a.iters) { a.iters[e] = cpt; a.iters[a.emir[ei]] = cpt; }
    }
  }
}

}  // namespace

// bytes of shared memory a launch with support capacity `cap` needs
static size_t ricci_smem(int cap, bool codes_smem) {
  return (size_t)cap * (6 * 8 + 2 * 4) + (codes_smem ? (size_t)cap * cap : 0) + 16;
}

// launches over a host-prepared edge list (device arrays); edges must satisfy max(support) <= cap
void launch_ricci(const int32_t* rowptr, const int32_t* col, const uint32_t* ball1, const uint32_t* ball2, int W,
                  const int64_t* epos, const int64_t* emir, const int32_t* esrc, int64_t E, double alpha, const double* kval4,
                  const double* wsum, double wnb, int topk, int max_iter, double stop_thr, int cap, bool codes_smem,
                  uint8_t* slab, size_t slab_stride, int grid, double* out, int32_t* iters, cudaStream_t st) {
  if (E <= 0) return;
  RicciArgs a{};
  a.rowptr = rowptr; a.col = col; a.ball1 = ball1; a.ball2 = ball2; a.W = W;
  a.epos = epos; a.emir = emir; a.esrc = esrc; a.E = E; a.alpha = alpha;
  for (int i = 0; i < 4; i++) a.kval[i] = kval4[i];
  a.wsum = wsum; a.wnb = wnb; a.topk = topk; a.max_iter = max_iter; a.stop_thr = stop_thr;
  a.cap = cap; a.codes_smem = codes_smem ? 1 : 0; a.slab = slab; a.slab_stride = slab_stride;
  a.out = out; a.iters = iters;
  const size_t bytes = ricci_smem(cap, codes_smem);
  cudaFuncSetAttribute((const void*)ricci_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  ricci_kernel<<<grid, 256, bytes, st>>>(a);
  count_launch();
}

size_t ricci_smem_bytes(int cap, bool codes_smem) { return ricci_smem(cap, codes_smem); }

}  // namespace tlc
