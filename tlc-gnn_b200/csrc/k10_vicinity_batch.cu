// k10_vicinity_batch.cu -- kernel 10: vicinities in graph-batch layout (tlc_vicinity_batch_dev), and the device-side check
// of a graph batch handed over in canonical form (tlc_graph_batch_create_dev).
//
// export : after kernel 1's fill, the filtration and kernel 1c's edge list, one CTA per target of the chunk writes its
//          vertex list, its edges (local ids + the target's first batch id) and its filtration values straight to their
//          final positions in TARGET order.  Those positions are the exclusive scans of the counting pass's n and m (kernel
//          7's scan), so no compaction pass follows.  The sweeps are skipped, so the CTA decides the connectivity test of
//          riccidist2dgm.py:318 itself: a union-find over the target's edges in the arena (hooking roots to the smaller
//          index with a compare-and-swap; the component count does not depend on the order of the hooks).
// check  : a thread per edge finds its graph by bisection in eoff and tests range, self-loop, orientation and strict
//          ascent against the previous edge of its graph; the smallest (edge, reason) key wins through atomicMin.
#include <algorithm>
#include <cmath>

#include "tlc_common.cuh"

namespace tlc {
namespace {

__device__ __forceinline__ int uf_find(volatile int32_t* par, int x) {
  int p = par[x];
  while (p != x) { x = p; p = par[x]; }
  return x;
}

__global__ void __launch_bounds__(256) vicinity_export_kernel(ChunkView c, const int64_t* __restrict__ voff,
                                                              const int64_t* __restrict__ eoff, int32_t* __restrict__ vert,
                                                              int32_t* __restrict__ ea, int32_t* __restrict__ eb,
                                                              double* __restrict__ fval, uint8_t* __restrict__ status,
                                                              int bad_desc) {
  __shared__ int32_t red[32];
  const int t = blockIdx.x;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int n = c.tn[t], m = c.tm[t];
  const int64_t row = c.tidx[t];
  const int64_t vo = voff[row], eo = eoff[row], cvo = c.voff[t], ceo = c.eoff[t];
  const int32_t* __restrict__ elo = c.elo + ceo;
  const int32_t* __restrict__ ehi = c.ehi + ceo;
  uint8_t st = c.tstatus[t];
  if (bad_desc) {
    st = TLC_ST_BAD_DESCRIPTOR;  // (the host has written the statuses)
  } else if (st <= TLC_ST_TRIVIAL && n > 1) {
    int32_t* par = c.vs1 + cvo;
    for (int x = tid; x < n; x += nt) par[x] = x;
    __syncthreads();
    for (int k = tid; k < m; k += nt) {
      int a = elo[k], b = ehi[k];
      for (;;) {
        a = uf_find(par, a);
        b = uf_find(par, b);
        if (a == b) break;
        const int lo = min(a, b), hi = max(a, b);
        if (atomicCAS(&par[hi], hi, lo) == hi) break;
      }
    }
    __syncthreads();
    int roots = 0;
    for (int x = tid; x < n; x += nt) roots += ((volatile int32_t*)par)[x] == x;
    roots = block_reduce_sum(roots, red);
    if (roots != 1) st = TLC_ST_DISCONNECTED;  // assert len(components) == 1   riccidist2dgm.py:318
    if (status && tid == 0) status[row] = st;
  } else if (status && tid == 0) {
    status[row] = st;
  }
  if (vert)
    for (int x = tid; x < n; x += nt) vert[vo + x] = c.vert[cvo + x];
  if (ea)
    for (int k = tid; k < m; k += nt) ea[eo + k] = (int32_t)(vo + elo[k]);
  if (eb)
    for (int k = tid; k < m; k += nt) eb[eo + k] = (int32_t)(vo + ehi[k]);
  if (fval) {
    const bool live = st <= TLC_ST_TRIVIAL;
    for (int x = tid; x < n; x += nt) fval[vo + x] = live ? c.fval[cvo + x] : __longlong_as_double(0x7ff8000000000000ll);
  }
}

__global__ void __launch_bounds__(256) batch_check_kernel(int64_t D, int64_t M, const int64_t* __restrict__ noff,
                                                          const int64_t* __restrict__ eoff, const int32_t* __restrict__ ea,
                                                          const int32_t* __restrict__ eb, unsigned long long* first) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < M; k += (int64_t)gridDim.x * blockDim.x) {
    int64_t lo = 0, hi = D;  // the graph t with eoff[t] <= k < eoff[t + 1]
    while (hi - lo > 1) {
      const int64_t mid = (lo + hi) >> 1;
      if (eoff[mid] <= k) lo = mid; else hi = mid;
    }
    const int64_t t = lo;
    const int64_t a = ea[k], b = eb[k];
    int reason = -1;
    if (a < noff[t] || a >= noff[t + 1] || b < noff[t] || b >= noff[t + 1]) reason = BATCH_BAD_RANGE;
    else if (a == b) reason = BATCH_BAD_LOOP;
    else if (a > b) reason = BATCH_BAD_ORIENT;
    else if (k > eoff[t]) {
      const int64_t pa = ea[k - 1], pb = eb[k - 1];
      if (pa > a || (pa == a && pb >= b)) reason = BATCH_BAD_ORDER;
    }
    if (reason >= 0) atomicMin(first, (unsigned long long)k * 4ull + (unsigned long long)reason);
  }
}

}  // namespace

void launch_vicinity_export(const ChunkView& c, const int64_t* voff, const int64_t* eoff, int32_t* vert, int32_t* ea,
                            int32_t* eb, double* fval, uint8_t* status, int bad_desc, cudaStream_t st) {
  if (c.T <= 0) return;
  vicinity_export_kernel<<<c.T, 256, 0, st>>>(c, voff, eoff, vert, ea, eb, fval, status, bad_desc);
  count_launch();
}

void launch_batch_check(int64_t D, int64_t M, const int64_t* noff, const int64_t* eoff, const int32_t* ea, const int32_t* eb,
                        unsigned long long* first, int sm_count, cudaStream_t st) {
  if (M <= 0 || D <= 0) return;
  const int grid = (int)std::min<int64_t>((M + 255) / 256, (int64_t)sm_count * 8);
  batch_check_kernel<<<grid, 256, 0, st>>>(D, M, noff, eoff, ea, eb, first);
  count_launch();
}

}  // namespace tlc
