// k7_diagrams.cu -- kernel 7: the persistence diagrams of a batch call (tlc_vicinity_diagrams).
//
// The stages leave every target's pairs in the chunk arena (ChunkView::pkind/pbv/pdv/pbirth/pdeath at poff(t), local
// vertex ids), kernel S in its own staging area.  Three small kernels turn them into one diagram array in target order:
//   export : after each chunk, its pairs are copied into the call's staging area at offsets the host fixed from the
//            chunk's pair counts, vertex ids mapped to graph ids (c.vert: written by kernel 1 on the materialised route and
//            by kernels 1b / 1t on the graph-row route), and the target's count / staging offset recorded at its row
//   scan   : exclusive offsets of the per-target counts in target order (one CTA, 64-bit)
//   gather : every target's segment from the staging area to its final place in the caller's arrays
// No atomics decide where a segment lands: the output, offsets included, is the same from run to run.
#include <algorithm>

#include "tlc_common.cuh"

namespace tlc {
namespace {

// a warp per target of the chunk
__global__ void __launch_bounds__(256) export_pairs_kernel(ChunkView c, const int64_t* __restrict__ dst,
                                                           const int64_t* __restrict__ rows, DiagArea area, int64_t area_base,
                                                           int32_t* __restrict__ np_out, int64_t* __restrict__ soff_out) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < c.T; t += nwarps) {
    const int64_t row = rows[t];
    if (row < 0) continue;  // (a target redone by a later sub-call)
    const int cnt = diag_pairs(c.tstatus[t], c.tnp[t]);
    const int64_t d = dst[t];
    if (lane == 0) { np_out[row] = cnt; soff_out[row] = d; }
    const int64_t po = c.poff((int)t);
    const int32_t* vert = c.vert + c.voff[t];
    for (int i = lane; i < cnt; i += 32) {
      const int64_t o = d - area_base + i;
      area.kind[o] = c.pkind[po + i];
      area.bv[o] = vert[c.pbv[po + i]];
      area.dv[o] = vert[c.pdv[po + i]];
      area.birth[o] = c.pbirth[po + i];
      area.death[o] = c.pdeath[po + i];
    }
  }
}

// poff[0..E] = exclusive scan of np[0..E): one CTA of 1024 threads, each a contiguous slice
__global__ void __launch_bounds__(1024) scan_counts_kernel(const int32_t* __restrict__ np, int64_t E, int64_t* __restrict__ poff) {
  __shared__ int64_t sh[1024];
  const int tid = threadIdx.x, nt = blockDim.x;
  const int64_t per = (E + nt - 1) / nt;
  const int64_t lo = min((int64_t)tid * per, E), hi = min(lo + per, E);
  int64_t s = 0;
  for (int64_t i = lo; i < hi; i++) s += np[i];
  sh[tid] = s;
  __syncthreads();
  for (int off = 1; off < nt; off <<= 1) {
    const int64_t v = tid >= off ? sh[tid - off] : 0;
    __syncthreads();
    sh[tid] += v;
    __syncthreads();
  }
  int64_t run = sh[tid] - s;
  for (int64_t i = lo; i < hi; i++) { poff[i] = run; run += np[i]; }
  if (tid == nt - 1) poff[E] = sh[nt - 1];
}

// a warp per target: staging offsets below split_at are in area a, the others in area b (at offset - split_at)
__global__ void __launch_bounds__(256) gather_pairs_kernel(const int32_t* __restrict__ np, const int64_t* __restrict__ soff,
                                                           const int64_t* __restrict__ poff, int64_t E, DiagArea a, DiagArea b,
                                                           int64_t split_at, DiagArea out) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < E; t += nwarps) {
    const int cnt = np[t];
    if (cnt == 0) continue;
    const int64_t s = soff[t], d = poff[t];
    const DiagArea& src = s < split_at ? a : b;
    const int64_t s0 = s < split_at ? s : s - split_at;
    for (int i = lane; i < cnt; i += 32) {
      if (out.kind) out.kind[d + i] = src.kind[s0 + i];
      if (out.bv) out.bv[d + i] = src.bv[s0 + i];
      if (out.dv) out.dv[d + i] = src.dv[s0 + i];
      if (out.birth) out.birth[d + i] = src.birth[s0 + i];
      if (out.death) out.death[d + i] = src.death[s0 + i];
    }
  }
}

int grid_for(int64_t warps, int sm_count) {
  return (int)std::max<int64_t>(1, std::min<int64_t>((warps + 7) / 8, (int64_t)sm_count * 16));
}

}  // namespace

void launch_export_pairs(const ChunkView& c, const int64_t* dst, const int64_t* rows, const DiagArea& area,
                         int64_t area_base, int32_t* np_out, int64_t* soff_out, int sm_count, cudaStream_t st) {
  if (c.T <= 0) return;
  export_pairs_kernel<<<grid_for(c.T, sm_count), 256, 0, st>>>(c, dst, rows, area, area_base, np_out, soff_out);
  count_launch();
}

void launch_scan_counts(const int32_t* np, int64_t E, int64_t* poff, cudaStream_t st) {
  scan_counts_kernel<<<1, 1024, 0, st>>>(np, E, poff);
  count_launch();
}

void launch_gather_pairs(const int32_t* np, const int64_t* soff, const int64_t* poff, int64_t E, const DiagArea& a,
                         const DiagArea& b, int64_t split_at, const DiagArea& out, int sm_count, cudaStream_t st) {
  if (E <= 0) return;
  gather_pairs_kernel<<<grid_for(E, sm_count), 256, 0, st>>>(np, soff, poff, E, a, b, split_at, out);
  count_launch();
}

}  // namespace tlc
