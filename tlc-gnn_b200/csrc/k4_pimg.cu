// k4_pimg.cu -- kernel 4: persistence-image splat, one CTA per diagram.
//
// Replaces PersistenceImager(resolution).transform(dgm, skew=True) (PersistenceImager.pyx:352-388,
// isotropic sigma = 1 branch) with linear_ramp weights (:9-30), the mesh of _create_mesh (:302-314) and
// _norm_cdf (:54-60).  The reference accumulates, per point, a (res+1)x(res+1) outer product of normal
// CDFs and a 4-term inclusion-exclusion (:385-388); algebraically that is the separable form
//     PI[i][j] = sum_k w_k * (Phi(b_{i+1}-beta_k) - Phi(b_i-beta_k)) * (Phi(p_{j+1}-pi_k) - Phi(p_j-pi_k))
// = Gx^T diag(w) Gy, which is what is evaluated here: 2(res+1) erfc + res^2 FMAs per point, float64
// throughout (contract: 1e-5 relative; measured ~1e-14 against the reference).  Points with weight 0
// (death <= birth: PD_down, [max,min], zero-persistence pairs) are skipped (SURVEY.md F6).
// Rows are written birth-major (riccidist2dgm.py:353 `.reshape(-1)`) straight into the caller's
// [E, res^2] table at the target's row; failed targets get a zero row and their status code.
#include "tlc_common.cuh"

namespace tlc {
namespace {

template <int RES>
__device__ __forceinline__ void splat_point(double birth, double death, double step, double* acc) {
  const double pers = death - birth;  // skew :366
  const double w = ramp_weight(pers);
  if (w == 0.0) return;
  double gb[RES > 0 ? RES : 1], gp[RES > 0 ? RES : 1];
  cdf_diffs(RES, step, birth, pers, gb, gp);
#pragma unroll
  for (int i = 0; i < RES; i++) {
    const double wb = w * gb[i];
#pragma unroll
    for (int j = 0; j < RES; j++) acc[i * RES + j] = fma(wb, gp[j], acc[i * RES + j]);
  }
}

// generic resolution: per-point partial sums go to shared memory with atomics (rare path)
__device__ void splat_point_generic(int res, double birth, double death, double step, double* simg) {
  const double pers = death - birth;
  const double w = ramp_weight(pers);
  if (w == 0.0) return;
  double gb[16], gp[16];
  cdf_diffs(res, step, birth, pers, gb, gp);
  for (int i = 0; i < res; i++)
    for (int j = 0; j < res; j++) atomicAdd(&simg[i * res + j], w * gb[i] * gp[j]);
}

template <int RES>
__device__ void block_image(const uint8_t* pkind, const double* pbirth, const double* pdeath, int64_t np,
                            uint32_t img_mask, int res, double* out, float* out32) {
  __shared__ double simg[256];
  __shared__ double wsum[32][RES > 0 ? RES * RES : 1];
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  const int r2 = res * res;
  // np.linspace(0, 1 + pixel, res + 1, endpoint=False)   PersistenceImager.pyx:311-314
  const double step = ((1.0 + 1.0 / res) - 0.0) / (res + 1);
  if constexpr (RES > 0) {
    double acc[RES > 0 ? RES * RES : 1];
#pragma unroll
    for (int i = 0; i < RES * RES; i++) acc[i] = 0.0;
    for (int64_t k = tid; k < np; k += nt)
      if (!pkind || ((img_mask >> pkind[k]) & 1u)) splat_point<RES>(pbirth[k], pdeath[k], step, acc);
#pragma unroll
    for (int i = 0; i < RES * RES; i++) {
      double v = acc[i];
      for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) wsum[wid][i] = v;
    }
    __syncthreads();
    for (int i = tid; i < r2; i += nt) {
      double v = 0.0;
      for (int w = 0; w < nw; w++) v += wsum[w][i];
      out[i] = v;
      if (out32) out32[i] = (float)v;
    }
  } else {
    for (int i = tid; i < r2; i += nt) simg[i] = 0.0;
    __syncthreads();
    for (int64_t k = tid; k < np; k += nt)
      if (!pkind || ((img_mask >> pkind[k]) & 1u)) splat_point_generic(res, pbirth[k], pdeath[k], step, simg);
    __syncthreads();
    for (int i = tid; i < r2; i += nt) {
      out[i] = simg[i];
      if (out32) out32[i] = (float)simg[i];
    }
  }
}

template <int RES>
__global__ void pimg_kernel(Params p, ChunkView c, double* out_pi, float* out_pi_f32, uint8_t* out_status) {
  const int t = blockIdx.x;
  const int64_t row = c.tidx[t];
  const int r2 = p.resolution * p.resolution;
  const uint8_t st = c.tstatus[t];
  double* out = out_pi + row * r2;
  float* out32 = out_pi_f32 ? out_pi_f32 + row * r2 : nullptr;
  if (threadIdx.x == 0 && out_status) out_status[row] = st;
  if (st > TLC_ST_TRIVIAL || c.tn[t] == 0) {  // except BaseException: zeros   riccidist2dgm.py:356-357
    for (int i = threadIdx.x; i < r2; i += blockDim.x) { out[i] = 0.0; if (out32) out32[i] = 0.f; }
    return;
  }
  const int64_t po = c.poff(t);
  block_image<RES>(c.pkind + po, c.pbirth + po, c.pdeath + po, c.tnp[t], p.img_mask, p.resolution, out, out32);
}

template <int RES>
__global__ void pimg_single_kernel(const double* dgm, int64_t K, int res, double* out) {
  // dgm is [K][2] interleaved: stage through de-interleaving pointers is not possible, so splat directly
  __shared__ double simg[256];
  const int tid = threadIdx.x, nt = blockDim.x;
  const int r2 = res * res;
  const double step = ((1.0 + 1.0 / res) - 0.0) / (res + 1);
  for (int i = tid; i < r2; i += nt) simg[i] = 0.0;
  __syncthreads();
  if constexpr (RES > 0) {
    double acc[RES > 0 ? RES * RES : 1];
#pragma unroll
    for (int i = 0; i < RES * RES; i++) acc[i] = 0.0;
    for (int64_t k = tid; k < K; k += nt) splat_point<RES>(dgm[2 * k], dgm[2 * k + 1], step, acc);
#pragma unroll
    for (int i = 0; i < RES * RES; i++) {
      double v = acc[i];
      for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if ((tid & 31) == 0) atomicAdd(&simg[i], v);
    }
  } else {
    for (int64_t k = tid; k < K; k += nt) splat_point_generic(res, dgm[2 * k], dgm[2 * k + 1], step, simg);
  }
  __syncthreads();
  for (int i = tid; i < r2; i += nt) out[i] = simg[i];
}

}  // namespace

void launch_pimg(const Params& p, const ChunkView& c, double* out_pi, float* out_pi_f32, uint8_t* out_status,
                 int block, cudaStream_t st) {
  if (p.resolution == 5) pimg_kernel<5><<<c.T, block, 0, st>>>(p, c, out_pi, out_pi_f32, out_status);
  else pimg_kernel<0><<<c.T, block, 0, st>>>(p, c, out_pi, out_pi_f32, out_status);
  count_launch();
}

void launch_pimg_single(const double* dgm, int64_t K, int res, double* out, cudaStream_t st) {
  const int block = K >= 4096 ? 256 : 64;
  if (res == 5) pimg_single_kernel<5><<<1, block, 0, st>>>(dgm, K, res, out);
  else pimg_single_kernel<0><<<1, block, 0, st>>>(dgm, K, res, out);
  count_launch();
}

}  // namespace tlc
