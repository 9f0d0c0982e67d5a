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
// The same image of diagrams the caller holds on the device, and its gradient, is the batch imager below
// (tlc_pimg_batch_dev / tlc_pimg_batch_grad_dev; tlc_pimg_transform is its one-diagram host call).
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

// ---- the batch imager of device-resident diagrams (tlc_pimg_batch_dev / tlc_pimg_batch_grad_dev) ----
// Diagram t is points poff[t] .. poff[t+1] of birth[] / death[]; a decreasing segment is empty.  A point counts when
// kind is NULL or its kind is < 32 with bit `kind` of img_mask set.
constexpr int PB_THREADS = 256;              // forward CTA: one per diagram
constexpr int PB_CHUNK = PB_THREADS / 2;     // points staged per pass: one thread per (point, axis)
constexpr int PB_LD = 17;                    // row stride of the staged vectors (odd: no bank conflicts)
constexpr int PG_THREADS = 128;              // backward CTA: one per diagram, one thread per point

__device__ __forceinline__ bool point_counts(const uint8_t* kind, uint32_t img_mask, int64_t k) {
  return !kind || (kind[k] < 32 && ((img_mask >> kind[k]) & 1u));
}

// Forward.  Per pass, the chunk's w * A_i(birth) and B_j(pers) vectors (res + 1 erfc each, as cdf_diffs) are staged in
// shared memory; thread (group g, pixel p) then sums the products of the points g, g + G, ... of the chunk, G = 256 / res^2
// groups, and the groups' partial sums are added in group order.  The order of every sum depends on res alone: a row
// is the same bits whatever the batch around it, and no atomics are involved.
__global__ void __launch_bounds__(PB_THREADS) pimg_batch_kernel(const int64_t* poff, const double* birth,
                                                                const double* death, const uint8_t* kind,
                                                                uint32_t img_mask, int res, double* out) {
  __shared__ double sa[PB_CHUNK * PB_LD], sb[PB_CHUNK * PB_LD];
  const int64_t t = blockIdx.x, k0 = poff[t], k1 = poff[t + 1];
  const int tid = threadIdx.x, r2 = res * res, groups = PB_THREADS / r2;
  const int grp = tid / r2, pix = tid % r2, pi = pix / res, pj = pix % res;
  const int q = tid % PB_CHUNK;
  const bool pers_axis = tid >= PB_CHUNK;
  const double step = ((1.0 + 1.0 / res) - 0.0) / (res + 1);  // PersistenceImager.pyx:311-314
  double acc = 0.0;
  for (int64_t c = k0; c < k1; c += PB_CHUNK) {
    const int n = k1 - c < PB_CHUNK ? (int)(k1 - c) : PB_CHUNK;
    if (q < n) {
      const int64_t k = c + q;
      const double b = birth[k], pers = death[k] - b;  // skew :366
      const double w = point_counts(kind, img_mask, k) ? ramp_weight(pers) : 0.0;
      double* row = (pers_axis ? sb : sa) + q * PB_LD;
      if (w == 0.0) {
        for (int i = 0; i < res; i++) row[i] = 0.0;
      } else {
        const double x = pers_axis ? pers : b, scale = pers_axis ? 1.0 : w;
        double prev = norm_cdf(0.0 - x);
        for (int i = 1; i <= res; i++) {
          const double cur = norm_cdf(i * step - x);
          row[i - 1] = scale * (cur - prev);
          prev = cur;
        }
      }
    }
    __syncthreads();
    if (grp < groups)
      for (int m = grp; m < n; m += groups) acc = fma(sa[m * PB_LD + pi], sb[m * PB_LD + pj], acc);
    __syncthreads();
  }
  if (grp < groups) sa[grp * r2 + pix] = acc;
  __syncthreads();
  if (tid < r2) {
    double v = 0.0;
    for (int g = 0; g < groups; g++) v += sa[g * r2 + tid];
    out[t * r2 + tid] = v;
  }
}

// Backward.  For a point of diagram t with p = death - birth, G = grad_out[t], w = clamp(p, 0, 1), w' = 1 on [0, 1]:
//   grad_death = A^T G (w' B + w B'),   grad_birth = w A'^T G B - grad_death
// A'_i = phi(x_i - b) - phi(x_{i+1} - b) and B'_j likewise are the derivatives of A_i(b) and B_j(p).  G is staged in
// shared memory; each thread keeps its point's B and B' in its own shared column and walks the birth axis.  Points at
// p = 0 are not skipped: w = 0 there but w' = 1.
__global__ void __launch_bounds__(PG_THREADS) pimg_batch_grad_kernel(const int64_t* poff, const double* birth,
                                                                     const double* death, const uint8_t* kind,
                                                                     uint32_t img_mask, int res, const double* grad_out,
                                                                     double* grad_birth, double* grad_death) {
  __shared__ double sg[256];
  __shared__ double sB[16 * PG_THREADS], sdB[16 * PG_THREADS];
  const int64_t t = blockIdx.x, k0 = poff[t], k1 = poff[t + 1];
  const int tid = threadIdx.x, r2 = res * res;
  for (int i = tid; i < r2; i += PG_THREADS) sg[i] = grad_out[t * r2 + i];
  __syncthreads();
  const double step = ((1.0 + 1.0 / res) - 0.0) / (res + 1);
  double* B = sB + tid;
  double* dB = sdB + tid;
  for (int64_t k = k0 + tid; k < k1; k += PG_THREADS) {
    double gd = 0.0, gb = 0.0;
    const double b = birth[k], pers = death[k] - b;
    if (point_counts(kind, img_mask, k) && !(pers < 0.0)) {  // p < 0: w = w' = 0
      const double w = ramp_weight(pers), wp = (pers >= 0.0 && pers <= 1.0) ? 1.0 : 0.0;
      double cprev = norm_cdf(0.0 - pers), fprev = norm_pdf(0.0 - pers);
      for (int j = 1; j <= res; j++) {
        const double x = j * step - pers, c = norm_cdf(x), f = norm_pdf(x);
        B[(j - 1) * PG_THREADS] = c - cprev;
        dB[(j - 1) * PG_THREADS] = fprev - f;
        cprev = c; fprev = f;
      }
      double ga = 0.0;  // A'^T G B
      cprev = norm_cdf(0.0 - b); fprev = norm_pdf(0.0 - b);
      for (int i = 1; i <= res; i++) {
        const double x = i * step - b, c = norm_cdf(x), f = norm_pdf(x);
        const double a = c - cprev, da = fprev - f;
        cprev = c; fprev = f;
        const double* g = sg + (i - 1) * res;
        double s1 = 0.0, s2 = 0.0;  // (G B)_i, (G B')_i
        for (int j = 0; j < res; j++) {
          s1 = fma(g[j], B[j * PG_THREADS], s1);
          s2 = fma(g[j], dB[j * PG_THREADS], s2);
        }
        gd = fma(a, wp * s1 + w * s2, gd);
        ga = fma(da, s1, ga);
      }
      gb = w * ga - gd;
    }
    if (grad_birth) grad_birth[k] = gb;
    if (grad_death) grad_death[k] = gd;
  }
}

}  // namespace

void launch_pimg(const Params& p, const ChunkView& c, double* out_pi, float* out_pi_f32, uint8_t* out_status,
                 int block, cudaStream_t st) {
  if (p.resolution == 5) pimg_kernel<5><<<c.T, block, 0, st>>>(p, c, out_pi, out_pi_f32, out_status);
  else pimg_kernel<0><<<c.T, block, 0, st>>>(p, c, out_pi, out_pi_f32, out_status);
  count_launch();
}

void launch_pimg_batch(const int64_t* poff, const double* birth, const double* death, const uint8_t* kind,
                       uint32_t img_mask, int res, int64_t D, double* out, cudaStream_t st) {
  pimg_batch_kernel<<<(unsigned)D, PB_THREADS, 0, st>>>(poff, birth, death, kind, img_mask, res, out);
  count_launch();
}

void launch_pimg_batch_grad(const int64_t* poff, const double* birth, const double* death, const uint8_t* kind,
                            uint32_t img_mask, int res, int64_t D, const double* grad_out, double* grad_birth,
                            double* grad_death, cudaStream_t st) {
  pimg_batch_grad_kernel<<<(unsigned)D, PG_THREADS, 0, st>>>(poff, birth, death, kind, img_mask, res, grad_out,
                                                             grad_birth, grad_death);
  count_launch();
}

}  // namespace tlc
