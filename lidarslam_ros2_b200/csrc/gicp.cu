// GICP on the GPU: K5 kNN covariances, K6 correspondences + Mahalanobis matrices, K7 cost / gradient reductions, and
// the host-side outer loop + BFGS driver.
//
// Replaces pclomp::GeneralizedIterativeClosestPoint (Thirdparty/ndt_omp_ros2/include/pclomp/gicp_omp_impl.hpp):
//   computeCovariances :48-122 (K5), computeTransformation :369-515 (outer loop; correspondence search :420-456 = K6),
//   OptimizationFunctorWithIndices operator()/df/fdf :244-366 (K7), estimateRigidTransformationBFGS :180-241 with PCL's
//   BFGS (GSL vector_bfgs2; external) restated in bfgs6.hpp, computeRDerivative :125-177, applyState :517-528.
// Nearest neighbours come from the exact cell-grid search of nn_search.cuh instead of FLANN kd-trees.
// Algorithmic HBM bytes (SURVEY.md §8d): K6/K7 per evaluation m*(16+16+48); K5 N*(16 + k*16) + visited cells.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstring>
#include <vector>

#include "bfgs6.hpp"
#include <chrono>
#include <cstdio>
#include <cstdlib>

#include "gicp.hpp"
#include "nn_search.cuh"

namespace b200 {

namespace {

// ---- small f64 3x3 helpers ----------------------------------------------------------------------------------
__device__ __forceinline__ void sym_eig_smallest(const double* c6, double* u3) {
  // eigenvector of the SMALLEST eigenvalue of the symmetric matrix (xx xy xz yy yz zz) by cyclic Jacobi
  double a00 = c6[0], a01 = c6[1], a02 = c6[2], a11 = c6[3], a12 = c6[4], a22 = c6[5];
  double v[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  for (int sweep = 0; sweep < 48; sweep++) {
    const double off = a01 * a01 + a02 * a02 + a12 * a12;
    const double diag = a00 * a00 + a11 * a11 + a22 * a22;
    if (off == 0.0 || off <= 1e-34 * diag) break;
#define B200_ROT(app, aqq, apq, apr, aqr, P, Q)                                        \
  if (apq != 0.0) {                                                                    \
    double theta = (aqq - app) / (2.0 * apq);                                          \
    double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));  \
    double c = 1.0 / sqrt(t * t + 1.0), s = t * c;                                     \
    double napp = app - t * apq, naqq = aqq + t * apq;                                 \
    double napr = c * apr - s * aqr, naqr = s * apr + c * aqr;                         \
    app = napp; aqq = naqq; apq = 0.0; apr = napr; aqr = naqr;                         \
    for (int k = 0; k < 3; k++) {                                                      \
      double vp = v[k * 3 + P], vq = v[k * 3 + Q];                                     \
      v[k * 3 + P] = c * vp - s * vq;                                                  \
      v[k * 3 + Q] = s * vp + c * vq;                                                  \
    }                                                                                  \
  }
    B200_ROT(a00, a11, a01, a02, a12, 0, 1)
    B200_ROT(a00, a22, a02, a01, a12, 0, 2)
    B200_ROT(a11, a22, a12, a01, a02, 1, 2)
#undef B200_ROT
  }
  // JacobiSVD orders singular values (= |eigenvalues|) descending; the last column of U belongs to the smallest
  const double e0 = fabs(a00), e1 = fabs(a11), e2 = fabs(a22);
  int m = 0;
  double em = e0;
  if (e1 < em) { em = e1; m = 1; }
  if (e2 < em) { em = e2; m = 2; }
  u3[0] = v[0 * 3 + m];
  u3[1] = v[1 * 3 + m];
  u3[2] = v[2 * 3 + m];
}

__device__ __forceinline__ void inverse3(const double* m, double* o) {
  const double c00 = m[4] * m[8] - m[5] * m[7];
  const double c01 = m[5] * m[6] - m[3] * m[8];
  const double c02 = m[3] * m[7] - m[4] * m[6];
  const double id = 1.0 / (m[0] * c00 + m[1] * c01 + m[2] * c02);
  o[0] = c00 * id;
  o[1] = (m[2] * m[7] - m[1] * m[8]) * id;
  o[2] = (m[1] * m[5] - m[2] * m[4]) * id;
  o[3] = c01 * id;
  o[4] = (m[0] * m[8] - m[2] * m[6]) * id;
  o[5] = (m[2] * m[3] - m[0] * m[5]) * id;
  o[6] = c02 * id;
  o[7] = (m[1] * m[6] - m[0] * m[7]) * id;
  o[8] = (m[0] * m[4] - m[1] * m[3]) * id;
}

// ---- K5: k nearest neighbours + regularised covariance ---------------------------------------------------------
// One thread per point. The k best (d2, index) pairs are kept in a small unsorted array with the current worst
// tracked; candidates come from Chebyshev rings of the cell grid until the k-th best distance is inside the
// searched radius (exact, ties → lower index like the oracle).
__device__ __forceinline__ void gicp_cov_point(const NnView& V, const float4* __restrict__ pts, int i, int k, double eps,
                                               double* __restrict__ cov6) {
  const float4 q = pts[i];
  float bd[GICP_MAX_K];
  int bi[GICP_MAX_K];
  int cnt = 0;
  float worst = -1.0f;
  int worst_slot = 0, worst_idx = -1;
  const NnGeom& g = V.g;
  const int cx = nn_cell_coord(q.x, g.origin[0], g.inv_h, g.dims[0]);
  const int cy = nn_cell_coord(q.y, g.origin[1], g.inv_h, g.dims[1]);
  const int cz = nn_cell_coord(q.z, g.origin[2], g.inv_h, g.dims[2]);
  const int max_r = max(g.dims[0], max(g.dims[1], g.dims[2]));
  for (int r = 0; r <= max_r; r++) {
    nn_visit_ring(V, cx, cy, cz, r, [&](float4 t) {
      const float d2 = nn_dist2(q.x, q.y, q.z, t);
      const int ti = __float_as_int(t.w);
      if (cnt < k) {
        bd[cnt] = d2;
        bi[cnt] = ti;
        cnt++;
        if (cnt == k) {  // find the worst (largest d2, then largest index)
          worst = -1.0f;
          for (int s = 0; s < k; s++)
            if (bd[s] > worst || (bd[s] == worst && bi[s] > worst_idx)) { worst = bd[s]; worst_idx = bi[s]; worst_slot = s; }
        }
      } else if (d2 < worst || (d2 == worst && ti < worst_idx)) {
        bd[worst_slot] = d2;
        bi[worst_slot] = ti;
        worst = -1.0f;
        worst_idx = -1;
        for (int s = 0; s < k; s++)
          if (bd[s] > worst || (bd[s] == worst && bi[s] > worst_idx)) { worst = bd[s]; worst_idx = bi[s]; worst_slot = s; }
      }
    });
    const float bound = (float)r * g.h;
    if (cnt == k && worst <= bound * bound * 0.99999f) break;
  }
  // mean / covariance of the k neighbours in f64 (gicp_omp_impl.hpp:82-107); the sum order follows ascending
  // (d2, index) like nearestKSearch's sorted result
  for (int a = 1; a < cnt; a++) {  // insertion sort of <= 32 entries
    float d = bd[a];
    int id = bi[a];
    int b = a - 1;
    while (b >= 0 && (bd[b] > d || (bd[b] == d && bi[b] > id))) {
      bd[b + 1] = bd[b];
      bi[b + 1] = bi[b];
      b--;
    }
    bd[b + 1] = d;
    bi[b + 1] = id;
  }
  double mean[3] = {0, 0, 0}, c[6] = {0, 0, 0, 0, 0, 0};
  for (int s = 0; s < cnt; s++) {
    const float4 p = pts[bi[s]];
    mean[0] += (double)p.x; mean[1] += (double)p.y; mean[2] += (double)p.z;
    // the reference forms the products in FLOAT (pt.x * pt.x with float operands, gicp_omp_impl.hpp:89-96)
    c[0] += (double)__fmul_rn(p.x, p.x); c[1] += (double)__fmul_rn(p.y, p.x); c[2] += (double)__fmul_rn(p.z, p.x);
    c[3] += (double)__fmul_rn(p.y, p.y); c[4] += (double)__fmul_rn(p.z, p.y); c[5] += (double)__fmul_rn(p.z, p.z);
  }
  const double kk = (double)k;
  mean[0] /= kk; mean[1] /= kk; mean[2] /= kk;
  c[0] = c[0] / kk - mean[0] * mean[0];
  c[1] = c[1] / kk - mean[1] * mean[0];
  c[2] = c[2] / kk - mean[2] * mean[0];
  c[3] = c[3] / kk - mean[1] * mean[1];
  c[4] = c[4] / kk - mean[2] * mean[1];
  c[5] = c[5] / kk - mean[2] * mean[2];
  // SVD, singular values replaced by (1, 1, gicp_epsilon) (:110-120): cov = I - (1 - eps) u3 u3^T
  double u[3];
  sym_eig_smallest(c, u);
  const double w = 1.0 - eps;
  double* o = cov6 + (size_t)i * 6;
  o[0] = 1.0 - w * u[0] * u[0];
  o[1] = -w * u[0] * u[1];
  o[2] = -w * u[0] * u[2];
  o[3] = 1.0 - w * u[1] * u[1];
  o[4] = -w * u[1] * u[2];
  o[5] = 1.0 - w * u[2] * u[2];
}

__global__ void __launch_bounds__(128) gicp_cov_kernel(NnView V, const float4* __restrict__ pts, int n, int k, double eps,
                                                       double* __restrict__ cov6) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  gicp_cov_point(V, pts, i, k, eps, cov6);
}

}  // namespace

// the clouds of a batched covariance launch: each against its own grid, into its own buffer
struct GicpCovSource {
  NnView V;
  const float4* pts;
  double* cov6;
  int n;
};

namespace {

// K5 over several clouds in one launch (b200reg_gicp_align_batch): blockIdx.y picks the cloud, the points of a cloud are
// covered exactly as gicp_cov_kernel covers them, so every covariance is bitwise the single path's. (128, 8): 64 registers
// and no spills with the table entry held in registers.
__global__ void __launch_bounds__(128, 8) gicp_cov_batch_kernel(const GicpCovSource* __restrict__ sources, int k, double eps) {
  const GicpCovSource S = sources[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= S.n) return;
  gicp_cov_point(S.V, S.pts, i, k, eps, S.cov6);
}

// ---- K6: correspondences + Mahalanobis matrices (gicp_omp_impl.hpp:420-456) ----------------------------------
struct CorrParams {
  const double* cov_src;   // 6 per point
  const double* cov_tgt;
  double R[9];             // (transformation_ * guess) rotation in f64
  float dist_threshold;    // corr_dist^2 as the f32 the comparison effectively sees
  double dist_threshold_d;
  int n;
};

// nearest neighbours come from nn1_query (ring search + brute-force pass for outliers); this kernel applies the
// distance gate and forms M = (R C1 R^T + C2)^-1 in f64
__global__ void __launch_bounds__(128) gicp_corr_kernel(CorrParams P, const int* __restrict__ nn_idx, const float* __restrict__ nn_d2,
                                                        int* __restrict__ corr, float* __restrict__ maha,
                                                        unsigned* __restrict__ count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  int found = 0;
  if (i < P.n) {
    const int bi = nn_idx[i];
    const float best = nn_d2[i];
    int c = -1;
    if (bi >= 0 && (double)best < P.dist_threshold_d) {
      c = bi;
      const double* C1 = P.cov_src + (size_t)i * 6;
      const double* C2 = P.cov_tgt + (size_t)bi * 6;
      const double A[9] = {C1[0], C1[1], C1[2], C1[1], C1[3], C1[4], C1[2], C1[4], C1[5]};
      double M[9], Tm[9];
      for (int r = 0; r < 3; r++)
        for (int cc = 0; cc < 3; cc++) M[r * 3 + cc] = P.R[r * 3] * A[cc] + P.R[r * 3 + 1] * A[3 + cc] + P.R[r * 3 + 2] * A[6 + cc];
      for (int r = 0; r < 3; r++)
        for (int cc = 0; cc < 3; cc++) Tm[r * 3 + cc] = M[r * 3] * P.R[cc * 3] + M[r * 3 + 1] * P.R[cc * 3 + 1] + M[r * 3 + 2] * P.R[cc * 3 + 2];
      Tm[0] += C2[0]; Tm[1] += C2[1]; Tm[2] += C2[2];
      Tm[3] += C2[1]; Tm[4] += C2[3]; Tm[5] += C2[4];
      Tm[6] += C2[2]; Tm[7] += C2[4]; Tm[8] += C2[5];
      inverse3(Tm, M);
      float* mo = maha + (size_t)i * 9;
      for (int k = 0; k < 9; k++) mo[k] = (float)M[k];
      found = 1;
    }
    corr[i] = c;
  }
  const unsigned ballot = __ballot_sync(0xffffffffu, found);
  if ((threadIdx.x & 31) == 0 && ballot) atomicAdd(count, (unsigned)__popc(ballot));
}

// ---- K7: cost / gradient sums over the correspondences (gicp_omp_impl.hpp:244-366) ---------------------------
// slots: 0 f (f32 path, operator()), 1 f (f64 path, fdf), 2..4 sum temp, 5..13 sum p (temp)^T; fixed-order reduction
constexpr int K7_SLOTS = 16;
struct CostParams {
  const float4* moved;
  const float4* target;
  const int* corr;
  const float* maha;
  float T[12];
  int n;
  int want_grad;
};

// one correspondence's contribution to the 14 sums (operator() :264-270; fdf / df :347-360)
__device__ __forceinline__ void cost_point(const CostParams& P, const float* T, int want_grad, int i, double (&acc)[14]) {
  const int c = P.corr[i];
  if (c < 0) return;
  const float4 ps = P.moved[i];
  const float4 pt = __ldg(P.target + c);
  const float px = T[0] * ps.x + T[1] * ps.y + T[2] * ps.z + T[3];
  const float py = T[4] * ps.x + T[5] * ps.y + T[6] * ps.z + T[7];
  const float pz = T[8] * ps.x + T[9] * ps.y + T[10] * ps.z + T[11];
  const float r0 = px - pt.x, r1 = py - pt.y, r2 = pz - pt.z;
  const float* M = P.maha + (size_t)i * 9;
  if (!want_grad) {  // operator(): f32 residual, f32 M * res, f64 accumulation (:264-270)
    const float m0 = M[0] * r0 + M[1] * r1 + M[2] * r2;
    const float m1 = M[3] * r0 + M[4] * r1 + M[5] * r2;
    const float m2 = M[6] * r0 + M[7] * r1 + M[8] * r2;
    acc[0] += (double)(r0 * m0 + r1 * m1 + r2 * m2);
  } else {  // fdf / df: residual to f64, temp = M(f64) * res (:347-360)
    const double d0 = (double)r0, d1 = (double)r1, d2 = (double)r2;
    const double t0 = (double)M[0] * d0 + (double)M[1] * d1 + (double)M[2] * d2;
    const double t1 = (double)M[3] * d0 + (double)M[4] * d1 + (double)M[5] * d2;
    const double t2 = (double)M[6] * d0 + (double)M[7] * d1 + (double)M[8] * d2;
    acc[1] += d0 * t0 + d1 * t1 + d2 * t2;
    acc[2] += t0; acc[3] += t1; acc[4] += t2;
    const double bx = ps.x, by = ps.y, bz = ps.z;  // base_transformation_ = identity (:393)
    acc[5] += bx * t0; acc[6] += bx * t1; acc[7] += bx * t2;
    acc[8] += by * t0; acc[9] += by * t1; acc[10] += by * t2;
    acc[11] += bz * t0; acc[12] += bz * t1; acc[13] += bz * t2;
  }
}

__global__ void __launch_bounds__(256) gicp_cost_kernel(CostParams P, double* __restrict__ partials, unsigned* __restrict__ ticket,
                                                        double* __restrict__ result, double* __restrict__ result_host) {
  double acc[14];
#pragma unroll
  for (int k = 0; k < 14; k++) acc[k] = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < P.n; i += gridDim.x * blockDim.x) cost_point(P, P.T, P.want_grad, i, acc);
  __shared__ double sm[8][K7_SLOTS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 14; k++) {
    double v = acc[k];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    if (lane == 0) sm[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < 14) {
    double s = 0;
    for (int w = 0; w < 8; w++) s += sm[w][threadIdx.x];
    partials[(size_t)blockIdx.x * K7_SLOTS + threadIdx.x] = s;
  }
  __threadfence();
  __shared__ unsigned last;
  __syncthreads();
  if (threadIdx.x == 0) last = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
  __syncthreads();
  if (last) {  // the last CTA sums the per-CTA partials in a fixed order (16 interleaved chains per slot): deterministic
    __threadfence();
    __shared__ double red[16][16];
    const int slot = threadIdx.x & 15, part = threadIdx.x >> 4;
    double s = 0;
    if (slot < 14)
      for (unsigned b = part; b < gridDim.x; b += 16) s += __ldcg(&partials[(size_t)b * K7_SLOTS + slot]);
    red[part][slot] = s;
    __syncthreads();
    if (threadIdx.x < 14) {
      double t = 0;
#pragma unroll
      for (int q = 0; q < 16; q++) t += red[q][threadIdx.x];
      result[threadIdx.x] = t;
      result_host[threadIdx.x] = t;  // pinned host memory mapped into the device address space: no D2H copy to wait for
      __threadfence_system();
    }
    if (threadIdx.x == 0) *ticket = 0;
  }
}

__global__ void __launch_bounds__(256) transform_kernel(const float4* __restrict__ in, int n, float4* out, const float* __restrict__ T12) {
  __shared__ float T[12];
  if (threadIdx.x < 12) T[threadIdx.x] = T12[threadIdx.x];
  __syncthreads();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = in[i];
  out[i] = make_float4(T[0] * p.x + T[1] * p.y + T[2] * p.z + T[3], T[4] * p.x + T[5] * p.y + T[6] * p.z + T[7],
                       T[8] * p.x + T[9] * p.y + T[10] * p.z + T[11], 1.0f);
}

// ---- host-side helpers -------------------------------------------------------------------------------------------
void set_identity16(float* T) {
  for (int k = 0; k < 16; k++) T[k] = (k % 5 == 0) ? 1.0f : 0.0f;
}
void mul3f(const float* a, const float* b, float* c) {
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      float s = 0;
      for (int k = 0; k < 3; k++) s += a[i * 3 + k] * b[k * 3 + j];
      c[i * 3 + j] = s;
    }
}
// gicp_omp_impl.hpp:517-528 (Z * Y * X Euler order, f32)
void apply_state(float* t, const double* x) {
  const float cx = std::cos((float)x[3]), sx = std::sin((float)x[3]);
  const float cy = std::cos((float)x[4]), sy = std::sin((float)x[4]);
  const float cz = std::cos((float)x[5]), sz = std::sin((float)x[5]);
  const float Rz[9] = {cz, -sz, 0, sz, cz, 0, 0, 0, 1}, Ry[9] = {cy, 0, sy, 0, 1, 0, -sy, 0, cy}, Rx[9] = {1, 0, 0, 0, cx, -sx, 0, sx, cx};
  float A[9], R[9], N[9], old[9];
  mul3f(Rz, Ry, A);
  mul3f(A, Rx, R);
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) old[r * 3 + c] = t[r * 4 + c];
  mul3f(R, old, N);
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) t[r * 4 + c] = N[r * 3 + c];
  t[3] += (float)x[0];
  t[7] += (float)x[1];
  t[11] += (float)x[2];
}
// gicp_omp_impl.hpp:125-177
void r_derivative(const double* x, const double* R, double* g) {
  const double phi = x[3], theta = x[4], psi = x[5];
  const double cphi = std::cos(phi), sphi = std::sin(phi), ctheta = std::cos(theta), stheta = std::sin(theta);
  const double cpsi = std::cos(psi), spsi = std::sin(psi);
  const double dPhi[9] = {0, sphi * spsi + cphi * cpsi * stheta, cphi * spsi - cpsi * sphi * stheta,
                          0, -cpsi * sphi + cphi * spsi * stheta, -cphi * cpsi - sphi * spsi * stheta,
                          0, cphi * ctheta, -ctheta * sphi};
  const double dTheta[9] = {-cpsi * stheta, cpsi * ctheta * sphi, cphi * cpsi * ctheta,
                            -spsi * stheta, ctheta * sphi * spsi, cphi * ctheta * spsi,
                            -ctheta, -sphi * stheta, -cphi * stheta};
  const double dPsi[9] = {-ctheta * spsi, -cphi * cpsi - sphi * spsi * stheta, cpsi * sphi - cphi * spsi * stheta,
                          cpsi * ctheta, -cphi * spsi + cpsi * sphi * stheta, sphi * spsi + cphi * cpsi * stheta,
                          0, 0, 0};
  auto inner = [&](const double* m1) {  // matricesInnerProd (gicp_omp.h:316-326)
    double r = 0;
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) r += m1[j * 3 + i] * R[i * 3 + j];
    return r;
  };
  g[3] = inner(dPhi);
  g[4] = inner(dTheta);
  g[5] = inner(dPsi);
}

// ---- outer-loop steps of computeTransformation (:369-515), shared by align() and align_batch() --------------------
// K6 parameters of one outer iteration: transform_R = transformation_ * guess in f64 (:412-418)
CorrParams corr_params(const float* transformation, const float* guess16, const GicpConfig& cfg, const double* cov_src,
                       const double* cov_tgt, size_t n_source) {
  double TR[16] = {0};
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++)
      for (int kk = 0; kk < 4; kk++) TR[i * 4 + j] += double(transformation[i * 4 + kk]) * double(guess16[kk * 4 + j]);
  CorrParams P;
  P.cov_src = cov_src;
  P.cov_tgt = cov_tgt;
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) P.R[r * 3 + c] = TR[r * 4 + c];
  const double dist_threshold = cfg.corr_dist * cfg.corr_dist;
  P.dist_threshold_d = dist_threshold;
  P.dist_threshold = dist_threshold > 3.0e38 ? 3.0e38f : (float)dist_threshold;
  P.n = (int)n_source;
  return P;
}
// the BFGS start: translation and Z-Y-X Euler angles of transformation_ (:198-200)
void bfgs_start(const float* transformation, double* x) {
  x[0] = transformation[3];
  x[1] = transformation[7];
  x[2] = transformation[11];
  x[3] = std::atan2(transformation[9], transformation[10]);
  x[4] = std::asin(-transformation[8]);
  x[5] = std::atan2(transformation[4], transformation[0]);
}
// estimateRigidTransformationBFGS accepts these outcomes and throws on any other (:231-240)
bool bfgs_accepted(int result, int inner, const GicpConfig& cfg) {
  return result == BFGS_NoProgress || result == BFGS_Success || inner == cfg.max_inner_iterations;
}
// convergence test after outer iteration nr_iterations (:479-505); on convergence previous = transformation
bool outer_converged(float* previous, const float* transformation, const GicpConfig& cfg, int nr_iterations) {
  double delta = 0.;
  for (int a = 0; a < 4; a++)
    for (int b = 0; b < 4; b++) {
      const double ratio = (a < 3 && b < 3) ? 1. / cfg.rotation_eps : 1. / cfg.trans_eps;
      const double cd = ratio * std::fabs(previous[a * 4 + b] - transformation[a * 4 + b]);
      if (cd > delta) delta = cd;
    }
  if (nr_iterations >= cfg.max_iterations || delta < 1) {
    std::memcpy(previous, transformation, 16 * sizeof(float));
    return true;
  }
  return false;
}
// final = previous * guess in f32 (:511)
void final_transform(const float* previous, const float* guess16, float* out) {
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++) {
      float acc = 0;
      for (int kk = 0; kk < 4; kk++) acc += previous[i * 4 + kk] * guess16[kk * 4 + j];
      out[i * 4 + j] = acc;
    }
}


// =====================================================================================================================
// Persistent inner loop: estimateRigidTransformationBFGS (gicp_omp_impl.hpp:180-241) for one set of correspondences in ONE
// cooperative launch. The host-driven path above pays a kernel launch and a stream synchronisation for each of the ~65
// functor evaluations of an outer iteration; here evaluator CTAs keep their chunk of correspondences and loop
//   wait for the next transform -> 14 partial sums -> publish a row,
// while EVERY thread of the controller CTA runs the BFGS state machine (bfgs6.hpp) redundantly and identically: each functor
// evaluation is a CTA-wide step — publish the transform, sum the evaluators' rows in a fixed order (the loads are the
// arrival poll), continue. Signalling is the flag-in-data scheme of the NDT solver (ndt_solver.cuh): {payload, sequence}
// control words, self-validating partial rows double-buffered by round parity.
// =====================================================================================================================
constexpr int GI_THREADS = 256;
constexpr int GI_MAX_CTAS = 160;  // one CTA per SM at most (148 on B200); rows per controller thread = GI_MAX_CTAS / 16
constexpr int GI_CTL_WORDS = 14;  // T[12] (float bits), want_grad, mode
constexpr int GI_CTL_COPIES = 4;
constexpr unsigned long long GI_EMPTY = 0xFFF8DEADFFF8DEADull;
constexpr long long GI_TIMEOUT_CYCLES = 4000000000LL;
enum { GI_MODE_RUN = 0, GI_MODE_EXIT = 1 };

}  // namespace

struct GicpInnerWork {
  alignas(128) unsigned long long ctl[GI_CTL_COPIES][16];
  alignas(128) double rows[2][GI_MAX_CTAS][K7_SLOTS];
  unsigned error;
};

namespace {

struct GicpInnerLaunch {
  CostParams P;  // P.T / P.want_grad are unused here: the controller publishes them per evaluation
  GicpInnerWork* work;
  GicpInnerResult* result_host;
  double x0[6];
  double m;  // number of correspondences (the functor's normalisation, gicp_omp_impl.hpp:270, 363-365)
  double gradient_tol;
  int max_inner;
  unsigned epoch;
};

__device__ __forceinline__ unsigned long long gi_ld(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void gi_st(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// gicp_omp_impl.hpp:517-528 (Z * Y * X Euler order, f32), device edition of apply_state()
__device__ void apply_state_dev(float* t, const double* x) {
  const float cx = cosf((float)x[3]), sx = sinf((float)x[3]);
  const float cy = cosf((float)x[4]), sy = sinf((float)x[4]);
  const float cz = cosf((float)x[5]), sz = sinf((float)x[5]);
  const float Rz[9] = {cz, -sz, 0, sz, cz, 0, 0, 0, 1}, Ry[9] = {cy, 0, sy, 0, 1, 0, -sy, 0, cy}, Rx[9] = {1, 0, 0, 0, cx, -sx, 0, sx, cx};
  float A[9], R[9];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      float a = 0;
      for (int k = 0; k < 3; k++) a = __fadd_rn(a, __fmul_rn(Rz[i * 3 + k], Ry[k * 3 + j]));
      A[i * 3 + j] = a;
    }
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      float a = 0;
      for (int k = 0; k < 3; k++) a = __fadd_rn(a, __fmul_rn(A[i * 3 + k], Rx[k * 3 + j]));
      R[i * 3 + j] = a;
    }
  // base = identity: R * I = R
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) t[r * 4 + c] = R[r * 3 + c];
  t[3] = (float)x[0];
  t[7] = (float)x[1];
  t[11] = (float)x[2];
}

// gicp_omp_impl.hpp:125-177
__device__ void r_derivative_dev(const double* x, const double* R, double* g) {
  const double phi = x[3], theta = x[4], psi = x[5];
  const double cphi = cos(phi), sphi = sin(phi), ctheta = cos(theta), stheta = sin(theta), cpsi = cos(psi), spsi = sin(psi);
  const double dPhi[9] = {0, sphi * spsi + cphi * cpsi * stheta, cphi * spsi - cpsi * sphi * stheta,
                          0, -cpsi * sphi + cphi * spsi * stheta, -cphi * cpsi - sphi * spsi * stheta,
                          0, cphi * ctheta, -ctheta * sphi};
  const double dTheta[9] = {-cpsi * stheta, cpsi * ctheta * sphi, cphi * cpsi * ctheta,
                            -spsi * stheta, ctheta * sphi * spsi, cphi * ctheta * spsi,
                            -ctheta, -sphi * stheta, -cphi * stheta};
  const double dPsi[9] = {-ctheta * spsi, -cphi * cpsi - sphi * spsi * stheta, cpsi * sphi - cphi * spsi * stheta,
                          cpsi * ctheta, -cphi * spsi + cpsi * sphi * stheta, sphi * spsi + cphi * cpsi * stheta,
                          0, 0, 0};
  double r3 = 0, r4 = 0, r5 = 0;
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {  // matricesInnerProd (gicp_omp.h:316-326)
      r3 += dPhi[j * 3 + i] * R[i * 3 + j];
      r4 += dTheta[j * 3 + i] * R[i * 3 + j];
      r5 += dPsi[j * 3 + i] * R[i * 3 + j];
    }
  g[3] = r3;
  g[4] = r4;
  g[5] = r5;
}

// the functor the controller CTA's BFGS drives: every thread of the CTA calls it with identical arguments. It reads the work
// area (control words + rows), the epoch and m through L: the single launch's own parameters, or those a batched controller
// fills in for the slot and job it is serving.
struct GicpDeviceFunctor {
  const GicpInnerLaunch* L;
  double (*red)[K7_SLOTS];  // shared [16][16]
  double* tot;              // shared [16]
  int n_eval;
  int round;                // evaluations published so far (identical in every thread)
  int failed;

  __device__ void evaluate(const double* x, int want_grad, double& f, double* g) {
    GicpInnerWork* W = L->work;
    const int tid = threadIdx.x;
    float T[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    apply_state_dev(T, x);
    // publish {payload, sequence}: thread k owns word k
    if (tid < GI_CTL_WORDS) {
      const unsigned payload = tid < 12 ? __float_as_uint(T[tid]) : (tid == 12 ? (unsigned)want_grad : (unsigned)GI_MODE_RUN);
      const unsigned long long v = ((unsigned long long)(L->epoch * 65536u + (unsigned)round + 1u) << 32) | payload;
#pragma unroll
      for (int c = 0; c < GI_CTL_COPIES; c++) gi_st(&W->ctl[c][tid], v);
    }
    // fixed-order reduction of the evaluators' rows; the loads are the arrival poll; consumed words are re-armed
    const int slot = tid & 15, part = tid >> 4;
    double* buf = &W->rows[round & 1][0][0];
    // thread (part, slot) owns words slot of rows part, part + 16, ...: all of them are loaded at once (one L2 round trip),
    // the ones that are still empty are re-loaded
    constexpr int OWN = GI_MAX_CTAS / 16;
    unsigned long long v[OWN];
    unsigned pend = 0;
#pragma unroll
    for (int k = 0; k < OWN; k++) {
      const int b = part + 16 * k;
      v[k] = 0ull;  // bits of +0.0
      if (b < n_eval) {
        v[k] = gi_ld(reinterpret_cast<const unsigned long long*>(buf + (size_t)b * K7_SLOTS + slot));
        if (v[k] == GI_EMPTY) pend |= 1u << k;
      }
    }
    const long long t0 = clock64();
    while (pend && !failed) {
#pragma unroll
      for (int k = 0; k < OWN; k++) {
        if ((pend >> k) & 1u) {
          v[k] = gi_ld(reinterpret_cast<const unsigned long long*>(buf + (size_t)(part + 16 * k) * K7_SLOTS + slot));
          if (v[k] != GI_EMPTY) pend &= ~(1u << k);
        }
      }
      if (clock64() - t0 > GI_TIMEOUT_CYCLES) {
        failed = 1;
        W->error = 1;
      }
    }
    double s = 0;
#pragma unroll
    for (int k = 0; k < OWN; k++) {
      s += __longlong_as_double((long long)v[k]);  // fixed order; rows beyond n_eval contribute +0.0
      const int b = part + 16 * k;
      if (b < n_eval) gi_st(reinterpret_cast<unsigned long long*>(buf + (size_t)b * K7_SLOTS + slot), GI_EMPTY);
    }
    __syncthreads();  // previous evaluation's readers of red/tot are done
    red[part][slot] = s;
    __syncthreads();
    if (tid < K7_SLOTS) {
      double t = 0;
#pragma unroll
      for (int q = 0; q < 16; q++) t += red[q][tid];
      tot[tid] = t;
    }
    __threadfence();  // re-arming stores are performed before the next control words go out
    __syncthreads();
    failed = __syncthreads_or(failed);
    round += 1;
    const double m = L->m;
    if (!want_grad) {
      f = tot[0] / m;
      return;
    }
    f = tot[1] / m;
    double R[9];
    for (int k = 0; k < 3; k++) g[k] = tot[2 + k] * (2.0 / m);
    for (int k = 0; k < 9; k++) R[k] = tot[5 + k] * (2.0 / m);
    r_derivative_dev(x, R, g);
  }
  __device__ double f(const double* x) {
    double v;
    evaluate(x, 0, v, nullptr);
    return v;
  }
  __device__ void fdf(const double* x, double& fo, double* g) { evaluate(x, 1, fo, g); }
  __device__ void df(const double* x, double* g) {
    double fo;
    evaluate(x, 1, fo, g);
  }
};

// estimateRigidTransformationBFGS's inner loop (gicp_omp_impl.hpp:215-230) on the controller CTA; x is updated in place
__device__ __forceinline__ int gi_minimize(GicpDeviceFunctor& fn, double* x, double gradient_tol, int max_inner, int& inner,
                                           double& f) {
  Bfgs6T<GicpDeviceFunctor> bfgs(fn);
  inner = 0;
  int result = bfgs.minimizeInit(x);
  result = BFGS_Running;
  do {
    inner++;
    result = bfgs.minimizeOneStep(x);
    if (result) break;
    result = bfgs.testGradient(gradient_tol);
  } while (result == BFGS_Running && inner < max_inner && !fn.failed);
  f = bfgs.f;
  return result;
}

// the controller tells the evaluators to leave
__device__ __forceinline__ void gi_publish_exit(GicpInnerWork* W, unsigned seq) {
  const int tid = threadIdx.x;
  if (tid < GI_CTL_WORDS) {
    const unsigned payload = tid == 13 ? (unsigned)GI_MODE_EXIT : 0u;
    const unsigned long long v = ((unsigned long long)seq << 32) | payload;
#pragma unroll
    for (int c = 0; c < GI_CTL_COPIES; c++) gi_st(&W->ctl[c][tid], v);
  }
}

__device__ __forceinline__ void gi_write_result(GicpInnerResult* r, const double* x, double f, int status, int inner,
                                                int evaluations, int failed) {
  for (int k = 0; k < 6; k++) r->x[k] = x[k];
  r->f = f;
  r->status = status;
  r->inner = inner;
  r->evaluations = evaluations;
  r->error = failed ? 1 : 0;
  __threadfence_system();
}

// evaluator side of a batched launch: the newest evaluation of a slot whose round is at least `want_round`, as one
// consistent snapshot of the 14 control words (thread k polls word k) → ctl[], its sequence → seq. Words count when their
// sequence lies in the launch's block of epochs: seq - base < span (see GicpBatchLaunch). A controller waits only for the
// evaluators that hold chunks of its job, so an evaluator without one may fall behind by several evaluations and skips
// them (it has nothing to add to them); an evaluator that holds a chunk blocks its controller and so always sees exactly
// the evaluation it has to compute. false when the watchdog fired.
__device__ __forceinline__ bool gi_snapshot_ctl(const unsigned long long* words, unsigned base, unsigned span, unsigned want_round,
                                                unsigned* ctl, unsigned* seq_sh, int* abort_flag, unsigned* error, unsigned& seq) {
  const int tid = threadIdx.x;
  const long long t0 = clock64();
  for (;;) {
    if (tid < GI_CTL_WORDS) {
      unsigned long long v;
      for (;;) {
        v = gi_ld(words + tid);
        const unsigned d = (unsigned)(v >> 32) - base;
        if (d < span && (d & 0xFFFFu) >= want_round + 1u) break;
        if (clock64() - t0 > GI_TIMEOUT_CYCLES) {
          *error = 1;
          *abort_flag = 1;
          break;
        }
      }
      ctl[tid] = (unsigned)v;
      seq_sh[tid] = (unsigned)(v >> 32) - base;
    }
    __syncthreads();
    if (*abort_flag) return false;
    unsigned newest = seq_sh[0];
    bool same = true;
    for (int k = 1; k < GI_CTL_WORDS; k++) {
      same = same && seq_sh[k] == newest;
      newest = max(newest, seq_sh[k]);  // a slot's sequences only grow within a launch (its jobs are taken in order)
    }
    __syncthreads();  // seq_sh / ctl are rewritten by a retry
    if (same) {
      seq = newest;
      return true;
    }
    want_round = (newest & 0xFFFFu) - 1u;  // the controller moved on while the words were read: take the newer evaluation whole
  }
}

// evaluator side: the 14 sums of correspondences [i0, i1) by the whole CTA (strided loop, warp shuffles, then the 8 warps
// in order) published as one row of 16 words. The bits depend only on [i0, i1), not on which CTA computes them.
__device__ __forceinline__ void gi_chunk_row(const CostParams& P, const float* T, int want_grad, int i0, int i1,
                                             double (*sm)[K7_SLOTS], double* row) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double acc[14];
#pragma unroll
  for (int k = 0; k < 14; k++) acc[k] = 0.0;
  for (int i = i0 + tid; i < i1; i += GI_THREADS) cost_point(P, T, want_grad, i, acc);
#pragma unroll
  for (int k = 0; k < 14; k++) {
    double v = acc[k];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    if (lane == 0) sm[warp][k] = v;
  }
  __syncthreads();
  if (tid < K7_SLOTS) {
    double t = 0;
    if (tid < 14)
#pragma unroll
      for (int w = 0; w < GI_THREADS / 32; w++) t += sm[w][tid];
    gi_st(reinterpret_cast<unsigned long long*>(row + tid), (unsigned long long)__double_as_longlong(t));
  }
  __syncthreads();  // sm (and the caller's ctl) are reused by the next chunk / round
}

// evaluator CTAs of a launch for a job of n correspondences (the single launch's geometry; the batch keeps it as virtual
// chunks so that its rows are bitwise the single launch's)
__host__ __device__ __forceinline__ int gi_eval_chunks(int n, int max_ctas) {
  const int c = (n + GI_THREADS - 1) / GI_THREADS;
  return c < max_ctas - 1 ? (c > 1 ? c : 1) : (max_ctas - 1 > 1 ? max_ctas - 1 : 1);
}

__global__ void __launch_bounds__(GI_THREADS) gicp_inner_kernel(const __grid_constant__ GicpInnerLaunch L) {
  GicpInnerWork* W = L.work;
  const int tid = threadIdx.x;
  const int n_eval = (int)gridDim.x - 1;
  if ((int)blockIdx.x == n_eval) {  // ---- controller CTA: every thread runs the same BFGS ----
    __shared__ double red[16][K7_SLOTS];
    __shared__ double tot[K7_SLOTS];
    GicpDeviceFunctor fn{&L, red, tot, n_eval, 0, 0};
    Bfgs6T<GicpDeviceFunctor> bfgs(fn);
    double x[6];
    for (int k = 0; k < 6; k++) x[k] = L.x0[k];
    int inner = 0;
    int result = bfgs.minimizeInit(x);
    result = BFGS_Running;
    do {  // gicp_omp_impl.hpp:215-230
      inner++;
      result = bfgs.minimizeOneStep(x);
      if (result) break;
      result = bfgs.testGradient(L.gradient_tol);
    } while (result == BFGS_Running && inner < L.max_inner && !fn.failed);
    // tell the evaluators to leave
    if (tid < GI_CTL_WORDS) {
      const unsigned payload = tid == 13 ? (unsigned)GI_MODE_EXIT : 0u;
      const unsigned long long v = ((unsigned long long)(L.epoch * 65536u + (unsigned)fn.round + 1u) << 32) | payload;
#pragma unroll
      for (int c = 0; c < GI_CTL_COPIES; c++) gi_st(&W->ctl[c][tid], v);
    }
    if (tid == 0) {
      GicpInnerResult* r = L.result_host;
      for (int k = 0; k < 6; k++) r->x[k] = x[k];
      r->f = bfgs.f;
      r->status = result;
      r->inner = inner;
      r->evaluations = fn.round;
      r->error = fn.failed ? 1 : 0;
      __threadfence_system();
    }
    return;
  }
  // ---- evaluator CTAs ----
  __shared__ unsigned ctl[16];
  __shared__ double sm[GI_THREADS / 32][K7_SLOTS];
  __shared__ int abort_flag;
  if (tid == 0) abort_flag = 0;
  const int rank = (int)blockIdx.x;
  const int chunk = (L.P.n + n_eval - 1) / n_eval;
  const int i0 = rank * chunk, i1 = min(L.P.n, i0 + chunk);
  const int lane = tid & 31, warp = tid >> 5;
  __syncthreads();
  for (int round = 0;; round++) {
    if (tid < GI_CTL_WORDS) {
      const unsigned long long* w = &W->ctl[rank % GI_CTL_COPIES][tid];
      const unsigned want = L.epoch * 65536u + (unsigned)round + 1u;
      const long long t0 = clock64();
      unsigned long long v;
      for (;;) {
        v = gi_ld(w);
        if ((unsigned)(v >> 32) == want) break;
        if (clock64() - t0 > GI_TIMEOUT_CYCLES) {
          W->error = 1;
          abort_flag = 1;
          break;
        }
      }
      ctl[tid] = (unsigned)v;
    }
    __syncthreads();
    if (abort_flag || ctl[13] != (unsigned)GI_MODE_RUN) break;
    float T[12];
#pragma unroll
    for (int k = 0; k < 12; k++) T[k] = __uint_as_float(ctl[k]);
    const int want_grad = (int)ctl[12];
    double acc[14];
#pragma unroll
    for (int k = 0; k < 14; k++) acc[k] = 0.0;
    for (int i = i0 + tid; i < i1; i += GI_THREADS) cost_point(L.P, T, want_grad, i, acc);
#pragma unroll
    for (int k = 0; k < 14; k++) {
      double v = acc[k];
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
      if (lane == 0) sm[warp][k] = v;
    }
    __syncthreads();
    if (tid < K7_SLOTS) {
      double t = 0;
      if (tid < 14)
#pragma unroll
        for (int w = 0; w < GI_THREADS / 32; w++) t += sm[w][tid];
      gi_st(reinterpret_cast<unsigned long long*>(&W->rows[round & 1][rank][tid]), (unsigned long long)__double_as_longlong(t));
    }
    __syncthreads();  // sm and ctl are reused by the next round
  }
}

// =====================================================================================================================
// Batched inner loops (b200reg_gicp_align_batch): the inner solves of one lock-step round of several registrations in ONE
// cooperative launch. CTAs 0 .. S-1 are controllers, one per slot, each running the BFGS of one job at a time exactly as
// the single launch's controller does (same functor, own work area); a slot that finishes a job takes the next one from
// an atomic counter. The other E CTAs are evaluators that serve the slots in turn: wait for slot s's control words (their
// epoch field names the job), compute the job's virtual chunks e, e + E, ... (the single launch's partition of the job),
// publish the rows, go on to the next slot. While one slot's controller is in its BFGS arithmetic the evaluators work for
// the others. A slot takes a further job only while its rounds stay within the 16-bit round field of the sequence words;
// jobs left untaken go to the next launch.
// =====================================================================================================================
constexpr int GI_MAX_ROUNDS = 65534;  // round + 1 must fit below the epoch field of a sequence word
constexpr int kMaxJobsPerLaunch = 4096;  // the launch's block of epochs (jobs + 1) stays far inside 16 bits

}  // namespace

struct GicpBatchJob {
  const float4* moved;
  const int* corr;
  const float* maha;
  int n;
  double x0[6];
  double m;
};

namespace {

struct GicpBatchLaunch {
  const float4* target;
  const GicpBatchJob* jobs;
  GicpInnerResult* results;  // pinned host memory, one per job; error stays 3 for a job no slot took
  GicpInnerWork* work;       // one per slot
  unsigned* next_job;        // zero at launch
  int n_jobs, slots, max_ctas;
  int evals_per_job;         // bound on the evaluations of one job (BFGS line-search limits times max_inner)
  double gradient_tol;
  int max_inner;
  // first of the n_jobs + 1 epochs this launch owns: job j's evaluations carry epoch + j in their sequence words (that is
  // how the evaluators learn the job), the slots' exit words epoch + n_jobs
  unsigned epoch;
};

__global__ void __launch_bounds__(GI_THREADS, 1) gicp_inner_batch_kernel(const __grid_constant__ GicpBatchLaunch L) {
  const int tid = threadIdx.x;
  const int S = L.slots;
  const unsigned seq_base = L.epoch * 65536u;  // sequence of round 0 of job 0
  if ((int)blockIdx.x < S) {  // ---- controller of slot blockIdx.x ----
    __shared__ double red[16][K7_SLOTS];
    __shared__ double tot[K7_SLOTS];
    __shared__ int job_sh;
    __shared__ GicpInnerLaunch job_launch;  // what the functor reads: this slot's work area, the epoch, the job's m
    GicpInnerWork* W = L.work + blockIdx.x;
    int round = 0, failed = 0;
    for (;;) {
      __syncthreads();  // every thread has read the previous job_sh / job_launch
      if (tid == 0) {
        int j = -1;
        if (!failed && (round == 0 || round + L.evals_per_job <= GI_MAX_ROUNDS)) {
          j = (int)atomicAdd(L.next_job, 1u);
          if (j >= L.n_jobs) j = -1;
        }
        job_sh = j;
        if (j >= 0) {
          job_launch.work = W;
          job_launch.epoch = L.epoch + (unsigned)j;  // the job travels in the epoch field of the sequence words
          job_launch.m = L.jobs[j].m;
        }
      }
      __syncthreads();
      const int job = job_sh;
      if (job < 0) break;
      const GicpBatchJob& J = L.jobs[job];
      GicpDeviceFunctor fn{&job_launch, red, tot, gi_eval_chunks(J.n, L.max_ctas), round, 0};
      double x[6];
      for (int k = 0; k < 6; k++) x[k] = J.x0[k];
      int inner;
      double f;
      const int result = gi_minimize(fn, x, L.gradient_tol, L.max_inner, inner, f);
      if (tid == 0) gi_write_result(L.results + job, x, f, result, inner, fn.round - round, fn.failed);
      round = fn.round;
      failed = fn.failed;
    }
    gi_publish_exit(W, (L.epoch + (unsigned)L.n_jobs) * 65536u + (unsigned)round + 1u);
    return;
  }
  // ---- evaluator CTAs ----
  __shared__ unsigned ctl[16];
  __shared__ double sm[GI_THREADS / 32][K7_SLOTS];
  __shared__ int abort_flag;
  __shared__ unsigned seq_sh[16];
  if (tid == 0) abort_flag = 0;
  const int e = (int)blockIdx.x - S, E = (int)gridDim.x - S;
  const unsigned span = (unsigned)(L.n_jobs + 1) << 16;  // the jobs' epochs + the exit words' one
  unsigned long long rounds = 0;  // 16 bits per slot: the slot's next evaluation this CTA expects
  unsigned live = (1u << S) - 1u;
  __syncthreads();
  while (live) {
    for (int s = 0; s < S; s++) {
      if (!((live >> s) & 1u)) continue;
      GicpInnerWork* W = L.work + s;
      unsigned seq;  // relative to the launch's first epoch: (job << 16) + round + 1
      if (!gi_snapshot_ctl(&W->ctl[e % GI_CTL_COPIES][0], seq_base, span, (unsigned)(rounds >> (16 * s)) & 0xFFFFu, ctl, seq_sh,
                           &abort_flag, &W->error, seq))
        return;
      const unsigned round = (seq & 0xFFFFu) - 1u;
      rounds = (rounds & ~(0xFFFFull << (16 * s))) | ((unsigned long long)(round + 1u) << (16 * s));
      const unsigned mode = ctl[13];
      float T[12];
#pragma unroll
      for (int k = 0; k < 12; k++) T[k] = __uint_as_float(ctl[k]);
      const int want_grad = (int)ctl[12];
      __syncthreads();  // ctl is rewritten by the next wait
      if (mode & (unsigned)GI_MODE_EXIT) {
        live &= ~(1u << s);
        continue;
      }
      const GicpBatchJob& J = L.jobs[seq >> 16];
      CostParams P;
      P.moved = J.moved;
      P.target = L.target;
      P.corr = J.corr;
      P.maha = J.maha;
      const int n = J.n, n_eval = gi_eval_chunks(n, L.max_ctas), chunk = (n + n_eval - 1) / n_eval;
      for (int c = e; c < n_eval; c += E) {
        const int i0 = c * chunk;
        gi_chunk_row(P, T, want_grad, i0, min(n, i0 + chunk), sm, &W->rows[round & 1][c][0]);
      }
    }
  }
}

__global__ void gi_arm_kernel(unsigned long long* p, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = GI_EMPTY;
}

}  // namespace

void gicp_covariances(const NnGrid& grid, const float4* pts, size_t n, int k, double gicp_epsilon, double* d_cov6,
                      cudaStream_t s) {
  if (n == 0) return;
  // (A warp-cooperative form — the k best one per lane, bitonic sort + merge networks folding 32 candidates at a time — was
  // measured at 6.1 ms for the 94 k-point scan against 3.3 ms for this thread-per-point kernel: the networks cost more
  // instructions than 32 independent insertion lists, and a warp serialises its 32 queries.)
  gicp_cov_kernel<<<(int)((n + 127) / 128), 128, 0, s>>>(nn_view(grid), pts, (int)n, k, gicp_epsilon, d_cov6);
  B200_CUDA(cudaGetLastError());
}

void GicpSolver::init(int device, cudaStream_t s) {
  device_ = device;
  stream_ = s;
  B200_CUDA(cudaMallocHost(&h_result_, K7_SLOTS * sizeof(double)));
  counter_.ensure(4);
  B200_CUDA(cudaMemset(counter_.ptr, 0, 4 * sizeof(unsigned)));
  result_.ensure(K7_SLOTS);
  partials_.ensure((size_t)148 * 4 * K7_SLOTS);
  cudaDeviceProp prop;
  B200_CUDA(cudaGetDeviceProperties(&prop, device));
  sm_count_ = prop.multiProcessorCount;
  B200_CUDA(cudaMalloc(&d_inner_work_, sizeof(GicpInnerWork)));
  B200_CUDA(cudaMemset(d_inner_work_, 0, sizeof(GicpInnerWork)));
  gi_arm_kernel<<<64, 256>>>(reinterpret_cast<unsigned long long*>(&d_inner_work_->rows[0][0][0]), (size_t)2 * GI_MAX_CTAS * K7_SLOTS);
  B200_CUDA(cudaGetLastError());
  B200_CUDA(cudaDeviceSynchronize());
  B200_CUDA(cudaMallocHost(&h_inner_result_, sizeof(GicpInnerResult)));
}

int GicpSolver::inner_loop_device(double* x, const GicpConfig& cfg, int* inner_iterations) {
  GicpInnerLaunch L{};
  L.P.moved = moved_.ptr;
  L.P.target = target_;
  L.P.corr = corr_.ptr;
  L.P.maha = maha_.ptr;
  L.P.n = (int)n_source_;
  L.work = d_inner_work_;
  L.result_host = h_inner_result_;
  for (int k = 0; k < 6; k++) L.x0[k] = x[k];
  L.m = (double)last_m_;
  L.gradient_tol = cfg.gradient_tol;
  L.max_inner = cfg.max_inner_iterations;
  L.epoch = inner_epoch_++;
  h_inner_result_->error = 3;  // "the kernel never wrote a result"
  const int max_ctas = std::min(sm_count_, GI_MAX_CTAS);
  const int n_eval = std::max(1, std::min((int)((n_source_ + GI_THREADS - 1) / GI_THREADS), max_ctas - 1));
  void* args[] = {&L};
  if (!ev0_) {
    B200_CUDA(cudaEventCreate(&ev0_));
    B200_CUDA(cudaEventCreate(&ev1_));
  }
  {
    std::lock_guard<std::mutex> coop(cooperative_launch_mutex(device_));
    B200_CUDA(cudaEventRecord(ev0_, stream_));
    B200_CUDA(cudaLaunchCooperativeKernel((const void*)gicp_inner_kernel, dim3(n_eval + 1), dim3(GI_THREADS), args, 0, stream_));
    B200_CUDA(cudaEventRecord(ev1_, stream_));
    B200_CUDA(cudaStreamSynchronize(stream_));
  }
  launches += 1;
  {  // roofline accounting of the persistent inner kernel (bench.py --workload c3)
    float ms = 0;
    B200_CUDA(cudaEventElapsedTime(&ms, ev0_, ev1_));
    inner_ms += ms;
    inner_launches += 1;
  }
  const GicpInnerResult& r = *h_inner_result_;
  if (r.error != 0) {  // watchdog (or the kernel never ran): re-arm the rows and report
    gi_arm_kernel<<<64, 256, 0, stream_>>>(reinterpret_cast<unsigned long long*>(&d_inner_work_->rows[0][0][0]), (size_t)2 * GI_MAX_CTAS * K7_SLOTS);
    B200_CUDA(cudaMemsetAsync(&d_inner_work_->error, 0, sizeof(unsigned), stream_));
    B200_CUDA(cudaStreamSynchronize(stream_));
    throw CudaError("GICP inner-loop kernel watchdog fired");
  }
  for (int k = 0; k < 6; k++) x[k] = r.x[k];
  evaluations_ += r.evaluations;
  inner_pair_evaluations += (double)r.evaluations * (double)last_m_;
  *inner_iterations = r.inner;
  return r.status;
}

size_t GicpSolver::covariances(int which, std::vector<double>& out, cudaStream_t s) {
  const DeviceBuffer<double>& buf = which ? target_cov_ : source_cov_;
  const size_t n = which ? n_target_ : n_source_;
  std::vector<double> c6(n * 6);
  if (n) {
    B200_CUDA(cudaMemcpyAsync(c6.data(), buf.ptr, n * 6 * sizeof(double), cudaMemcpyDeviceToHost, s));
    B200_CUDA(cudaStreamSynchronize(s));
  }
  out.resize(n * 9);
  for (size_t i = 0; i < n; i++) {
    const double* c = &c6[i * 6];
    double* o = &out[i * 9];
    o[0] = c[0]; o[1] = c[1]; o[2] = c[2]; o[3] = c[1]; o[4] = c[3]; o[5] = c[4]; o[6] = c[2]; o[7] = c[4]; o[8] = c[5];
  }
  return n;
}

// one evaluation of the fixed-correspondence objective on the device; T = base (identity) with the state applied
void GicpSolver::fdf(const float* T16, bool want_grad, double* f, double* g_t3, double* R9) {
  CostParams P;
  P.moved = moved_.ptr;
  P.target = target_;
  P.corr = corr_.ptr;
  P.maha = maha_.ptr;
  for (int k = 0; k < 12; k++) P.T[k] = T16[k];
  P.n = (int)n_source_;
  P.want_grad = want_grad ? 1 : 0;
  const int blocks = (int)std::min<size_t>((n_source_ + 255) / 256, 148 * 2);
  gicp_cost_kernel<<<std::max(blocks, 1), 256, 0, stream_>>>(P, partials_.ptr, counter_.ptr + 1, result_.ptr, h_result_);
  B200_CUDA(cudaGetLastError());
  B200_CUDA(cudaStreamSynchronize(stream_));
  launches += 1;
  evaluations_ += 1;
  const double m = (double)last_m_;
  if (!want_grad) {
    *f = h_result_[0] / m;
    return;
  }
  *f = h_result_[1] / m;
  for (int k = 0; k < 3; k++) g_t3[k] = h_result_[2 + k] * (2.0 / m);
  for (int k = 0; k < 9; k++) R9[k] = h_result_[5 + k] * (2.0 / m);
}

GicpOutcome GicpSolver::align(const NnGrid& target_grid, const float4* target, size_t n_target, const float4* source,
                              size_t n_source, const GicpConfig& cfg, const float* guess16, cudaStream_t s) {
  // developer trace (env B200REG_GICP_TRACE=1): host wall clock per phase of one align, printed to stderr
  static const bool trace = getenv("B200REG_GICP_TRACE") != nullptr;
  auto now = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  double t_prev = trace ? now() : 0, t_cov = 0, t_nn = 0, t_inner = 0;
  auto lap = [&](double& acc) {
    if (!trace) return;
    B200_CUDA(cudaStreamSynchronize(s));
    const double t = now();
    acc += t - t_prev;
    t_prev = t;
  };
  stream_ = s;
  target_ = target;
  n_target_ = n_target;
  n_source_ = n_source;
  evaluations_ = 0;
  inner_ms = 0;
  inner_launches = 0;
  inner_pair_evaluations = 0;
  GicpOutcome out;
  set_identity16(out.final_T);
  out.converged = 0;
  out.iterations = 0;
  out.evaluations = 0;
  const int k = std::min(cfg.k_correspondences, GICP_MAX_K);
  // covariances (lazy, cached per cloud; :381-391). Clouds smaller than k are rejected like :54-58 (left zero).
  ensure_target_covariances(target_grid, cfg, s);
  if (!source_grid_valid_) {
    source_grid_.build(source, n_source, s);
    source_grid_valid_ = true;
  }
  if (!source_cov_valid_) {
    source_cov_.ensure(n_source * 6 + 6);
    B200_CUDA(cudaMemsetAsync(source_cov_.ptr, 0, n_source * 6 * sizeof(double), s));
    if ((size_t)k <= n_source) gicp_covariances(source_grid_, source, n_source, k, cfg.gicp_epsilon, source_cov_.ptr, s);
    source_cov_valid_ = true;
    launches += 1;
  }
  maha_.ensure(n_source * 9);
  corr_.ensure(n_source);
  moved_.ensure(n_source);
  const int blocks_pts = (int)((n_source + 255) / 256);
  // "output" = source transformed by the guess (:397)
  DeviceBuffer<float>& tbuf = maha_;  // reuse the head of maha_ as a 12-float scratch before K6 overwrites it
  B200_CUDA(cudaMemcpyAsync(tbuf.ptr, guess16, 12 * sizeof(float), cudaMemcpyHostToDevice, s));
  transform_kernel<<<blocks_pts, 256, 0, s>>>(source, (int)n_source, moved_.ptr, tbuf.ptr);
  launches += 1;

  lap(t_cov);
  float transformation[16], previous[16];
  set_identity16(transformation);
  set_identity16(previous);
  bool converged = false;
  int nr_iterations = 0;
  while (!converged) {
    const CorrParams P = corr_params(transformation, guess16, cfg, source_cov_.ptr, target_cov_.ptr, n_source);
    B200_CUDA(cudaMemsetAsync(counter_.ptr, 0, sizeof(unsigned), s));
    // query = transformation_ * output[i] (:426-427); nn1_query applies the 3x4 transform in f32
    nn_idx_.ensure(n_source);
    nn_d2_.ensure(n_source);
    nn1_query(target_grid, moved_.ptr, n_source, transformation, nn_idx_.ptr, nn_d2_.ptr, s, P.dist_threshold * 1.0001f);
    gicp_corr_kernel<<<(int)((n_source + 127) / 128), 128, 0, s>>>(P, nn_idx_.ptr, nn_d2_.ptr, corr_.ptr, maha_.ptr, counter_.ptr);
    unsigned m = 0;
    B200_CUDA(cudaMemcpyAsync(&m, counter_.ptr, sizeof(unsigned), cudaMemcpyDeviceToHost, s));
    B200_CUDA(cudaStreamSynchronize(s));
    launches += 1;
    last_m_ = (int)m;
    lap(t_nn);
    std::memcpy(previous, transformation, sizeof(previous));
    if (m < 4) break;  // NotEnoughPointsException → caught → break (:187-192, :494-498)

    // estimateRigidTransformationBFGS (:180-241)
    double x[6];
    bfgs_start(transformation, x);
    BfgsFunctor6 fn;
    fn.f = [&](const double* xx) {
      float T[16];
      set_identity16(T);
      apply_state(T, xx);
      double f;
      fdf(T, false, &f, nullptr, nullptr);
      return f;
    };
    fn.fdf = [&](const double* xx, double& f, double* gg) {
      float T[16];
      set_identity16(T);
      apply_state(T, xx);
      double gt[3], R[9];
      fdf(T, true, &f, gt, R);
      for (int q = 0; q < 3; q++) gg[q] = gt[q];
      r_derivative(xx, R, gg);
    };
    fn.df = [&](const double* xx, double* gg) {
      double f;
      fn.fdf(xx, f, gg);
    };
    int inner = 0;
    int result;
    if (device_bfgs) {
      result = inner_loop_device(x, cfg, &inner);
    } else {
      Bfgs6 bfgs(fn);
      result = bfgs.minimizeInit(x);
      result = BFGS_Running;
      do {
        inner++;
        result = bfgs.minimizeOneStep(x);
        if (result) break;
        result = bfgs.testGradient(cfg.gradient_tol);
      } while (result == BFGS_Running && inner < cfg.max_inner_iterations);
    }
    lap(t_inner);
    if (!bfgs_accepted(result, inner, cfg)) break;  // throws in the reference
    set_identity16(transformation);
    apply_state(transformation, x);
    nr_iterations++;
    converged = outer_converged(previous, transformation, cfg, nr_iterations);
  }
  final_transform(previous, guess16, out.final_T);
  out.converged = converged ? 1 : 0;
  out.iterations = nr_iterations;
  out.evaluations = evaluations_;
  if (trace)
    std::fprintf(stderr, "[gicp trace] source grid + covariances + transform %.3f ms, correspondences (NN + Mahalanobis) %.3f ms, "
                         "inner BFGS launches %.3f ms (kernel events %.3f ms), %d outer iterations, %d evaluations\n",
                 t_cov, t_nn, t_inner, inner_ms, nr_iterations, evaluations_);
  return out;
}

void GicpSolver::ensure_target_covariances(const NnGrid& target_grid, const GicpConfig& cfg, cudaStream_t s) {
  const int k = std::min(cfg.k_correspondences, GICP_MAX_K);
  if (cov_k_ != k || cov_eps_ != cfg.gicp_epsilon) {
    target_cov_valid_ = source_cov_valid_ = false;
    cov_k_ = k;
    cov_eps_ = cfg.gicp_epsilon;
  }
  if (!target_cov_valid_) {
    target_cov_.ensure(n_target_ * 6 + 6);
    B200_CUDA(cudaMemsetAsync(target_cov_.ptr, 0, n_target_ * 6 * sizeof(double), s));
    if ((size_t)k <= n_target_) gicp_covariances(target_grid, target_, n_target_, k, cfg.gicp_epsilon, target_cov_.ptr, s);
    target_cov_valid_ = true;
    launches += 1;
  }
}

void GicpSolver::inner_batch_device(int n_jobs, const GicpConfig& cfg, int slots) {
  const int max_ctas = std::min(sm_count_, GI_MAX_CTAS);
  if (!d_batch_work_) {
    B200_CUDA(cudaMalloc(&d_batch_work_, GICP_MAX_SLOTS * sizeof(GicpInnerWork)));
    B200_CUDA(cudaMemsetAsync(d_batch_work_, 0, GICP_MAX_SLOTS * sizeof(GicpInnerWork), stream_));
    for (int w = 0; w < GICP_MAX_SLOTS; w++)
      gi_arm_kernel<<<64, 256, 0, stream_>>>(reinterpret_cast<unsigned long long*>(&d_batch_work_[w].rows[0][0][0]),
                                            (size_t)2 * GI_MAX_CTAS * K7_SLOTS);
    B200_CUDA(cudaGetLastError());
  }
  if (!ev0_) {
    B200_CUDA(cudaEventCreate(&ev0_));
    B200_CUDA(cudaEventCreate(&ev1_));
  }
  d_jobs_.ensure((size_t)n_jobs);
  B200_CUDA(cudaMemcpyAsync(d_jobs_.ptr, h_jobs_.ptr, n_jobs * sizeof(GicpBatchJob), cudaMemcpyHostToDevice, stream_));
  for (int j = 0; j < n_jobs; j++) h_batch_results_.ptr[j].error = 3;  // "no slot took this job"
  // a line search evaluates at most 2 * 100 times, plus up to 2 + 2 around it; minimizeInit once
  const long long per_job = 1 + (long long)std::max(cfg.max_inner_iterations, 1) * (2 * 100 + 4);
  GicpBatchLaunch L{};
  L.target = target_;
  L.work = d_batch_work_;
  L.next_job = batch_counts_.ptr;
  L.max_ctas = max_ctas;
  L.evals_per_job = (int)std::min<long long>(per_job, GI_MAX_ROUNDS + 1);
  L.gradient_tol = cfg.gradient_tol;
  L.max_inner = cfg.max_inner_iterations;
  bool failed = false;
  for (int first = 0; first < n_jobs && !failed;) {
    L.jobs = d_jobs_.ptr + first;
    L.results = h_batch_results_.ptr + first;
    L.n_jobs = std::min(n_jobs - first, kMaxJobsPerLaunch);
    L.slots = std::max(1, std::min({slots, L.n_jobs, max_ctas - 1}));
    L.epoch = inner_epoch_;
    inner_epoch_ += (unsigned)L.n_jobs + 1u;
    void* args[] = {&L};
    {
      std::lock_guard<std::mutex> coop(cooperative_launch_mutex(device_));
      // no control word of an earlier launch may pass for one of this launch (whatever the epochs have wrapped to)
      for (int w = 0; w < L.slots; w++) B200_CUDA(cudaMemsetAsync(&d_batch_work_[w].ctl[0][0], 0, sizeof(d_batch_work_[w].ctl), stream_));
      B200_CUDA(cudaMemsetAsync(L.next_job, 0, sizeof(unsigned), stream_));
      B200_CUDA(cudaEventRecord(ev0_, stream_));
      B200_CUDA(cudaLaunchCooperativeKernel((const void*)gicp_inner_batch_kernel, dim3(max_ctas), dim3(GI_THREADS), args, 0, stream_));
      B200_CUDA(cudaEventRecord(ev1_, stream_));
      B200_CUDA(cudaStreamSynchronize(stream_));
    }
    launches += 1;
    float ms = 0;
    B200_CUDA(cudaEventElapsedTime(&ms, ev0_, ev1_));
    inner_ms += ms;
    inner_launches += 1;
    // the slots take jobs in order from the counter: the solved ones are a prefix
    const int before = first;
    while (first < n_jobs && h_batch_results_.ptr[first].error != 3) failed |= h_batch_results_.ptr[first++].error != 0;
    if (first == before) failed = true;  // no progress: only a launch that never ran leaves every job untaken
  }
  if (failed) {  // watchdog: re-arm the rows of every slot and report (the untaken jobs keep error 3)
    for (int w = 0; w < GICP_MAX_SLOTS; w++) {
      gi_arm_kernel<<<64, 256, 0, stream_>>>(reinterpret_cast<unsigned long long*>(&d_batch_work_[w].rows[0][0][0]),
                                            (size_t)2 * GI_MAX_CTAS * K7_SLOTS);
      B200_CUDA(cudaMemsetAsync(&d_batch_work_[w].error, 0, sizeof(unsigned), stream_));
    }
    B200_CUDA(cudaStreamSynchronize(stream_));
  }
}

void GicpSolver::align_batch(const NnGrid& target_grid, const float4* target, size_t n_target, const GicpBatchItem* items,
                             int count, const GicpConfig& cfg, int slots, cudaStream_t s, GicpBatchOutcome* out) {
  stream_ = s;
  target_ = target;
  n_target_ = n_target;
  evaluations_ = 0;
  inner_ms = 0;
  inner_launches = 0;
  inner_pair_evaluations = 0;
  ensure_target_covariances(target_grid, cfg, s);
  if (count <= 0) return;
  const int k = std::min(cfg.k_correspondences, GICP_MAX_K);
  while ((int)batch_.size() < count) batch_.emplace_back(new BatchScratch());
  // source grids and covariances: the grid builds back to back (each reads its cloud's bounds back), then ONE K5 launch
  // over every cloud of at least k points (smaller ones keep zero covariances, :54-58)
  h_cov_sources_.ensure((size_t)count);
  int n_cov = 0;
  size_t max_n = 0;
  for (int r = 0; r < count; r++) {
    BatchScratch& B = *batch_[r];
    const size_t n = items[r].n;
    B.grid.build(items[r].src, n, s);
    B.cov.ensure(n * 6 + 6);
    B200_CUDA(cudaMemsetAsync(B.cov.ptr, 0, n * 6 * sizeof(double), s));
    B.maha.ensure(n * 9);
    B.corr.ensure(n);
    B.nn_idx.ensure(n);
    B.nn_d2.ensure(n);
    B.moved.ensure(n);
    if ((size_t)k <= n) {
      h_cov_sources_.ptr[n_cov++] = GicpCovSource{nn_view(B.grid), items[r].src, B.cov.ptr, (int)n};
      max_n = std::max(max_n, n);
    }
  }
  if (n_cov > 0) {
    d_cov_sources_.ensure((size_t)n_cov);
    B200_CUDA(cudaMemcpyAsync(d_cov_sources_.ptr, h_cov_sources_.ptr, n_cov * sizeof(GicpCovSource), cudaMemcpyHostToDevice, s));
    for (int first = 0; first < n_cov; first += 65535) {  // gridDim.y limit
      const dim3 grid((unsigned)((max_n + 127) / 128), (unsigned)std::min(65535, n_cov - first));
      gicp_cov_batch_kernel<<<grid, 128, 0, s>>>(d_cov_sources_.ptr + first, k, cfg.gicp_epsilon);
      B200_CUDA(cudaGetLastError());
      launches += 1;
    }
  }
  // "output" = each source transformed by its guess (:397)
  h_guess12_.ensure((size_t)count * 12);
  d_guess12_.ensure((size_t)count * 12);
  for (int r = 0; r < count; r++) std::memcpy(h_guess12_.ptr + 12 * r, items[r].guess, 12 * sizeof(float));
  B200_CUDA(cudaMemcpyAsync(d_guess12_.ptr, h_guess12_.ptr, count * 12 * sizeof(float), cudaMemcpyHostToDevice, s));
  for (int r = 0; r < count; r++) {
    transform_kernel<<<(int)((items[r].n + 255) / 256), 256, 0, s>>>(items[r].src, (int)items[r].n, batch_[r]->moved.ptr,
                                                                      d_guess12_.ptr + 12 * r);
    launches += 1;
  }
  B200_CUDA(cudaGetLastError());

  // the outer loops in lock-step rounds: round i is outer iteration i of every registration still running
  struct Reg {
    float transformation[16], previous[16];
    bool active = true, converged = false, timed_out = false;
    int nr_iterations = 0, evaluations = 0, m = 0;
  };
  std::vector<Reg> R((size_t)count);
  for (Reg& g : R) {
    set_identity16(g.transformation);
    set_identity16(g.previous);
  }
  batch_counts_.ensure((size_t)count + 1);
  h_batch_counts_.ensure((size_t)count + 1);
  h_jobs_.ensure((size_t)count);
  h_batch_results_.ensure((size_t)count);
  std::vector<int> job_reg;
  for (;;) {
    bool any = false;
    for (const Reg& g : R) any = any || g.active;
    if (!any) break;
    // correspondences of every running registration, back to back (stream order keeps the shared grid's query scratch
    // safe); one read-back of all counts
    unsigned* counts = batch_counts_.ptr + 1;
    B200_CUDA(cudaMemsetAsync(counts, 0, count * sizeof(unsigned), s));
    for (int r = 0; r < count; r++) {
      if (!R[r].active) continue;
      BatchScratch& B = *batch_[r];
      const size_t n = items[r].n;
      const CorrParams P = corr_params(R[r].transformation, items[r].guess, cfg, B.cov.ptr, target_cov_.ptr, n);
      nn1_query(target_grid, B.moved.ptr, n, R[r].transformation, B.nn_idx.ptr, B.nn_d2.ptr, s, P.dist_threshold * 1.0001f);
      gicp_corr_kernel<<<(int)((n + 127) / 128), 128, 0, s>>>(P, B.nn_idx.ptr, B.nn_d2.ptr, B.corr.ptr, B.maha.ptr, counts + r);
      launches += 1;
    }
    B200_CUDA(cudaGetLastError());
    B200_CUDA(cudaMemcpyAsync(h_batch_counts_.ptr, counts, count * sizeof(unsigned), cudaMemcpyDeviceToHost, s));
    B200_CUDA(cudaStreamSynchronize(s));
    // this round's inner solves
    job_reg.clear();
    for (int r = 0; r < count; r++) {
      Reg& g = R[r];
      if (!g.active) continue;
      g.m = (int)h_batch_counts_.ptr[r];
      std::memcpy(g.previous, g.transformation, sizeof(g.previous));
      if (g.m < 4) {  // NotEnoughPointsException → caught → break (:187-192, :494-498)
        g.active = false;
        continue;
      }
      GicpBatchJob& J = h_jobs_.ptr[job_reg.size()];
      J.moved = batch_[r]->moved.ptr;
      J.corr = batch_[r]->corr.ptr;
      J.maha = batch_[r]->maha.ptr;
      J.n = (int)items[r].n;
      bfgs_start(g.transformation, J.x0);
      J.m = (double)g.m;
      job_reg.push_back(r);
    }
    if (job_reg.empty()) continue;
    inner_batch_device((int)job_reg.size(), cfg, slots);
    for (size_t j = 0; j < job_reg.size(); j++) {
      Reg& g = R[job_reg[j]];
      const GicpInnerResult& res = h_batch_results_.ptr[j];
      if (res.error != 0) {
        g.timed_out = true;
        g.active = false;
        continue;
      }
      g.evaluations += res.evaluations;
      evaluations_ += res.evaluations;
      inner_pair_evaluations += (double)res.evaluations * (double)g.m;
      if (!bfgs_accepted(res.status, res.inner, cfg)) {  // throws in the reference
        g.active = false;
        continue;
      }
      set_identity16(g.transformation);
      apply_state(g.transformation, res.x);
      g.nr_iterations++;
      if (outer_converged(g.previous, g.transformation, cfg, g.nr_iterations)) {
        g.converged = true;
        g.active = false;
      }
    }
  }
  for (int r = 0; r < count; r++) {
    const Reg& g = R[r];
    GicpBatchOutcome& o = out[r];
    final_transform(g.previous, items[r].guess, o.final_T);
    o.converged = g.converged ? 1 : 0;
    o.iterations = g.nr_iterations;
    o.evaluations = g.evaluations;
    o.correspondences = g.m;
    o.timed_out = g.timed_out ? 1 : 0;
  }
  last_m_ = R[count - 1].m;
}

}  // namespace b200
