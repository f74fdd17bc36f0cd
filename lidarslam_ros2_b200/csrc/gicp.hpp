// GICP engine behind the C-ABI: K5 kNN covariances, K6 correspondences + Mahalanobis matrices, K7 cost / gradient
// reductions, and the host-side BFGS driver (pclomp::GeneralizedIterativeClosestPoint, gicp_omp_impl.hpp).
#pragma once
#include <memory>

#include "engine.hpp"

namespace b200 {

constexpr int GICP_MAX_K = 32;

struct GicpConfig {  // gicp_omp.h:108-128
  int k_correspondences = 20;
  double gicp_epsilon = 0.001;
  double rotation_eps = 2e-3;
  int max_inner_iterations = 20;
  int max_iterations = 200;
  double trans_eps = 5e-4;
  double corr_dist = 5.0;
  double gradient_tol = 1e-2;  // see oracle/gicp.hpp header note on testGradient
};

struct GicpOutcome {
  float final_T[16];
  int converged, iterations, evaluations;
};

struct GicpInnerWork;     // device work area of the persistent inner-loop kernel (gicp.cu)
struct GicpInnerResult {  // written by the kernel into pinned host memory
  double x[6];
  double f;
  int status, inner, evaluations, error;
};
struct GicpBatchJob;      // one inner solve of a batched round (gicp.cu)
struct GicpCovSource;     // one source cloud of the batched covariance launch (gicp.cu)

// registrations in flight per batched inner-loop launch (b200reg_gicp_align_batch; like the NDT batch, three at most)
constexpr int GICP_MAX_SLOTS = 3;

struct GicpBatchItem {
  const float4* src;  // device memory, float4 points
  size_t n;
  float guess[16];    // row-major
};
struct GicpBatchOutcome {
  float final_T[16];  // row-major
  int converged, iterations, evaluations;
  int correspondences;  // m of the last outer iteration
  int timed_out;        // the inner-loop watchdog fired during this registration (the other fields are not valid)
};

class GicpSolver {
 public:
  void init(int device, cudaStream_t s);
  void invalidate_target() { target_cov_valid_ = false; }
  void invalidate_source() {
    source_cov_valid_ = false;
    source_grid_valid_ = false;
  }
  GicpOutcome align(const NnGrid& target_grid, const float4* target, size_t n_target, const float4* source,
                    size_t n_source, const GicpConfig& cfg, const float* guess_rowmajor16, cudaStream_t s);
  // `count` independent registrations against the same target, each bitwise what align() gives for its (source, guess).
  // The outer loops run in lock-step rounds; each round's inner solves share one cooperative launch with up to `slots`
  // (1 .. GICP_MAX_SLOTS) of them in flight. The handle's own source, its grid and its covariances are not touched.
  // inner_ms / inner_launches / inner_pair_evaluations describe the whole batch afterwards.
  void align_batch(const NnGrid& target_grid, const float4* target, size_t n_target, const GicpBatchItem* items, int count,
                   const GicpConfig& cfg, int slots, cudaStream_t s, GicpBatchOutcome* out);
  // read-back for parity tests (row-major 3x3 doubles per point); which: 0 source, 1 target
  size_t covariances(int which, std::vector<double>& out, cudaStream_t s);
  int last_correspondences() const { return last_m_; }
  int launches = 0;
  // true: estimateRigidTransformationBFGS runs as ONE persistent cooperative kernel per outer iteration (BFGS on the
  // device); false: host-side BFGS, one K7 launch + synchronisation per functor evaluation
  bool device_bfgs = true;
  // accounting of the last align(): device time of the persistent inner kernel(s), their launches, and the
  // (correspondence, evaluation) products they processed (algorithmic bytes = that times 72, DESIGN.md section 4)
  float inner_ms = 0;
  int inner_launches = 0;
  double inner_pair_evaluations = 0;

 private:
  void fdf(const float* T_rowmajor16, bool want_grad, double* f, double* g_t3, double* R9);
  // returns the BFGS status; x is updated in place
  int inner_loop_device(double* x, const GicpConfig& cfg, int* inner_iterations);
  // the target covariances, computed once per (target, k, gicp_epsilon)
  void ensure_target_covariances(const NnGrid& target_grid, const GicpConfig& cfg, cudaStream_t s);
  // the inner solves of one batched round (h_jobs_[0..n_jobs)) → h_batch_results_[0..n_jobs); error != 0: not solved
  void inner_batch_device(int n_jobs, const GicpConfig& cfg, int slots);
  struct BatchScratch {  // per registration of a batch, reused across calls
    NnGrid grid;
    DeviceBuffer<double> cov;
    DeviceBuffer<float> maha;
    DeviceBuffer<int> corr, nn_idx;
    DeviceBuffer<float> nn_d2;
    DeviceBuffer<float4> moved;
  };
  std::vector<std::unique_ptr<BatchScratch>> batch_;
  GicpInnerWork* d_batch_work_ = nullptr;  // GICP_MAX_SLOTS work areas (one per slot)
  DeviceBuffer<GicpBatchJob> d_jobs_;
  PinnedBuffer<GicpBatchJob> h_jobs_;
  PinnedBuffer<GicpInnerResult> h_batch_results_;  // written by the batch kernel
  DeviceBuffer<GicpCovSource> d_cov_sources_;
  PinnedBuffer<GicpCovSource> h_cov_sources_;
  DeviceBuffer<unsigned> batch_counts_;            // [0] next job of the inner launch, [1 + k] correspondences of k
  PinnedBuffer<unsigned> h_batch_counts_;
  DeviceBuffer<float> d_guess12_;
  PinnedBuffer<float> h_guess12_;
  GicpInnerWork* d_inner_work_ = nullptr;
  GicpInnerResult* h_inner_result_ = nullptr;  // pinned
  unsigned inner_epoch_ = 0;
  cudaEvent_t ev0_ = nullptr, ev1_ = nullptr;
  int sm_count_ = 0;
  int device_ = 0;
  cudaStream_t stream_ = nullptr;
  bool target_cov_valid_ = false, source_cov_valid_ = false, source_grid_valid_ = false;
  int cov_k_ = 0;
  double cov_eps_ = 0;
  NnGrid source_grid_;
  DeviceBuffer<double> target_cov_, source_cov_;  // 6 doubles per point (xx xy xz yy yz zz)
  DeviceBuffer<float> maha_;                      // 9 floats per source point
  DeviceBuffer<int> corr_;                        // target index per source point, -1 = none
  DeviceBuffer<int> nn_idx_;
  DeviceBuffer<float> nn_d2_;
  DeviceBuffer<float4> moved_;                    // source transformed by the guess ("output" cloud)
  DeviceBuffer<double> partials_;                 // per-CTA partial sums (16 doubles each)
  DeviceBuffer<double> result_;                   // 16 doubles
  DeviceBuffer<unsigned> counter_;
  double* h_result_ = nullptr;                    // pinned
  size_t n_source_ = 0, n_target_ = 0;
  const float4* target_ = nullptr;
  int last_m_ = 0;
  int evaluations_ = 0;
};

// k-NN based point covariances of a cloud against its own grid (gicp_omp_impl.hpp:48-122)
void gicp_covariances(const NnGrid& grid, const float4* pts, size_t n, int k, double gicp_epsilon, double* d_cov6,
                      cudaStream_t s);

}  // namespace b200
