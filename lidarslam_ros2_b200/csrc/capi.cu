// extern "C" implementation of include/b200reg.h. No CPU fallback: every compute entry point launches CUDA
// kernels; if no device is present b200reg_create fails.
#include <cfloat>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <dlfcn.h>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/b200reg.h"
#include "engine.hpp"
#include "gicp.hpp"

using namespace b200;

static size_t g_vg_dense_budget = (size_t)4 << 20;  // b200reg_voxelgrid: dense-bitmap budget in words (debug hook below)
static constexpr int NDT_BATCH_SLOTS_DEFAULT = 3;  // registrations in flight per batch launch (engine.hpp / ndt_solver.cuh)

struct b200reg_engine {
  int kind = B200REG_NDT;
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::string err;

  // pcl::Registration parameters
  double corr_dist = std::sqrt(DBL_MAX);  // PCL default corr_dist_threshold_
  double euclid_eps = -DBL_MAX;
  int ransac_iters = 0;
  NdtConfig ndt;
  int min_points_per_voxel = 6;           // voxel_grid_covariance_omp.h:204
  double min_covar_eigvalue_mult = 0.01;  // voxel_grid_covariance_omp.h:205
  GicpConfig gicp;

  DeviceBuffer<float4> d_target, d_source, d_aligned;
  const float4* src_view = nullptr;  // the source cloud the solves read: d_source, or a caller-owned device buffer (b200reg_adopt_source_device)
  PinnedBuffer<float4> staging;
  CloudUploader uploader;
  size_t n_target = 0, n_source = 0;
  bool have_target = false, have_source = false;
  bool map_valid = false, nn_valid = false;
  float map_resolution = 0;
  Bounds target_bounds{};            // min/max of the target, measured once (during the upload when it comes from the host)
  bool target_bounds_valid = false;

  VoxelMap map;
  NnGrid nn;
  NdtSolver solver;
  GicpSolver gicp_solver;

  DeviceBuffer<int> nn_idx;
  DeviceBuffer<float> nn_d2;
  DeviceBuffer<unsigned> scratch_bounds;
  DeviceBuffer<double> scratch_d;   // >= 64 doubles
  DeviceBuffer<float> scratch_f;    // >= 16 floats
  DeviceBuffer<float4> query_buf;

  // results of the last align (row-major)
  float final_T[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
  int converged = 0, iterations = 0, evaluations = 0;
  double trans_probability = 0;
  long long hits_last = 0, hits_total = 0;
  float solve_ms = 0, target_build_ms = 0;
  bool align_pending = false;
  std::unique_lock<std::mutex> coop_lock;  // held from a solver launch until its completion (cooperative_launch_mutex)
  bool grid_overflow = false;  // the last voxel-map build hit the int32 guard (voxel_grid_covariance_omp_impl.hpp:79)
  int other_launches = 0;

  // batched registrations (b200reg_ndt_align_batch*)
  DeviceBuffer<float4> d_batch;          // host-buffer form: all sources of the batch, back to back
  CloudUploader batch_uploader;
  std::vector<NdtSolver::BatchItem> batch_items;
  int batch_slots = NDT_BATCH_SLOTS_DEFAULT;
  b200comm_board* board = nullptr;  // attached pose board (not owned): batch launches also publish their poses to the peers
  int board_valid = 0;              // the last batch call filled board->h_rows
  int sibling_launches_seen[3] = {0, 0, 0};
  cudaStream_t copy_stream = nullptr;    // streaming uploads of b200reg_ndt_align_batch
  DeviceBuffer<unsigned> batch_ready;    // one "scan k has arrived" flag per registration of a batch
  unsigned batch_tag = 0;                // value the flags take for the current call
  b200reg_engine* siblings[3] = {nullptr, nullptr, nullptr};  // further engines of b200reg_ndt_sweep (own stream and buffers each)
  int sweep_engines = 4;  // engines (host threads) the sweep pipelines over (developer switch: B200REG_SWEEP_ENGINES)
};

namespace {

void set_identity(float* T) {
  for (int k = 0; k < 16; k++) T[k] = (k % 5 == 0) ? 1.0f : 0.0f;
}
void col_to_row(const float* c, float* r) {
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++) r[i * 4 + j] = c[j * 4 + i];
}
void row_to_col(const float* r, float* c) {
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++) c[j * 4 + i] = r[i * 4 + j];
}

template <typename F>
int guarded(b200reg_t h, F&& f) {
  if (!h) return B200REG_ERR_ARG;
  try {
    cudaError_t e = cudaSetDevice(h->device);
    if (e != cudaSuccess) {
      h->err = std::string("cudaSetDevice: ") + cudaGetErrorString(e);
      return B200REG_ERR_CUDA;
    }
    return f();
  } catch (const CudaError& e) {
    h->err = e.what();
    cudaGetLastError();
    return B200REG_ERR_CUDA;
  } catch (const std::exception& e) {
    h->err = e.what();
    return B200REG_ERR_ARG;
  }
}

int fail(b200reg_t h, int code, const char* msg) {
  h->err = msg;
  return code;
}

// min/max of the target cloud: both the NDT voxel grid and the NN grid are sized from them
const Bounds* target_bounds(b200reg_t h) {
  if (!h->target_bounds_valid) {
    h->scratch_bounds.ensure(8);
    h->target_bounds = cloud_bounds(h->d_target.ptr, h->n_target, h->scratch_bounds.ptr, h->stream);
    h->target_bounds_valid = true;
    h->other_launches += 1;
  }
  return &h->target_bounds;
}

void ensure_map(b200reg_t h) {
  if (h->map_valid && h->map_resolution == h->ndt.resolution) return;
  const Bounds* tb = target_bounds(h);
  B200_CUDA(cudaEventRecord(h->ev0, h->stream));
  bool ok = h->map.build(h->d_target.ptr, h->n_target, h->ndt.resolution, h->min_points_per_voxel,
                         h->min_covar_eigvalue_mult, h->stream, tb);
  B200_CUDA(cudaEventRecord(h->ev1, h->stream));
  B200_CUDA(cudaEventSynchronize(h->ev1));
  B200_CUDA(cudaEventElapsedTime(&h->target_build_ms, h->ev0, h->ev1));
  h->map_valid = true;
  h->map_resolution = h->ndt.resolution;
  h->grid_overflow = !ok;
  if (!ok) h->err = "voxel grid would overflow int32: leaf size too small for the target cloud (map left empty)";
}

void ensure_nn(b200reg_t h) {
  if (h->nn_valid) return;
  h->nn.build(h->d_target.ptr, h->n_target, h->stream, target_bounds(h));
  h->nn_valid = true;
}

// developer trace (env B200REG_TRACE=1): host wall clock of the phases of one NDT align, printed to stderr
static const bool g_trace = getenv("B200REG_TRACE") != nullptr;
static double trace_now() {
  return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
static thread_local double g_trace_t[4];

// ---- NDT align: enqueue / complete ------------------------------------------------------------------------
int ndt_align_begin(b200reg_t h, const float* guess_colmajor) {
  if (g_trace) g_trace_t[0] = trace_now();
  h->converged = 0;
  set_identity(h->final_T);
  if (!h->have_target) return fail(h, B200REG_ERR_NO_TARGET, "align: no input target");
  if (!h->have_source) return fail(h, B200REG_ERR_NO_SOURCE, "align: no input source");
  ensure_map(h);
  float T[16];
  if (guess_colmajor) col_to_row(guess_colmajor, T);
  else set_identity(T);
  if (h->map.n_voxels == 0) {
    // no voxel holds >= 6 points: the reference's first solve returns delta_p == 0 → converged, final = guess
    std::memcpy(h->final_T, T, sizeof(T));
    h->converged = 1;
    h->iterations = 0;
    h->evaluations = 1;
    h->trans_probability = 0;
    h->hits_last = h->hits_total = 0;
    h->align_pending = false;
    return B200REG_OK;
  }
  if (g_trace) g_trace_t[1] = trace_now();
  h->coop_lock = std::unique_lock<std::mutex>(cooperative_launch_mutex(h->device));
  try {
    B200_CUDA(cudaEventRecord(h->ev0, h->stream));
    h->solver.launch(h->map, h->src_view, h->n_source, h->ndt, NDT_MODE_ALIGN, T, nullptr, 1, 0);
    B200_CUDA(cudaEventRecord(h->ev1, h->stream));  // solve_ms brackets the kernel(s) on the stream, nothing host-side
  } catch (...) {
    h->coop_lock.unlock();
    throw;
  }
  if (g_trace) g_trace_t[2] = trace_now();
  h->align_pending = true;
  return B200REG_OK;
}

int ndt_align_end(b200reg_t h) {
  if (!h->align_pending) return B200REG_OK;
  h->align_pending = false;
  struct Release {  // the solver kernel(s) of this align are complete (or failed) whenever this function returns
    std::unique_lock<std::mutex>& l;
    ~Release() {
      if (l.owns_lock()) l.unlock();
    }
  } release{h->coop_lock};
  for (int rounds = 0; rounds < 4096; rounds++) {
    B200_CUDA(cudaStreamSynchronize(h->stream));
    if (h->solver.result().error == 3) h->solver.fetch_result();
    const NdtResult& r = h->solver.result();
    if (r.error == 100) {
      // the More-Thuente loop ran (only when step_max <= step_min): f64 radius Hessian (K2), then resume
      h->scratch_d.ensure(64);
      ndt_hessian_radius(h->map, h->src_view, h->n_source, h->ndt, h->solver.control_T(), h->solver.state_jd(),
                         h->solver.state_hd(), h->scratch_d.ptr, h->stream);
      ndt_hessian_into_state(h->scratch_d.ptr, h->solver.work(), h->stream);
      h->other_launches += 2;
      float dummyT[16];
      set_identity(dummyT);
      h->solver.launch(h->map, h->src_view, h->n_source, h->ndt, NDT_MODE_ALIGN, dummyT, nullptr, 1, 1);
      B200_CUDA(cudaEventRecord(h->ev1, h->stream));
      continue;
    }
    if (r.error != 0) {
      h->solver.reset_barrier();
      B200_CUDA(cudaStreamSynchronize(h->stream));
      return fail(h, B200REG_ERR_TIMEOUT, "NDT solver kernel watchdog fired (grid barrier timeout)");
    }
    B200_CUDA(cudaEventElapsedTime(&h->solve_ms, h->ev0, h->ev1));
    if (g_trace) {
      const double t = trace_now();
      std::fprintf(stderr, "[trace] align: prologue %.1f us, launch calls %.1f us, wait %.1f us (kernel events %.1f us)\n",
                   g_trace_t[1] - g_trace_t[0], g_trace_t[2] - g_trace_t[1], t - g_trace_t[2], 1e3 * h->solve_ms);
    }
    std::memcpy(h->final_T, r.final_T, sizeof(h->final_T));
    h->converged = r.converged;
    h->iterations = r.iterations;
    h->evaluations = r.evaluations;
    h->trans_probability = r.trans_probability;
    h->hits_last = r.hits_last;
    h->hits_total = r.hits_total;
    return B200REG_OK;
  }
  return fail(h, B200REG_ERR_TIMEOUT, "NDT solver did not finish");
}

int gicp_align(b200reg_t h, const float* guess_colmajor) {
  h->converged = 0;
  set_identity(h->final_T);
  if (!h->have_target) return fail(h, B200REG_ERR_NO_TARGET, "align: no input target");
  if (!h->have_source) return fail(h, B200REG_ERR_NO_SOURCE, "align: no input source");
  ensure_nn(h);
  float T[16];
  if (guess_colmajor) col_to_row(guess_colmajor, T);
  else set_identity(T);
  h->gicp.corr_dist = h->corr_dist;
  B200_CUDA(cudaEventRecord(h->ev0, h->stream));
  GicpOutcome out = h->gicp_solver.align(h->nn, h->d_target.ptr, h->n_target, h->src_view, h->n_source, h->gicp, T,
                                         h->stream);
  B200_CUDA(cudaEventRecord(h->ev1, h->stream));
  B200_CUDA(cudaEventSynchronize(h->ev1));
  B200_CUDA(cudaEventElapsedTime(&h->solve_ms, h->ev0, h->ev1));
  std::memcpy(h->final_T, out.final_T, sizeof(h->final_T));
  h->converged = out.converged;
  h->iterations = out.iterations;
  h->evaluations = out.evaluations;
  return B200REG_OK;
}

int set_cloud(b200reg_t h, bool target, const float* base, size_t n, size_t stride, const void* dev) {
  // PCL: empty cloud → PCL_ERROR and the call is ignored (gicp_omp.h:137-141; Registration::setInputTarget)
  if (n == 0 || (!base && !dev)) return fail(h, B200REG_ERR_ARG, "empty input cloud ignored");
  if (!dev && stride < 12) return fail(h, B200REG_ERR_ARG, "stride_bytes must be >= 12");
  DeviceBuffer<float4>& dst = target ? h->d_target : h->d_source;
  if (!dev && (stride % 4) != 0) return fail(h, B200REG_ERR_ARG, "stride_bytes must be a multiple of 4 (float fields)");
  if (dev) {
    dst.ensure(n);
    B200_CUDA(cudaMemcpyAsync(dst.ptr, dev, n * sizeof(float4), cudaMemcpyDeviceToDevice, h->stream));
    // "caller memory may be reused on return" (b200reg.h): the copy runs on the handle's own stream, so wait for it —
    // the producer (a torch allocator, the frontend session's stream) is free to overwrite the buffer afterwards
    B200_CUDA(cudaStreamSynchronize(h->stream));
  } else if (target) {
    dst.ensure(n);
    h->uploader.upload_with_bounds(base, n, stride, -1, 1.0f, dst.ptr, h->stream);  // bounds measured in the unpack pass
    B200_CUDA(cudaStreamSynchronize(h->stream));  // the caller may reuse its buffer: wait for the copy engine
    h->target_bounds = h->uploader.finish_bounds();
  } else {
    upload_cloud(base, n, stride, dst, h->uploader, h->stream);
    // the caller may reuse its buffer (and the staging copy is reused by the next upload): wait for the copy engine
    B200_CUDA(cudaStreamSynchronize(h->stream));
  }
  if (target) {
    h->target_bounds_valid = !dev;
    h->n_target = n;
    h->have_target = true;
    h->map_valid = false;
    h->nn_valid = false;
    h->gicp_solver.invalidate_target();
    if (h->kind == B200REG_NDT) {
      ensure_map(h);  // setInputTarget → init() builds the voxel structure eagerly
      if (h->grid_overflow) return B200REG_ERR_GRID;
    }
  } else {
    h->n_source = n;
    h->have_source = true;
    h->src_view = h->d_source.ptr;
    h->gicp_solver.invalidate_source();
  }
  return B200REG_OK;
}

}  // namespace

extern "C" {

int b200reg_create(int kind, int device, b200reg_t* out) {
  if (!out || (kind != B200REG_NDT && kind != B200REG_GICP)) return B200REG_ERR_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
    cudaGetLastError();
    return B200REG_ERR_CUDA;  // no CPU fallback
  }
  b200reg_engine* h = new b200reg_engine();
  h->kind = kind;
  h->device = device;
  try {
    B200_CUDA(cudaSetDevice(device));
    B200_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    B200_CUDA(cudaEventCreate(&h->ev0));
    B200_CUDA(cudaEventCreate(&h->ev1));
    h->solver.init(device, h->stream);
    h->solver.timing_enabled = getenv("B200REG_TIMING") != nullptr;
    h->solver.batch_profile = getenv("B200REG_BATCH_PROFILE") != nullptr;
    if (const char* se = getenv("B200REG_SWEEP_ENGINES")) h->sweep_engines = std::max(1, std::min(4, atoi(se)));
    h->solver.scalar_controller = getenv("B200REG_SCALAR_CTL") != nullptr;
    h->solver.plain_launch = getenv("B200REG_PLAIN_LAUNCH") != nullptr;
    h->gicp_solver.device_bfgs = getenv("B200REG_GICP_HOST_BFGS") == nullptr;  // developer switch: host-driven BFGS
    h->gicp_solver.init(device, h->stream);
    if (kind == B200REG_GICP) {
      h->corr_dist = 5.0;  // gicp_omp.h:119
    }
    h->scratch_d.ensure(64);
    h->scratch_f.ensure(16);
  } catch (const std::exception&) {
    delete h;
    cudaGetLastError();
    return B200REG_ERR_CUDA;
  }
  *out = h;
  return B200REG_OK;
}

int b200reg_destroy(b200reg_t h) {
  if (!h) return B200REG_ERR_ARG;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  for (b200reg_engine* sib : h->siblings)
    if (sib) b200reg_destroy(sib);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  cudaStream_t s = h->stream;
  delete h;
  if (s) cudaStreamDestroy(s);
  return B200REG_OK;
}

const char* b200reg_last_error(b200reg_t h) { return h ? h->err.c_str() : "null handle"; }

// ---- setters ---------------------------------------------------------------------------------------------
int b200reg_set_transformation_epsilon(b200reg_t h, double eps) {
  if (!h) return B200REG_ERR_ARG;
  h->ndt.trans_eps = eps;
  h->gicp.trans_eps = eps;
  return B200REG_OK;
}
int b200reg_set_maximum_iterations(b200reg_t h, int n) {
  if (!h) return B200REG_ERR_ARG;
  h->ndt.max_iterations = n;
  h->gicp.max_iterations = n;
  return B200REG_OK;
}
int b200reg_set_max_correspondence_distance(b200reg_t h, double d) {
  if (!h) return B200REG_ERR_ARG;
  h->corr_dist = d;
  return B200REG_OK;
}
int b200reg_set_euclidean_fitness_epsilon(b200reg_t h, double eps) {
  if (!h) return B200REG_ERR_ARG;
  h->euclid_eps = eps;
  return B200REG_OK;
}
int b200reg_set_ransac_iterations(b200reg_t h, int n) {
  if (!h) return B200REG_ERR_ARG;
  h->ransac_iters = n;
  return B200REG_OK;
}

int b200reg_ndt_set_resolution(b200reg_t h, float resolution) {
  if (!h || h->kind != B200REG_NDT || !(resolution > 0)) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    if (h->ndt.resolution != resolution) {  // ndt_omp.h:127-137: re-voxelise only when it changes
      h->ndt.resolution = resolution;
      if (h->have_target && h->have_source) {  // reference re-inits `if (input_)`
        ensure_map(h);
        if (h->grid_overflow) return (int)B200REG_ERR_GRID;
      }
    }
    return (int)B200REG_OK;
  });
}
int b200reg_ndt_set_step_size(b200reg_t h, double step) {
  if (!h || h->kind != B200REG_NDT) return B200REG_ERR_ARG;
  h->ndt.step_size = step;
  return B200REG_OK;
}
int b200reg_ndt_set_outlier_ratio(b200reg_t h, double ratio) {
  if (!h || h->kind != B200REG_NDT) return B200REG_ERR_ARG;
  h->ndt.outlier_ratio = ratio;
  return B200REG_OK;
}
int b200reg_ndt_set_neighborhood_search_method(b200reg_t h, int m) {
  if (!h || h->kind != B200REG_NDT || m < 0 || m > 3) return B200REG_ERR_ARG;
  h->ndt.search_method = m;
  return B200REG_OK;
}
int b200reg_ndt_set_num_threads(b200reg_t h, int) { return h ? B200REG_OK : B200REG_ERR_ARG; }
int b200reg_ndt_get_transformation_probability(b200reg_t h, double* out) {
  if (!h || !out) return B200REG_ERR_ARG;
  *out = h->trans_probability;
  return B200REG_OK;
}
int b200reg_ndt_get_final_num_iteration(b200reg_t h, int* out) {
  if (!h || !out) return B200REG_ERR_ARG;
  *out = h->iterations;
  return B200REG_OK;
}

int b200reg_gicp_set_rotation_epsilon(b200reg_t h, double eps) {
  if (!h || h->kind != B200REG_GICP) return B200REG_ERR_ARG;
  h->gicp.rotation_eps = eps;
  return B200REG_OK;
}
int b200reg_gicp_set_correspondence_randomness(b200reg_t h, int k) {
  if (!h || h->kind != B200REG_GICP || k < 3 || k > GICP_MAX_K) return B200REG_ERR_ARG;
  h->gicp.k_correspondences = k;
  h->gicp_solver.invalidate_target();
  h->gicp_solver.invalidate_source();
  return B200REG_OK;
}
int b200reg_gicp_set_maximum_optimizer_iterations(b200reg_t h, int n) {
  if (!h || h->kind != B200REG_GICP) return B200REG_ERR_ARG;
  h->gicp.max_inner_iterations = n;
  return B200REG_OK;
}
int b200reg_gicp_set_epsilon(b200reg_t h, double e) {
  if (!h || h->kind != B200REG_GICP) return B200REG_ERR_ARG;
  h->gicp.gicp_epsilon = e;
  h->gicp_solver.invalidate_target();
  h->gicp_solver.invalidate_source();
  return B200REG_OK;
}

// ---- clouds ----------------------------------------------------------------------------------------------
int b200reg_set_input_target(b200reg_t h, const float* base, size_t n, size_t stride_bytes) {
  return guarded(h, [&]() { return set_cloud(h, true, base, n, stride_bytes, nullptr); });
}
int b200reg_set_input_source(b200reg_t h, const float* base, size_t n, size_t stride_bytes) {
  return guarded(h, [&]() { return set_cloud(h, false, base, n, stride_bytes, nullptr); });
}
int b200reg_set_input_target_device(b200reg_t h, const void* dev, size_t n) {
  return guarded(h, [&]() { return set_cloud(h, true, nullptr, n, 16, dev); });
}
int b200reg_set_input_source_device(b200reg_t h, const void* dev, size_t n) {
  return guarded(h, [&]() { return set_cloud(h, false, nullptr, n, 16, dev); });
}
// Library-internal (not in include/b200reg.h): the frontend session hands over its voxel-filtered scan WITHOUT a copy — the
// buffer stays valid and untouched until the session's next frame, and the session has synchronised its own stream.
int b200reg_adopt_source_device(b200reg_t h, const void* dev, size_t n) {
  if (!h || !dev || n == 0) return B200REG_ERR_ARG;
  h->src_view = static_cast<const float4*>(dev);
  h->n_source = n;
  h->have_source = true;
  h->gicp_solver.invalidate_source();
  return B200REG_OK;
}

// ---- align -----------------------------------------------------------------------------------------------
int b200reg_align(b200reg_t h, const float* guess, float* final_out) {
  return guarded(h, [&]() {
    int rc;
    if (h->kind == B200REG_NDT) {
      rc = ndt_align_begin(h, guess);
      if (rc == B200REG_OK) rc = ndt_align_end(h);
    } else {
      rc = gicp_align(h, guess);
    }
    if (final_out) row_to_col(h->final_T, final_out);
    return rc;
  });
}

int b200reg_align_batch(b200reg_t* handles, int count, const float* guesses, float* finals) {
  if (!handles || count < 0) return B200REG_ERR_ARG;
  int worst = B200REG_OK;
  for (int i = 0; i < count; i++) {
    // one handle after the other: every NDT / GICP solve is a persistent cooperative kernel that owns all SMs, and two
    // such kernels must not be in flight at once (cooperative_launch_mutex) — the entry point is a convenience loop
    b200reg_t h = handles[i];
    if (!h) return B200REG_ERR_ARG;
    const float* g = guesses ? guesses + 16 * i : nullptr;
    const int rc = guarded(h, [&]() {
      if (h->kind != B200REG_NDT) return gicp_align(h, g);
      int r = ndt_align_begin(h, g);
      if (r == B200REG_OK) r = ndt_align_end(h);
      return r;
    });
    if (finals) row_to_col(h->final_T, finals + 16 * i);
    if (rc != B200REG_OK) worst = rc;
  }
  return worst;
}

int b200reg_get_kind(b200reg_t h, int* kind) {
  if (!h || !kind) return B200REG_ERR_ARG;
  *kind = h->kind;
  return B200REG_OK;
}

int b200reg_get_final_transformation(b200reg_t h, float* out16) {
  if (!h || !out16) return B200REG_ERR_ARG;
  row_to_col(h->final_T, out16);
  return B200REG_OK;
}
int b200reg_has_converged(b200reg_t h, int* out) {
  if (!h || !out) return B200REG_ERR_ARG;
  *out = h->converged;
  return B200REG_OK;
}

int b200reg_get_fitness_score(b200reg_t h, double max_range, double* out) {
  if (!h || !out) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    if (!h->have_target) return fail(h, B200REG_ERR_NO_TARGET, "getFitnessScore: no input target");
    if (!h->have_source) return fail(h, B200REG_ERR_NO_SOURCE, "getFitnessScore: no input source");
    ensure_nn(h);
    h->nn_idx.ensure(h->n_source);
    h->nn_d2.ensure(h->n_source);
    // points farther than max_range do not contribute: let the search stop there
    const float bound = (max_range < 3.0e38) ? (float)max_range * 1.0001f + 1e-30f : 3.402823466e+38f;
    nn1_query(h->nn, h->src_view, h->n_source, h->final_T, h->nn_idx.ptr, h->nn_d2.ptr, h->stream, bound);
    double sum = 0;
    long long cnt = 0;
    fitness_reduce(h->nn_d2.ptr, h->nn_idx.ptr, h->n_source, max_range, h->scratch_d.ptr, &sum, &cnt, h->stream);
    h->other_launches += 2;
    *out = cnt > 0 ? sum / (double)cnt : DBL_MAX;
    return (int)B200REG_OK;
  });
}

int b200reg_get_aligned(b200reg_t h, float* out, size_t stride_bytes) {
  if (!h || !out || stride_bytes < 12 || (stride_bytes % 4) != 0) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    if (!h->have_source) return fail(h, B200REG_ERR_NO_SOURCE, "no input source");
    h->d_aligned.ensure(h->n_source);
    B200_CUDA(cudaMemcpyAsync(h->scratch_f.ptr, h->final_T, 12 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    transform_cloud_device(h->src_view, h->n_source, h->d_aligned.ptr, h->scratch_f.ptr, h->stream);
    h->other_launches += 1;
    h->staging.ensure(h->n_source);
    B200_CUDA(cudaMemcpyAsync(h->staging.ptr, h->d_aligned.ptr, h->n_source * sizeof(float4), cudaMemcpyDeviceToHost,
                              h->stream));
    B200_CUDA(cudaStreamSynchronize(h->stream));
    char* b = reinterpret_cast<char*>(out);
    for (size_t i = 0; i < h->n_source; i++) {
      float* f = reinterpret_cast<float*>(b + i * stride_bytes);
      f[0] = h->staging.ptr[i].x;
      f[1] = h->staging.ptr[i].y;
      f[2] = h->staging.ptr[i].z;
      if (stride_bytes >= 16) f[3] = 1.0f;
    }
    return (int)B200REG_OK;
  });
}

// ---- VoxelGrid ---------------------------------------------------------------------------------------------
int b200reg_voxelgrid(int device, const float* in, size_t n, size_t stride_bytes, long intensity_offset_bytes, float leaf,
                      float* out, size_t out_capacity, size_t* m) {
  if (!in || !out || !m || stride_bytes < 12 || (stride_bytes % 4) != 0 || !(leaf > 0) ||
      (intensity_offset_bytes >= 0 && (intensity_offset_bytes % 4) != 0))
    return B200REG_ERR_ARG;  // float fields: records and offsets are 4-byte aligned
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  try {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
      cudaGetLastError();
      return B200REG_ERR_CUDA;
    }
    B200_CUDA(cudaSetDevice(device));
    static VoxelGridFilter* filters[64] = {nullptr};
    static cudaStream_t streams[64] = {nullptr};
    if (device >= 64) return B200REG_ERR_ARG;
    if (!filters[device]) {
      filters[device] = new VoxelGridFilter();
      B200_CUDA(cudaStreamCreateWithFlags(&streams[device], cudaStreamNonBlocking));
    }
    VoxelGridFilter& F = *filters[device];
    F.dense_word_budget = g_vg_dense_budget;
    cudaStream_t s = streams[device];
    *m = 0;
    if (n == 0) return B200REG_OK;
    F.in.ensure(n);
    static CloudUploader* uploaders[64] = {nullptr};
    if (!uploaders[device]) uploaders[device] = new CloudUploader();
    const char* b = reinterpret_cast<const char*>(in);
    uploaders[device]->upload(in, n, stride_bytes, intensity_offset_bytes, 0.0f, F.in.ptr, s);  // raw records, unpacked on the device
    long long cnt = F.filter_device(F.in.ptr, n, leaf, s);
    char* ob = reinterpret_cast<char*>(out);
    if (cnt < 0) {  // overflow guard: PCL returns the input cloud unchanged
      size_t k = std::min(n, out_capacity);
      for (size_t i = 0; i < k; i++) std::memcpy(ob + i * stride_bytes, b + i * stride_bytes, stride_bytes);
      *m = n;
      return B200REG_OK;
    }
    size_t mm = (size_t)cnt;
    F.staging.ensure(std::max(mm, n));
    B200_CUDA(cudaMemcpyAsync(F.staging.ptr, F.out.ptr, mm * sizeof(float4), cudaMemcpyDeviceToHost, s));
    B200_CUDA(cudaStreamSynchronize(s));
    size_t k = std::min(mm, out_capacity);
    for (size_t i = 0; i < k; i++) {
      float* f = reinterpret_cast<float*>(ob + i * stride_bytes);
      const float4 v = F.staging.ptr[i];
      f[0] = v.x;
      f[1] = v.y;
      f[2] = v.z;
      if (intensity_offset_bytes >= 0) *reinterpret_cast<float*>(ob + i * stride_bytes + intensity_offset_bytes) = v.w;
      if (stride_bytes >= 32 || (stride_bytes >= 16 && intensity_offset_bytes != 12)) f[3] = 1.0f;
    }
    *m = mm;
    return B200REG_OK;
  } catch (const std::exception&) {
    cudaGetLastError();
    return B200REG_ERR_CUDA;
  }
}

// ---- introspection -----------------------------------------------------------------------------------------
int b200reg_get_stats(b200reg_t h, b200reg_stats* out) {
  if (!h || !out) return B200REG_ERR_ARG;
  std::memset(out, 0, sizeof(*out));
  out->evaluations = h->evaluations;
  out->iterations = h->iterations;
  out->hits = h->hits_last;
  out->hits_total = h->hits_total;
  out->solve_ms = h->solve_ms;
  out->target_build_ms = h->target_build_ms;
  out->kernel_launches = h->solver.launches + h->map.launches + h->nn.launches + h->gicp_solver.launches + h->other_launches;
  out->grid_ctas = h->solver.grid_ctas();
  out->block_threads = h->solver.block_threads();
  out->index_in_smem = h->solver.index_in_smem();
  out->n_voxels = (long long)h->map.n_voxels;
  out->n_cells = h->map.geom.n_cells;
  out->n_source = (long long)h->n_source;
  out->n_target = (long long)h->n_target;
  out->gicp_inner_ms = h->gicp_solver.inner_ms;
  out->gicp_inner_launches = h->gicp_solver.inner_launches;
  out->gicp_pair_evaluations = h->gicp_solver.inner_pair_evaluations;
  return B200REG_OK;
}

int b200reg_ndt_derivatives(b200reg_t h, const float* T, const double* p6, int compute_hessian, double* score, double* g6,
                            double* H36) {
  if (!h || h->kind != B200REG_NDT || !T || !p6) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    if (!h->have_target) return fail(h, B200REG_ERR_NO_TARGET, "no input target");
    if (!h->have_source) return fail(h, B200REG_ERR_NO_SOURCE, "no input source");
    ensure_map(h);
    if (h->map.n_voxels == 0) {
      if (score) *score = 0;
      if (g6) std::memset(g6, 0, 6 * sizeof(double));
      if (H36) std::memset(H36, 0, 36 * sizeof(double));
      h->hits_last = 0;
      return (int)B200REG_OK;
    }
    float Tr[16];
    col_to_row(T, Tr);
    {
      std::lock_guard<std::mutex> coop(cooperative_launch_mutex(h->device));
      B200_CUDA(cudaEventRecord(h->ev0, h->stream));
      h->solver.launch(h->map, h->src_view, h->n_source, h->ndt, NDT_MODE_DERIVATIVES, Tr, p6, compute_hessian, 0);
      B200_CUDA(cudaEventRecord(h->ev1, h->stream));
      B200_CUDA(cudaStreamSynchronize(h->stream));
    }
    B200_CUDA(cudaEventElapsedTime(&h->solve_ms, h->ev0, h->ev1));
    if (h->solver.result().error == 3) h->solver.fetch_result();
    const NdtResult& r = h->solver.result();
    if (r.error != 0) {
      h->solver.reset_barrier();
      B200_CUDA(cudaStreamSynchronize(h->stream));
      return fail(h, B200REG_ERR_TIMEOUT, "NDT derivative kernel watchdog fired");
    }
    if (score) *score = r.score;
    if (g6) std::memcpy(g6, r.g, sizeof(r.g));
    if (H36) std::memcpy(H36, r.H, sizeof(r.H));
    h->hits_last = r.hits_last;
    h->hits_total = r.hits_total;
    h->evaluations = r.evaluations;
    return (int)B200REG_OK;
  });
}

int b200reg_ndt_hessian_radius(b200reg_t h, const float* T, const double* p6, double* H36) {
  if (!h || h->kind != B200REG_NDT || !T || !p6 || !H36) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    if (!h->have_target) return fail(h, B200REG_ERR_NO_TARGET, "no input target");
    if (!h->have_source) return fail(h, B200REG_ERR_NO_SOURCE, "no input source");
    ensure_map(h);
    std::memset(H36, 0, 36 * sizeof(double));
    if (h->map.n_voxels == 0) return (int)B200REG_OK;
    float Tr[16], ja[24], ha[45];
    double tabs[69];
    col_to_row(T, Tr);
    angle_tables(p6, ja, ha, tabs, tabs + 24);
    h->scratch_d.ensure(128);
    B200_CUDA(cudaMemcpyAsync(h->scratch_d.ptr + 32, tabs, sizeof(tabs), cudaMemcpyHostToDevice, h->stream));
    B200_CUDA(cudaMemcpyAsync(h->scratch_f.ptr, Tr, 12 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    ndt_hessian_radius(h->map, h->src_view, h->n_source, h->ndt, h->scratch_f.ptr, h->scratch_d.ptr + 32,
                       h->scratch_d.ptr + 56, h->scratch_d.ptr, h->stream);
    h->other_launches += 1;
    double up[21];
    B200_CUDA(cudaMemcpyAsync(up, h->scratch_d.ptr, sizeof(up), cudaMemcpyDeviceToHost, h->stream));
    B200_CUDA(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < 6; i++)
      for (int j = i; j < 6; j++) H36[i * 6 + j] = H36[j * 6 + i] = up[tri_index(i, j)];
    return (int)B200REG_OK;
  });
}

int b200reg_ndt_calculate_score(b200reg_t h, const float* base, size_t n, size_t stride_bytes, double* out) {
  if (!h || h->kind != B200REG_NDT || !base || !out || stride_bytes < 12 || (stride_bytes % 4) != 0) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    if (!h->have_target) return fail(h, B200REG_ERR_NO_TARGET, "no input target");
    ensure_map(h);
    *out = 0;
    if (n == 0 || h->map.n_voxels == 0) return (int)B200REG_OK;
    upload_cloud(base, n, stride_bytes, h->query_buf, h->uploader, h->stream);
    ndt_score(h->map, h->query_buf.ptr, n, h->ndt, h->scratch_d.ptr, h->stream);
    h->other_launches += 1;
    double s = 0;
    B200_CUDA(cudaMemcpyAsync(&s, h->scratch_d.ptr, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    B200_CUDA(cudaStreamSynchronize(h->stream));
    *out = s / (double)n;
    return (int)B200REG_OK;
  });
}

int b200reg_ndt_num_voxels(b200reg_t h, size_t* out) {
  if (!h || !out) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    if (!h->have_target) return fail(h, B200REG_ERR_NO_TARGET, "no input target");
    ensure_map(h);
    *out = h->map.n_voxels;
    return (int)B200REG_OK;
  });
}

int b200reg_ndt_get_voxels(b200reg_t h, int* leaf_idx, int* npts, double* mean3, double* icov9, float* centroid3) {
  if (!h) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    if (!h->have_target) return fail(h, B200REG_ERR_NO_TARGET, "no input target");
    ensure_map(h);
    const size_t V = h->map.n_voxels;
    if (V == 0) return (int)B200REG_OK;
    std::vector<VoxelRecord> rec(V);
    std::vector<float4> cen(V);
    B200_CUDA(cudaMemcpyAsync(rec.data(), h->map.records.ptr, V * sizeof(VoxelRecord), cudaMemcpyDeviceToHost, h->stream));
    B200_CUDA(cudaMemcpyAsync(cen.data(), h->map.centroids.ptr, V * sizeof(float4), cudaMemcpyDeviceToHost, h->stream));
    if (npts) B200_CUDA(cudaMemcpyAsync(npts, h->map.npts.ptr, V * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    if (icov9)
      B200_CUDA(cudaMemcpyAsync(icov9, h->map.icov_d.ptr, V * 9 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    B200_CUDA(cudaStreamSynchronize(h->stream));
    for (size_t v = 0; v < V; v++) {
      if (mean3) {
        mean3[3 * v + 0] = record_mean(rec[v], 0);
        mean3[3 * v + 1] = record_mean(rec[v], 1);
        mean3[3 * v + 2] = record_mean(rec[v], 2);
      }
      if (centroid3) {
        centroid3[3 * v + 0] = cen[v].x;
        centroid3[3 * v + 1] = cen[v].y;
        centroid3[3 * v + 2] = cen[v].z;
      }
      if (leaf_idx) std::memcpy(&leaf_idx[v], &cen[v].w, sizeof(int));
    }
    return (int)B200REG_OK;
  });
}

// developer / test hook, not part of include/b200reg.h: size budget (8-byte words) up to which b200reg_voxelgrid uses the
// dense occupancy bitmap; beyond it the two-level sparse index (voxelgrid.cu). 0 forces the sparse path.
int b200reg_debug_set_voxelgrid_dense_budget(size_t words) {
  g_vg_dense_budget = words;
  return B200REG_OK;
}

// developer instrumentation, not part of include/b200reg.h: per-round phase stamps of the last solver launch
int b200reg_debug_timing(b200reg_t h, unsigned long long* out48x8) {
  if (!h || !out48x8) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    h->solver.read_timing(out48x8);
    return (int)B200REG_OK;
  });
}

int b200reg_debug_cta_eval_ns(b200reg_t h, unsigned* out, int n) {
  if (!h || !out) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    h->solver.read_cta_eval_ns(out, n);
    return (int)B200REG_OK;
  });
}

int b200reg_gicp_get_covariances(b200reg_t h, int which, double* out9, size_t* n) {
  if (!h || h->kind != B200REG_GICP || !n) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    std::vector<double> tmp;
    *n = h->gicp_solver.covariances(which, tmp, h->stream);
    if (out9 && !tmp.empty()) std::memcpy(out9, tmp.data(), tmp.size() * sizeof(double));
    return (int)B200REG_OK;
  });
}
int b200reg_gicp_num_correspondences(b200reg_t h, int* out) {
  if (!h || h->kind != B200REG_GICP || !out) return B200REG_ERR_ARG;
  *out = h->gicp_solver.last_correspondences();
  return B200REG_OK;
}

int b200reg_nn1(b200reg_t h, const float* base, size_t n, size_t stride_bytes, int* idx, float* d2) {
  if (!h || !base || !idx || !d2 || stride_bytes < 12 || (stride_bytes % 4) != 0) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    if (!h->have_target) return fail(h, B200REG_ERR_NO_TARGET, "no input target");
    if (n == 0) return (int)B200REG_OK;
    ensure_nn(h);
    upload_cloud(base, n, stride_bytes, h->query_buf, h->uploader, h->stream);
    h->nn_idx.ensure(n);
    h->nn_d2.ensure(n);
    nn1_query(h->nn, h->query_buf.ptr, n, nullptr, h->nn_idx.ptr, h->nn_d2.ptr, h->stream);
    h->other_launches += 1;
    B200_CUDA(cudaMemcpyAsync(idx, h->nn_idx.ptr, n * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    B200_CUDA(cudaMemcpyAsync(d2, h->nn_d2.ptr, n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    B200_CUDA(cudaStreamSynchronize(h->stream));
    return (int)B200REG_OK;
  });
}

}  // extern "C"

// ---- batched NDT registration: K independent scans against the current target in ONE persistent launch --------------
namespace {
// cuStreamWriteValue32 (driver API), bound at run time: a 32-bit store into device memory performed by the stream when it
// gets there — the copy stream marks "scan k has arrived" with it while the persistent solver kernel is already running
using StreamWriteValue32 = int (*)(cudaStream_t, unsigned long long, unsigned, unsigned);
StreamWriteValue32 stream_write_value32() {
  static StreamWriteValue32 fn = []() -> StreamWriteValue32 {
    if (getenv("B200REG_NO_STREAM_MEMOPS")) return nullptr;  // developer switch: upload everything first
    // The streaming form lets the solver kernel wait for data another stream is still delivering. Tools that serialise
    // the device (Nsight Compute replays one kernel at a time, compute-sanitizer, CUDA_LAUNCH_BLOCKING=1) would keep that
    // kernel spinning until its watchdog fires: under them everything is uploaded before the launch.
    const char* blocking = getenv("CUDA_LAUNCH_BLOCKING");
    if ((blocking && blocking[0] && blocking[0] != '0') || getenv("CUDA_INJECTION64_PATH") || getenv("NV_NSIGHT_INJECTION_PORT_BASE") ||
        getenv("NV_COMPUTE_PROFILER_PERFWORKS_DIR") || getenv("NVTX_INJECTION64_PATH"))
      return nullptr;
    void* lib = dlopen("libcuda.so.1", RTLD_NOW);
    if (!lib) return nullptr;
    void* p = dlsym(lib, "cuStreamWriteValue32_v2");
    if (!p) p = dlsym(lib, "cuStreamWriteValue32");
    return reinterpret_cast<StreamWriteValue32>(p);
  }();
  return fn;
}

bool batch_needs_sequential(b200reg_t h) {
  // One launch cannot serve: an empty map (the reference returns the guess), or a configuration whose line search runs
  // the More-Thuente inner loop (step_max <= step_min: it leaves the kernel for the f64 radius Hessian) — those take
  // the single-registration path one by one.
  return h->map.n_voxels == 0 || !((h->ndt.step_size - h->ndt.trans_eps / 2) > 0) || h->solver.timing_enabled;
}

// items: device-resident sources + row-major guesses, already in h->batch_items. after_launch (optional) runs on the host
// right after the solver launch of a chunk has been enqueued (the streaming upload of b200reg_ndt_align_batch).
int ndt_batch_run(b200reg_t h, int count, b200reg_batch_result* results, const std::function<void()>& after_launch = nullptr) {
  if (!h->have_target) return fail(h, B200REG_ERR_NO_TARGET, "align_batch: no input target");
  ensure_map(h);
  std::vector<NdtSolver::BatchItem>& items = h->batch_items;
  auto store = [&](int k, const float* T_row, int converged, int iterations, int evaluations, double tp, long long hits,
                   int status) {
    b200reg_batch_result& r = results[k];
    row_to_col(T_row, r.final_T);
    r.trans_probability = tp;
    r.converged = converged;
    r.iterations = iterations;
    r.evaluations = evaluations;
    r.status = status;
    r.hits_total = hits;
  };
  long long evals = 0, hits = 0;
  const bool sequential = batch_needs_sequential(h);
  if (sequential && h->board)
    return fail(h, B200REG_ERR_ARG, "align_batch with a pose board attached needs the one-launch path (non-empty map, step_size > transformation_epsilon / 2)");
  if (sequential) {
    int worst = B200REG_OK;
    float ms = 0;
    for (int k = 0; k < count; k++) {
      h->d_source.ensure(items[k].n_src);
      B200_CUDA(cudaMemcpyAsync(h->d_source.ptr, items[k].src, items[k].n_src * sizeof(float4), cudaMemcpyDeviceToDevice, h->stream));
      h->src_view = h->d_source.ptr;
      h->n_source = items[k].n_src;
      h->have_source = true;
      float Tc[16];
      row_to_col(items[k].T_rowmajor16, Tc);
      int rc = ndt_align_begin(h, Tc);
      if (rc == B200REG_OK) rc = ndt_align_end(h);
      store(k, h->final_T, h->converged, h->iterations, h->evaluations, h->trans_probability, h->hits_total, rc);
      evals += h->evaluations;
      hits += h->hits_total;
      ms += h->solve_ms;
      if (rc != B200REG_OK) worst = rc;
    }
    h->evaluations = (int)evals;
    h->hits_total = hits;
    h->solve_ms = ms;
    return worst;
  }
  // sequence numbers bound the rounds one slot may run inside a launch: chunk the batch accordingly
  const int per_launch = std::max(1, NdtSolver::kMaxRoundsPerLaunch / (h->ndt.max_iterations + 4));
  int worst = B200REG_OK;
  float ms_total = 0;
  h->board_valid = 0;
  if (h->board && (count > per_launch || count > h->board->view.rows || count == 0))
    return fail(h, B200REG_ERR_ARG, "align_batch with a pose board attached: 1 .. min(board rows, one launch) registrations per call");
  for (int first = 0; first < count; first += per_launch) {
    const int n = std::min(per_launch, count - first);
    const double tr0 = g_trace ? trace_now() : 0;
    double tr1 = 0, tr2 = 0;
    {
      std::lock_guard<std::mutex> coop(cooperative_launch_mutex(h->device));
      B200_CUDA(cudaEventRecord(h->ev0, h->stream));
      if (h->board) h->board->view.tag += 1;  // every rank of the board makes the same sequence of batch calls
      h->solver.launch_batch(h->map, items.data() + first, n, h->ndt, h->batch_slots, h->board);
      B200_CUDA(cudaEventRecord(h->ev1, h->stream));
      if (g_trace) tr1 = trace_now();
      if (after_launch) after_launch();
      if (g_trace) tr2 = trace_now();
      // The collect kernel goes in behind ev1 (solve_ms stays the solver kernel's own time) and only AFTER the streaming
      // uploads have been issued and drained: a launch parked behind the solver could otherwise sit in front of the
      // copy stream's memory operations on a shared hardware queue while the solver still waits for exactly those.
      if (h->board) h->solver.launch_board_collect(h->board);
      B200_CUDA(cudaStreamSynchronize(h->stream));
    }
    if (g_trace) {
      float kms = 0;
      cudaEventElapsedTime(&kms, h->ev0, h->ev1);
      std::fprintf(stderr, "[trace] batch of %d: job table + launch calls %.1f us, uploads issued %.1f us, wait %.1f us (kernel events %.1f us)\n", n,
                   tr1 - tr0, tr2 - tr1, trace_now() - tr2, 1e3 * kms);
    }
    float ms = 0;
    B200_CUDA(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    ms_total += ms;
    const NdtResult* R = h->solver.batch_results();
    bool failed = false;
    for (int k = 0; k < n; k++) {
      const NdtResult& r = R[k];
      if (r.error != 0) {
        failed = true;
        float I[16];
        set_identity(I);
        store(first + k, I, 0, 0, 0, 0.0, 0, B200REG_ERR_TIMEOUT);
        continue;
      }
      store(first + k, r.final_T, r.converged, r.iterations, r.evaluations, r.trans_probability, r.hits_total, B200REG_OK);
      evals += r.evaluations;
      hits += r.hits_total;
    }
    if (failed) {
      h->solver.reset_barrier();
      B200_CUDA(cudaStreamSynchronize(h->stream));
      worst = fail(h, B200REG_ERR_TIMEOUT, "NDT batch solver: a registration did not finish (device watchdog)");
    }
    if (h->board && !failed) {
      if (h->board->h_counts[h->board->view.world] != 0)
        worst = fail(h, B200REG_ERR_TIMEOUT, "pose board: a peer's poses did not arrive (did every rank make this batch call?)");
      else
        h->board_valid = 1;
    }
  }
  // the handle's "last align" state = the last registration of the batch
  if (count > 0 && results[count - 1].status == B200REG_OK) {
    col_to_row(results[count - 1].final_T, h->final_T);
    h->converged = results[count - 1].converged;
    h->iterations = results[count - 1].iterations;
    h->trans_probability = results[count - 1].trans_probability;
  }
  h->evaluations = (int)evals;
  h->hits_total = hits;
  h->solve_ms = ms_total;
  return worst;
}
}  // namespace

extern "C" {

int b200reg_ndt_align_batch_device(b200reg_t h, int count, const void* const* dev_sources, const size_t* n_points,
                                   const float* guesses, b200reg_batch_result* results) {
  if (!h || h->kind != B200REG_NDT || count < 0 || (count > 0 && (!dev_sources || !n_points || !results))) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    h->batch_items.resize((size_t)count);
    for (int k = 0; k < count; k++) {
      if (!dev_sources[k] || n_points[k] == 0) return fail(h, B200REG_ERR_ARG, "align_batch: empty source cloud");
      NdtSolver::BatchItem& it = h->batch_items[k];
      it.src = dev_sources[k];
      it.n_src = n_points[k];
      it.stride = 0;
      it.ready = nullptr;
      it.ready_tag = 0;
      if (guesses) col_to_row(guesses + 16 * k, it.T_rowmajor16);
      else set_identity(it.T_rowmajor16);
    }
    return ndt_batch_run(h, count, results);
  });
}

int b200reg_ndt_align_batch(b200reg_t h, int count, const float* const* sources, const size_t* n_points, size_t stride_bytes,
                            const float* guesses, b200reg_batch_result* results) {
  if (!h || h->kind != B200REG_NDT || count < 0 || (count > 0 && (!sources || !n_points || !results))) return B200REG_ERR_ARG;
  if (stride_bytes < 12 || (stride_bytes % 4) != 0) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    if (!h->have_target) return fail(h, B200REG_ERR_NO_TARGET, "align_batch: no input target");
    ensure_map(h);
    size_t total = 0, raw_total = 0;
    bool pageable = false;
    std::vector<char> pinned((size_t)count);
    std::vector<size_t> raw_off((size_t)count);
    for (int k = 0; k < count; k++) {
      if (!sources[k] || n_points[k] == 0) return fail(h, B200REG_ERR_ARG, "align_batch: empty source cloud");
      total += n_points[k];
      raw_off[k] = raw_total;
      raw_total += (n_points[k] * stride_bytes + 255) & ~(size_t)255;
      pinned[k] = CloudUploader::is_pinned(sources[k]) ? 1 : 0;
      pageable = pageable || !pinned[k];
    }
    h->batch_uploader.reserve(raw_total, pageable);
    h->batch_items.resize((size_t)count);
    for (int k = 0; k < count; k++) {
      NdtSolver::BatchItem& it = h->batch_items[k];
      it.n_src = n_points[k];
      if (guesses) col_to_row(guesses + 16 * k, it.T_rowmajor16);
      else set_identity(it.T_rowmajor16);
      it.stride = 0;
      it.ready = nullptr;
      it.ready_tag = 0;
    }
    const int per_launch = std::max(1, NdtSolver::kMaxRoundsPerLaunch / (h->ndt.max_iterations + 4));
    StreamWriteValue32 write_value = stream_write_value32();
    if (write_value && !batch_needs_sequential(h) && count <= per_launch) {
      // Streaming form: the solver kernel is launched FIRST and reads the caller's records as they are (no unpack pass);
      // the scans follow on a second stream, each DMA trailed by a stream memory operation that raises the scan's ready
      // flag. Registration k starts as soon as scan k is there, so the upload of the later scans (and, for pageable
      // memory, the CPU staging copy) is hidden behind the registration of the earlier ones.
      if (!h->copy_stream) B200_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
      h->batch_ready.ensure((size_t)count);
      const unsigned tag = ++h->batch_tag;
      for (int k = 0; k < count; k++) {
        NdtSolver::BatchItem& it = h->batch_items[k];
        it.src = h->batch_uploader.raw.ptr + raw_off[k];
        it.stride = (int)stride_bytes;
        it.ready = h->batch_ready.ptr + k;
        it.ready_tag = tag;
      }
      bool copy_failed = false;
      auto upload = [&]() {
        for (int k = 0; k < count && !copy_failed; k++) {
          h->batch_uploader.copy_at(sources[k], pinned[k] != 0, n_points[k] * stride_bytes, raw_off[k], h->copy_stream);
          if (write_value(h->copy_stream, (unsigned long long)(uintptr_t)(h->batch_ready.ptr + k), tag, 0) != 0) copy_failed = true;
        }
        if (copy_failed) {  // never leave the kernel waiting: raise the remaining flags from the host path
          std::vector<unsigned> tags((size_t)count, tag);
          cudaStreamSynchronize(h->copy_stream);
          cudaMemcpyAsync(h->batch_ready.ptr, tags.data(), sizeof(unsigned) * count, cudaMemcpyHostToDevice, h->copy_stream);
        }
        B200_CUDA(cudaStreamSynchronize(h->copy_stream));  // the caller may reuse its buffers on return
      };
      return ndt_batch_run(h, count, results, upload);
    }
    // fallback: upload + unpack everything, then register
    h->d_batch.ensure(total);
    size_t off = 0;
    for (int k = 0; k < count; k++) {  // copies and unpack kernels stream back to back; nothing waits in between
      h->batch_uploader.upload_at(sources[k], pinned[k] != 0, n_points[k], stride_bytes, -1, 1.0f, h->d_batch.ptr + off, raw_off[k],
                                  h->stream);
      h->batch_items[k].src = h->d_batch.ptr + off;
      off += n_points[k];
    }
    h->other_launches += count;
    return ndt_batch_run(h, count, results);
  });
}

int b200reg_ndt_attach_pose_board(b200reg_t h, b200comm_board* board) {
  if (!h || h->kind != B200REG_NDT) return B200REG_ERR_ARG;
  if (board && board->device != h->device) return fail(h, B200REG_ERR_ARG, "attach_pose_board: the board lives on another device");
  h->board = board;
  h->board_valid = 0;
  return B200REG_OK;
}

int b200reg_ndt_gathered_poses(b200reg_t h, float* poses, int* counts, int max_rows) {
  if (!h || h->kind != B200REG_NDT || !poses || !counts || max_rows < 0) return B200REG_ERR_ARG;
  if (!h->board || !h->board_valid) return fail(h, B200REG_ERR_ARG, "gathered_poses: no finished batch call with a pose board attached");
  const b200::PoseBoardView& B = h->board->view;
  for (int r = 0; r < B.world; r++) {
    const int n = h->board->h_counts[r];
    counts[r] = n;
    if (n > max_rows) return fail(h, B200REG_ERR_ARG, "gathered_poses: max_rows is smaller than a rank's count");
    for (int k = 0; k < n; k++) row_to_col(h->board->h_rows + ((size_t)r * B.rows + k) * 16, poses + ((size_t)r * max_rows + k) * 16);
  }
  return B200REG_OK;
}

int b200reg_ndt_set_batch_slots(b200reg_t h, int slots) {
  if (!h || slots < 1) return B200REG_ERR_ARG;
  h->batch_slots = slots;
  return B200REG_OK;
}

}  // extern "C"

// ---- batched GICP registration: K independent scans against the current target, lock-step outer loops ----------------
namespace {
// items: device-resident float4 sources + row-major guesses
int gicp_batch_run(b200reg_t h, int count, const std::vector<GicpBatchItem>& items, b200reg_gicp_batch_result* results) {
  for (int k = 0; k < count; k++) {  // what a registration that never ran reports
    std::memset(&results[k], 0, sizeof(results[k]));
    set_identity(results[k].final_T);
    results[k].status = B200REG_ERR_NO_TARGET;
  }
  if (!h->have_target) return fail(h, B200REG_ERR_NO_TARGET, "gicp_align_batch: no input target");
  if (count == 0) return B200REG_OK;
  ensure_nn(h);
  h->gicp.corr_dist = h->corr_dist;
  std::vector<GicpBatchOutcome> out((size_t)count);
  const int slots = std::min(h->batch_slots, GICP_MAX_SLOTS);
  B200_CUDA(cudaEventRecord(h->ev0, h->stream));
  h->gicp_solver.align_batch(h->nn, h->d_target.ptr, h->n_target, items.data(), count, h->gicp, slots, h->stream, out.data());
  B200_CUDA(cudaEventRecord(h->ev1, h->stream));
  B200_CUDA(cudaEventSynchronize(h->ev1));
  B200_CUDA(cudaEventElapsedTime(&h->solve_ms, h->ev0, h->ev1));
  int worst = B200REG_OK;
  long long evals = 0;
  for (int k = 0; k < count; k++) {
    b200reg_gicp_batch_result& r = results[k];
    const GicpBatchOutcome& o = out[k];
    if (o.timed_out) {
      r.status = B200REG_ERR_TIMEOUT;
      worst = fail(h, B200REG_ERR_TIMEOUT, "GICP batch: the inner-loop kernel watchdog fired");
      continue;
    }
    row_to_col(o.final_T, r.final_T);
    r.converged = o.converged;
    r.iterations = o.iterations;
    r.evaluations = o.evaluations;
    r.correspondences = o.correspondences;
    r.status = B200REG_OK;
    evals += o.evaluations;
  }
  // the handle's "last align" state = the last registration of the batch
  if (count > 0 && results[count - 1].status == B200REG_OK) {
    std::memcpy(h->final_T, out[count - 1].final_T, sizeof(h->final_T));
    h->converged = out[count - 1].converged;
    h->iterations = out[count - 1].iterations;
  }
  h->evaluations = (int)evals;
  return worst;
}
}  // namespace

extern "C" {

int b200reg_gicp_align_batch_device(b200reg_t h, int count, const void* const* dev_sources, const size_t* n_points,
                                    const float* guesses, b200reg_gicp_batch_result* results) {
  if (!h || h->kind != B200REG_GICP || count < 0 || (count > 0 && (!dev_sources || !n_points || !results))) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    std::vector<GicpBatchItem> items((size_t)count);
    for (int k = 0; k < count; k++) {
      if (!dev_sources[k] || n_points[k] == 0) return fail(h, B200REG_ERR_ARG, "gicp_align_batch: empty source cloud");
      items[k].src = static_cast<const float4*>(dev_sources[k]);
      items[k].n = n_points[k];
      if (guesses) col_to_row(guesses + 16 * k, items[k].guess);
      else set_identity(items[k].guess);
    }
    return gicp_batch_run(h, count, items, results);
  });
}

int b200reg_gicp_align_batch(b200reg_t h, int count, const float* const* sources, const size_t* n_points, size_t stride_bytes,
                             const float* guesses, b200reg_gicp_batch_result* results) {
  if (!h || h->kind != B200REG_GICP || count < 0 || (count > 0 && (!sources || !n_points || !results))) return B200REG_ERR_ARG;
  if (stride_bytes < 12 || (stride_bytes % 4) != 0) return B200REG_ERR_ARG;
  return guarded(h, [&]() {
    size_t total = 0, raw_total = 0;
    bool pageable = false;
    std::vector<char> pinned((size_t)count);
    std::vector<size_t> raw_off((size_t)count);
    for (int k = 0; k < count; k++) {
      if (!sources[k] || n_points[k] == 0) return fail(h, B200REG_ERR_ARG, "gicp_align_batch: empty source cloud");
      total += n_points[k];
      raw_off[k] = raw_total;
      raw_total += (n_points[k] * stride_bytes + 255) & ~(size_t)255;
      pinned[k] = CloudUploader::is_pinned(sources[k]) ? 1 : 0;
      pageable = pageable || !pinned[k];
    }
    if (!h->have_target) return gicp_batch_run(h, count, {}, results);
    // upload + unpack every source back to back into one device buffer, nothing waits in between
    h->batch_uploader.reserve(raw_total, pageable);
    h->d_batch.ensure(total);
    std::vector<GicpBatchItem> items((size_t)count);
    size_t off = 0;
    for (int k = 0; k < count; k++) {
      h->batch_uploader.upload_at(sources[k], pinned[k] != 0, n_points[k], stride_bytes, -1, 1.0f, h->d_batch.ptr + off, raw_off[k],
                                  h->stream);
      items[k].src = h->d_batch.ptr + off;
      items[k].n = n_points[k];
      if (guesses) col_to_row(guesses + 16 * k, items[k].guess);
      else set_identity(items[k].guess);
      off += n_points[k];
    }
    h->other_launches += count;
    return gicp_batch_run(h, count, items, results);
  });
}

}  // extern "C"

// ---- loop-closure candidate sweep on one GPU (generalises gbs.cpp:187-233 from the arg-min candidate to all of them) ----
namespace {
int sweep_one(b200reg_t e, const float* src, size_t n_src, const float* tgt, size_t n_tgt, size_t stride, const float* guess,
              double max_range, b200reg_sweep_result* out) {
  std::memset(out, 0, sizeof(*out));
  set_identity(out->final_T);
  out->fitness = DBL_MAX;
  return guarded(e, [&]() {
    int rc = set_cloud(e, true, tgt, n_tgt, stride, nullptr);   // setInputTarget: upload + voxel map (gbs.cpp:227)
    if (rc == B200REG_OK) rc = set_cloud(e, false, src, n_src, stride, nullptr);  // setInputSource (gbs.cpp:181)
    if (rc == B200REG_OK) rc = ndt_align_begin(e, guess);       // align (gbs.cpp:230)
    if (rc == B200REG_OK) rc = ndt_align_end(e);
    row_to_col(e->final_T, out->final_T);
    out->converged = e->converged;
    out->iterations = e->iterations;
    out->trans_probability = e->trans_probability;
    if (rc == B200REG_OK) {                                     // getFitnessScore (gbs.cpp:231)
      ensure_nn(e);
      e->nn_idx.ensure(e->n_source);
      e->nn_d2.ensure(e->n_source);
      const float bound = (max_range < 3.0e38) ? (float)max_range * 1.0001f + 1e-30f : 3.402823466e+38f;
      nn1_query(e->nn, e->src_view, e->n_source, e->final_T, e->nn_idx.ptr, e->nn_d2.ptr, e->stream, bound);
      double sum = 0;
      long long cnt = 0;
      fitness_reduce(e->nn_d2.ptr, e->nn_idx.ptr, e->n_source, max_range, e->scratch_d.ptr, &sum, &cnt, e->stream);
      e->other_launches += 3;
      out->fitness = cnt > 0 ? sum / (double)cnt : DBL_MAX;
    }
    return rc;
  });
}
}  // namespace

extern "C" int b200reg_ndt_sweep(b200reg_t h, int count, const float* const* sources, const size_t* n_src,
                                 const float* const* targets, const size_t* n_tgt, size_t stride_bytes, const float* guesses,
                                 double fitness_max_range, b200reg_sweep_result* results) {
  if (!h || h->kind != B200REG_NDT || count < 0 || (count > 0 && (!sources || !n_src || !targets || !n_tgt || !results)))
    return B200REG_ERR_ARG;
  if (stride_bytes < 12 || (stride_bytes % 4) != 0) return B200REG_ERR_ARG;
  if (count == 0) return B200REG_OK;
  const int n_eng = std::max(1, std::min(std::min(h->sweep_engines, 4), count));
  b200reg_t eng[4] = {h, nullptr, nullptr, nullptr};
  for (int e = 1; e < n_eng; e++) {
    if (!h->siblings[e - 1]) {
      b200reg_t sib = nullptr;
      const int rc = b200reg_create(B200REG_NDT, h->device, &sib);
      if (rc != B200REG_OK) return rc;
      h->siblings[e - 1] = sib;
    }
    eng[e] = h->siblings[e - 1];
    eng[e]->ndt = h->ndt;  // the further engines follow the first one's parameters
    eng[e]->min_points_per_voxel = h->min_points_per_voxel;
    eng[e]->min_covar_eigvalue_mult = h->min_covar_eigvalue_mult;
  }
  // A few host threads, one engine (stream + buffers) each: the upload and voxel-map build of one pair overlap the solve
  // and fitness pass of another, and the host-side launch / wait overheads of the pairs overlap too (a pair is ~25 small
  // launches and a handful of waits: more host time than device time). Every pair is computed exactly as the sequential
  // calls would compute it (the result does not depend on which engine served it). Pairs are dealt round-robin — pair i to
  // engine i mod n_eng — not taken from a shared counter: the pairs cost about the same, and a repeated sweep (the
  // backend revisiting its candidates, a warmed-up benchmark pass) then shows every engine the targets it has already
  // sized its bounding-box-dependent buffers for, instead of an occasional cudaFree + cudaMalloc (a device-wide
  // synchronisation) in the middle of the pipeline.
  std::atomic<int> worst{B200REG_OK};
  auto worker = [&](int e) {
    for (int i = e; i < count; i += n_eng) {
      const int rc = sweep_one(eng[e], sources[i], n_src[i], targets[i], n_tgt[i], stride_bytes, guesses ? guesses + 16 * i : nullptr,
                               fitness_max_range, &results[i]);
      results[i].status = rc;
      if (rc != B200REG_OK) worst.store(rc);
    }
  };
  std::vector<std::thread> threads;
  for (int e = 1; e < n_eng; e++) threads.emplace_back(worker, e);
  worker(0);
  for (std::thread& t : threads) t.join();
  for (int e = 1; e < n_eng; e++) {
    const int seen = eng[e]->solver.launches + eng[e]->map.launches + eng[e]->nn.launches + eng[e]->other_launches;
    h->other_launches += seen - h->sibling_launches_seen[e - 1];
    h->sibling_launches_seen[e - 1] = seen;
  }
  return worst.load();
}
