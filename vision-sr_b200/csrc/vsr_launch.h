// vsr_launch.h -- launch wrappers of the templated kernels.  Each (arithmetic type, tangent
// width) pair is compiled in its own translation unit (vsr_inst.cu with -DVSR_INST_T/-DVSR_INST_K)
// so the library builds in parallel; vsr_api.cu only sees these declarations.
#ifndef VSR_LAUNCH_H_
#define VSR_LAUNCH_H_

#include "vsr_kernels.cuh"

namespace vsr {

// points per thread for a tangent width: wide duals are register hungry
constexpr int points_per_thread(int K) { return K <= 8 ? 2 : 1; }

// The loss of a point slot: its per-point weights (nullptr: unweighted) and its robust loss (kind
// VSR_LOSS_LINEAR: none).  The fit, eval, eval-tile and Gram launchers take it and launch the kernel of
// mode M, which the caller picks from it; kLinear and kWeighted are compiled in the plain instantiation
// units, kRobust in the VSR_INST_RB units.
struct PointLoss {
  const void* w;
  RobustLoss loss;
};

// `clusters`: how many clusters the launch could use (runs / seats); clamped to what the device
// can keep resident, since the clusters are persistent
template <typename T, int K, LossMode M>
cudaError_t launch_fit_T(const FitArgs& a, int threads, int cs, size_t smem, int clusters, cudaStream_t st,
                         const PointLoss& pl);

template <typename T, int K, LossMode M>
cudaError_t launch_eval_T(const EvalArgs& a, int threads, size_t smem, cudaStream_t st, const PointLoss& pl);

// eval over shared tiles (large N): one CTA per chunk of the points, see eval_tile_kernel
template <typename T, int K, LossMode M>
cudaError_t launch_eval_tile_T(const EvalTileArgs& a, size_t smem, cudaStream_t st, const PointLoss& pl);

// Gauss-Newton statistics (gram_kernel, fp64 only): compiled in the double translation units
template <int K, LossMode M>
cudaError_t launch_gram_K(const GramArgs& a, size_t smem, cudaStream_t st, const PointLoss& pl);

// per-point values and variances (predict_kernel)
template <typename T, int K>
cudaError_t launch_predict_T(const PredictArgs& a, size_t smem, cudaStream_t st);

// forces the (lazily loaded) kernels of one instantiation onto the device
template <typename T, int K>
cudaError_t preload_T();

}  // namespace vsr

#endif  // VSR_LAUNCH_H_
