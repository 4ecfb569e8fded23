// vsr_inst.cu -- one instantiation of fit_kernel / eval_kernel / eval_tile_kernel / predict_kernel and their
// launch wrappers: compiled once per (VSR_INST_T, VSR_INST_K) pair, see the Makefile.  The double units
// (VSR_INST_GRAM) also hold gram_kernel of their width.  The fit, eval, eval-tile and Gram kernels come in
// one instantiation per LossMode: the plain units hold kLinear and kWeighted, the VSR_INST_RB units kRobust,
// so that the robust kernels build in parallel with the others.
#include <algorithm>

#include "vsr_launch.h"

namespace vsr {

// the kernel arguments of a launch of mode M: a, then the slot's weights and loss as far as M has them
template <LossMode M, typename A>
static LaunchArgs<A, M> launch_args(const A& a, const PointLoss& pl) {
  LaunchArgs<A, M> r{};
  static_cast<A&>(r) = a;
  if constexpr (M != LossMode::kLinear) r.w = pl.w;
  if constexpr (M == LossMode::kRobust) r.loss = pl.loss;
  return r;
}

template <typename T, int K, LossMode M>
cudaError_t launch_fit_T(const FitArgs& a, int threads, int cs, size_t smem, int clusters, cudaStream_t st,
                         const PointLoss& pl) {
  constexpr int P = points_per_thread(K);
  auto kern = fit_kernel<T, K, P, M>;
  if (threads > fit_max_threads<T, K>()) return cudaErrorInvalidConfiguration;
  // function attributes and the occupancy answer are cached per instantiation: they are driver
  // calls, and vsr_fit launches up to eleven groups per call
  struct Occ { int threads, cs; size_t smem; int resident; };
  struct PerDevice {
    size_t smem_limit = 0;
    bool wide_clusters = false;
    Occ occ[8];
    int n_occ = 0;
  };
  static PerDevice cache[32];
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  PerDevice& pd = cache[dev & 31];
  size_t& smem_limit = pd.smem_limit;
  bool& wide_clusters = pd.wide_clusters;
  Occ* occ = pd.occ;
  int& n_occ = pd.n_occ;
  if (smem > smem_limit) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024));
    if (e != cudaSuccess) return e;
    smem_limit = smem;
  }
  if (cs > 8 && !wide_clusters) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) return e;
    wide_clusters = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)cs);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cs;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int resident = -1;
  for (int i = 0; i < n_occ; ++i)
    if (occ[i].threads == threads && occ[i].cs == cs && occ[i].smem == smem) resident = occ[i].resident;
  if (resident < 0) {
    e = cudaOccupancyMaxActiveClusters(&resident, kern, &cfg);
    if (e != cudaSuccess) return e;
    occ[n_occ % 8] = Occ{threads, cs, smem, resident};
    ++n_occ;
    if (n_occ > 8) n_occ = 8;  // keep overwriting slot 0.. when full
  }
  if (resident < 1) return cudaErrorLaunchOutOfResources;
  cfg.gridDim = dim3((unsigned)(std::max(1, std::min(clusters, resident)) * cs));
  return cudaLaunchKernelEx(&cfg, kern, launch_args<M>(a, pl));
}

template <typename T, int K, LossMode M>
cudaError_t launch_eval_T(const EvalArgs& a, int threads, size_t smem, cudaStream_t st, const PointLoss& pl) {
  eval_kernel<T, K, points_per_thread(K), M><<<dim3(a.n_pairs, a.nsplit), threads, smem, st>>>(launch_args<M>(a, pl));
  return cudaGetLastError();
}

template <typename T, int K, LossMode M>
cudaError_t launch_eval_tile_T(const EvalTileArgs& a, size_t smem, cudaStream_t st, const PointLoss& pl) {
  auto kern = eval_tile_kernel<T, K, points_per_thread(K), M>;
  static size_t smem_limit[32] = {0};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (smem > smem_limit[dev & 31]) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    smem_limit[dev & 31] = smem;
  }
  kern<<<a.e.nsplit, eval_tile_threads<K>(), smem, st>>>(launch_args<M>(a, pl));
  return cudaGetLastError();
}

template <int K, LossMode M>
cudaError_t launch_gram_K(const GramArgs& a, size_t smem, cudaStream_t st, const PointLoss& pl) {
  gram_kernel<K, points_per_thread(K), M>
      <<<dim3(a.n_pairs, a.nsplit), kGramThreads, smem, st>>>(launch_args<M>(a, pl));
  return cudaGetLastError();
}

template <typename T, int K>
cudaError_t launch_predict_T(const PredictArgs& a, size_t smem, cudaStream_t st) {
  predict_kernel<T, K, points_per_thread(K)><<<dim3(a.n_pairs, a.nsplit), kPredictThreads, smem, st>>>(a);
  return cudaGetLastError();
}

template <typename T, int K>
cudaError_t preload_T() {
  constexpr int P = points_per_thread(K);
  cudaFuncAttributes attr;
  cudaError_t e = cudaFuncGetAttributes(&attr, fit_kernel<T, K, P, LossMode::kLinear>);
  if (e != cudaSuccess) return e;
  return cudaFuncGetAttributes(&attr, eval_kernel<T, K, P, LossMode::kLinear>);
}

// explicit instantiations, in the order of the kernels in the objects (gram, fit, eval, eval_tile, predict)
#define VSR_INST_FIT_EVAL(M)                                                                                        \
  template cudaError_t launch_fit_T<VSR_INST_T, VSR_INST_K, M>(const FitArgs&, int, int, size_t, int, cudaStream_t, \
                                                               const PointLoss&);                                   \
  template cudaError_t launch_eval_T<VSR_INST_T, VSR_INST_K, M>(const EvalArgs&, int, size_t, cudaStream_t,         \
                                                                const PointLoss&);
#define VSR_INST_EVAL_TILE(M)                                                                                   \
  template cudaError_t launch_eval_tile_T<VSR_INST_T, VSR_INST_K, M>(const EvalTileArgs&, size_t, cudaStream_t, \
                                                                     const PointLoss&);
#if defined(VSR_INST_GRAM)
#define VSR_INST_GRAM_MODE(M) \
  template cudaError_t launch_gram_K<VSR_INST_K, M>(const GramArgs&, size_t, cudaStream_t, const PointLoss&);
#else
#define VSR_INST_GRAM_MODE(M)
#endif

#if !defined(VSR_INST_RB)
VSR_INST_GRAM_MODE(LossMode::kLinear)
VSR_INST_GRAM_MODE(LossMode::kWeighted)
template cudaError_t preload_T<VSR_INST_T, VSR_INST_K>();
VSR_INST_FIT_EVAL(LossMode::kLinear)
VSR_INST_FIT_EVAL(LossMode::kWeighted)
VSR_INST_EVAL_TILE(LossMode::kLinear)
VSR_INST_EVAL_TILE(LossMode::kWeighted)
template cudaError_t launch_predict_T<VSR_INST_T, VSR_INST_K>(const PredictArgs&, size_t, cudaStream_t);
#else
VSR_INST_GRAM_MODE(LossMode::kRobust)
VSR_INST_FIT_EVAL(LossMode::kRobust)
VSR_INST_EVAL_TILE(LossMode::kRobust)
#endif

}  // namespace vsr
