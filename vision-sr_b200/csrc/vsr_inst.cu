// vsr_inst.cu -- one instantiation of fit_kernel / eval_kernel / predict_kernel and their launch wrappers:
// compiled once per (VSR_INST_T, VSR_INST_K) pair, see the Makefile.  The double units
// (VSR_INST_GRAM) also hold gram_kernel of their width.  fit, eval, eval_tile and gram kernels come in an
// unweighted (W = false) and a weighted (W = true) instantiation; a wrapper launches the weighted one
// when it is given the slot's weights (w != nullptr).  The robust instantiations (RB = true, launched by
// the *_rb wrappers) are compiled in units of their own (VSR_INST_RB), so that they build in parallel
// with the others.
#include <algorithm>

#include "vsr_launch.h"

namespace vsr {

template <typename T, int K, bool W, bool RB = false>
static cudaError_t launch_fit_TW(const KernelArgs<FitArgs, W, RB>& a, int threads, int cs, size_t smem,
                                 int clusters, cudaStream_t st) {
  constexpr int P = points_per_thread(K);
  auto kern = fit_kernel<T, K, P, W, RB>;
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
  return cudaLaunchKernelEx(&cfg, kern, a);
}

template <typename T, int K, bool W, bool RB = false>
static cudaError_t launch_eval_tile_TW(const KernelArgs<EvalTileArgs, W, RB>& a, size_t smem, cudaStream_t st) {
  constexpr int P = points_per_thread(K);
  auto kern = eval_tile_kernel<T, K, P, W, RB>;
  static size_t smem_limit[32] = {0};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (smem > smem_limit[dev & 31]) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    smem_limit[dev & 31] = smem;
  }
  kern<<<a.e.nsplit, eval_tile_threads<K>(), smem, st>>>(a);
  return cudaGetLastError();
}

#if !defined(VSR_INST_RB)

template <typename T, int K>
cudaError_t launch_fit_T(const FitArgs& a, int threads, int cs, size_t smem, int clusters, cudaStream_t st,
                         const void* w) {
  if (!w) return launch_fit_TW<T, K, false>(Weighted<FitArgs, false>{a}, threads, cs, smem, clusters, st);
  Weighted<FitArgs, true> aw{a};
  aw.w = w;
  return launch_fit_TW<T, K, true>(aw, threads, cs, smem, clusters, st);
}

template <typename T, int K>
cudaError_t launch_eval_T(const EvalArgs& a, int threads, size_t smem, cudaStream_t st, const void* w) {
  constexpr int P = points_per_thread(K);
  dim3 grid(a.n_pairs, a.nsplit);
  if (!w) {
    eval_kernel<T, K, P, false><<<grid, threads, smem, st>>>(Weighted<EvalArgs, false>{a});
  } else {
    Weighted<EvalArgs, true> aw{a};
    aw.w = w;
    eval_kernel<T, K, P, true><<<grid, threads, smem, st>>>(aw);
  }
  return cudaGetLastError();
}

template <typename T, int K>
cudaError_t launch_eval_tile_T(const EvalTileArgs& a, size_t smem, cudaStream_t st, const void* w) {
  if (!w) return launch_eval_tile_TW<T, K, false>(Weighted<EvalTileArgs, false>{a}, smem, st);
  Weighted<EvalTileArgs, true> aw{a};
  aw.w = w;
  return launch_eval_tile_TW<T, K, true>(aw, smem, st);
}

template <typename T, int K>
cudaError_t launch_predict_T(const PredictArgs& a, size_t smem, cudaStream_t st) {
  predict_kernel<T, K, points_per_thread(K)><<<dim3(a.n_pairs, a.nsplit), kPredictThreads, smem, st>>>(a);
  return cudaGetLastError();
}

#if defined(VSR_INST_GRAM)
template <int K>
cudaError_t launch_gram_K(const GramArgs& a, size_t smem, cudaStream_t st, const void* w) {
  const dim3 grid(a.n_pairs, a.nsplit);
  if (!w) {
    gram_kernel<K, points_per_thread(K), false><<<grid, kGramThreads, smem, st>>>(Weighted<GramArgs, false>{a});
  } else {
    Weighted<GramArgs, true> aw{a};
    aw.w = w;
    gram_kernel<K, points_per_thread(K), true><<<grid, kGramThreads, smem, st>>>(aw);
  }
  return cudaGetLastError();
}
template cudaError_t launch_gram_K<VSR_INST_K>(const GramArgs&, size_t, cudaStream_t, const void*);
#endif

template <typename T, int K>
cudaError_t preload_T() {
  constexpr int P = points_per_thread(K);
  cudaFuncAttributes attr;
  cudaError_t e = cudaFuncGetAttributes(&attr, fit_kernel<T, K, P, false>);
  if (e != cudaSuccess) return e;
  return cudaFuncGetAttributes(&attr, eval_kernel<T, K, P, false>);
}

template cudaError_t preload_T<VSR_INST_T, VSR_INST_K>();
template cudaError_t launch_fit_T<VSR_INST_T, VSR_INST_K>(const FitArgs&, int, int, size_t, int, cudaStream_t,
                                                          const void*);
template cudaError_t launch_eval_T<VSR_INST_T, VSR_INST_K>(const EvalArgs&, int, size_t, cudaStream_t, const void*);
template cudaError_t launch_eval_tile_T<VSR_INST_T, VSR_INST_K>(const EvalTileArgs&, size_t, cudaStream_t,
                                                                const void*);
template cudaError_t launch_predict_T<VSR_INST_T, VSR_INST_K>(const PredictArgs&, size_t, cudaStream_t);

#else  // VSR_INST_RB: the robust kernels of this (type, width)

// the robust argument struct of a launch: a, then the weights (nullptr: unweighted) and the loss
template <typename A>
static Robust<A> robust_args(const A& a, const void* w, const RobustLoss& L) {
  Robust<A> r{};
  static_cast<A&>(r) = a;
  r.w = w;
  r.loss = L;
  return r;
}

template <typename T, int K>
cudaError_t launch_fit_rb_T(const FitArgs& a, int threads, int cs, size_t smem, int clusters, cudaStream_t st,
                            const void* w, const RobustLoss& L) {
  return launch_fit_TW<T, K, false, true>(robust_args(a, w, L), threads, cs, smem, clusters, st);
}

template <typename T, int K>
cudaError_t launch_eval_rb_T(const EvalArgs& a, int threads, size_t smem, cudaStream_t st, const void* w,
                             const RobustLoss& L) {
  eval_kernel<T, K, points_per_thread(K), false, true>
      <<<dim3(a.n_pairs, a.nsplit), threads, smem, st>>>(robust_args(a, w, L));
  return cudaGetLastError();
}

template <typename T, int K>
cudaError_t launch_eval_tile_rb_T(const EvalTileArgs& a, size_t smem, cudaStream_t st, const void* w,
                                  const RobustLoss& L) {
  return launch_eval_tile_TW<T, K, false, true>(robust_args(a, w, L), smem, st);
}

#if defined(VSR_INST_GRAM)
template <int K>
cudaError_t launch_gram_rb_K(const GramArgs& a, size_t smem, cudaStream_t st, const void* w, const RobustLoss& L) {
  gram_kernel<K, points_per_thread(K), false, true>
      <<<dim3(a.n_pairs, a.nsplit), kGramThreads, smem, st>>>(robust_args(a, w, L));
  return cudaGetLastError();
}
template cudaError_t launch_gram_rb_K<VSR_INST_K>(const GramArgs&, size_t, cudaStream_t, const void*,
                                                  const RobustLoss&);
#endif

template cudaError_t launch_fit_rb_T<VSR_INST_T, VSR_INST_K>(const FitArgs&, int, int, size_t, int, cudaStream_t,
                                                             const void*, const RobustLoss&);
template cudaError_t launch_eval_rb_T<VSR_INST_T, VSR_INST_K>(const EvalArgs&, int, size_t, cudaStream_t,
                                                              const void*, const RobustLoss&);
template cudaError_t launch_eval_tile_rb_T<VSR_INST_T, VSR_INST_K>(const EvalTileArgs&, size_t, cudaStream_t,
                                                                   const void*, const RobustLoss&);
#endif  // VSR_INST_RB

}  // namespace vsr
