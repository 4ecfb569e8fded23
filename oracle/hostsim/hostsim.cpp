// hostsim.cpp -- TEST INFRASTRUCTURE ONLY.
//
// A g++ build of the portable cores of the CUDA extension (vsr_interp.h: the
// skeleton interpreter; vsr_bfgs.h: the BFGS state machine) with a serial loop over
// the points in place of the GPU sweep.  The CPU test-suite (`-m "not gpu"`) uses it to
// check the instruction semantics against sympy/numpy and the optimiser logic
// against scipy where no GPU exists.  Nothing in the product path
// (vision-sr_b200/src/visymre) links, loads or calls this library.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "vsr_bfgs.h"
#include "vsr_interp.h"

namespace {

template <typename T>
struct HostX {
  const T* X;  // column-major [d][N]
  long N;
  long i;
  T col(unsigned j, int) const { return X[(long)j * N + i]; }
};

// objective = scale * mean((f(x_i; c) - y_i)^2), gradient via K tangents.
template <typename T, int K>
void sweep(const vsr_insn_t* prog, const double* imm, const double* c, int k, const T* X,
           const T* y, long N, double* out_sum, double* out_gsum) {
  T cst[VSR_MAX_CONSTS];
  for (int i = 0; i < k; ++i) cst[i] = (T)c[i];
  double s = 0.0;
  double g[K > 0 ? K : 1];
  for (int i = 0; i < (K > 0 ? K : 1); ++i) g[i] = 0.0;
  vsr::Stack<T, K, 1> stk;
  HostX<T> xs{X, N, 0};
  for (long i = 0; i < N; ++i) {
    xs.i = i;
    vsr::Dual<T, K> acc[1];
    vsr::eval_points<T, K, 1>(prog, imm, cst, xs, acc, stk);
    const double r = (double)acc[0].v - (double)y[i];
    s += r * r;
    for (int t = 0; t < K; ++t) {
      const double gt = 2.0 * r * (double)acc[0].d[t];
      g[t] += std::isfinite(gt) ? gt : 0.0;
    }
  }
  *out_sum = s;
  for (int t = 0; t < K && t < k; ++t) out_gsum[t] = g[t];
}

template <typename T>
int sweep_dispatch(int K, const vsr_insn_t* prog, const double* imm, const double* c, int k,
                   const T* X, const T* y, long N, double* s, double* g) {
  switch (K) {
#define C(KK) case KK: sweep<T, KK>(prog, imm, c, k, X, y, N, s, g); return 0;
    C(0) C(1) C(2) C(3) C(4) C(6) C(8) C(12) C(16)
#undef C
  }
  return -1;
}

std::vector<vsr_insn_t> predecoded(const vsr_insn_t* prog) {
  std::vector<vsr_insn_t> out;
  for (int i = 0;; ++i) {
    out.push_back(vsr::predecode(prog[i]));
    if (VSR_OP(prog[i]) == VSR_END) break;
  }
  out.push_back(0);  // pad word: the interpreter fetches one word ahead
  return out;
}

// value and K tangents of every point; out_tangents is row-major [N][K]
template <typename T, int K>
void duals(const vsr_insn_t* prog, const double* imm, const double* c, int k, const T* X, long N,
           double* out_value, double* out_tangents) {
  T cst[VSR_MAX_CONSTS];
  for (int i = 0; i < k; ++i) cst[i] = (T)c[i];
  vsr::Stack<T, K, 1> stk;
  HostX<T> xs{X, N, 0};
  for (long i = 0; i < N; ++i) {
    xs.i = i;
    vsr::Dual<T, K> acc[1];
    vsr::eval_points<T, K, 1>(prog, imm, cst, xs, acc, stk);
    out_value[i] = (double)acc[0].v;
    for (int t = 0; t < K; ++t) out_tangents[i * K + t] = (double)acc[0].d[t];
  }
}

template <typename T>
int duals_dispatch(int K, const vsr_insn_t* prog, const double* imm, const double* c, int k,
                   const T* X, long N, double* v, double* d) {
  switch (K) {
#define C(KK) case KK: duals<T, KK>(prog, imm, c, k, X, N, v, d); return 0;
    C(0) C(1) C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(12) C(16)
#undef C
  }
  return -1;
}

int pick_K(int k) {
  static const int ks[] = {0, 1, 2, 3, 4, 6, 8, 12, 16};
  for (int v : ks)
    if (v >= k) return v;
  return -1;
}

}  // namespace

extern "C" {

// values f(x_i; c) for every point (K = 0), for interpreter-vs-lambdify tests
int hostsim_values(const vsr_insn_t* raw_prog, const double* imm, const double* c, int k,
                   const void* X, long N, int dtype, double* out) {
  const std::vector<vsr_insn_t> pd = predecoded(raw_prog);
  const vsr_insn_t* prog = pd.data();
  if (dtype == VSR_F64) {
    const double* Xd = (const double*)X;
    double cst[VSR_MAX_CONSTS];
    for (int i = 0; i < k; ++i) cst[i] = c[i];
    vsr::Stack<double, 0, 1> stk;
    HostX<double> xs{Xd, N, 0};
    for (long i = 0; i < N; ++i) {
      xs.i = i;
      vsr::Dual<double, 0> acc[1];
      vsr::eval_points<double, 0, 1>(prog, imm, cst, xs, acc, stk);
      out[i] = acc[0].v;
    }
  } else {
    const float* Xf = (const float*)X;
    float cst[VSR_MAX_CONSTS];
    for (int i = 0; i < k; ++i) cst[i] = (float)c[i];
    vsr::Stack<float, 0, 1> stk;
    HostX<float> xs{Xf, N, 0};
    for (long i = 0; i < N; ++i) {
      xs.i = i;
      vsr::Dual<float, 0> acc[1];
      vsr::eval_points<float, 0, 1>(prog, imm, cst, xs, acc, stk);
      out[i] = acc[0].v;
    }
  }
  return 0;
}

// value and all K tangents of every point, K one of the kernels' widths (0..8, 12, 16);
// out_tangents is [N][K] (untouched for K = 0).  For the per-opcode edge-of-domain tests.
int hostsim_duals(const vsr_insn_t* raw_prog, const double* imm, const double* c, int k,
                  const void* X, long N, int dtype, int K, double* out_value, double* out_tangents) {
  const std::vector<vsr_insn_t> pd = predecoded(raw_prog);
  if (dtype == VSR_F64)
    return duals_dispatch<double>(K, pd.data(), imm, c, k, (const double*)X, N, out_value, out_tangents);
  return duals_dispatch<float>(K, pd.data(), imm, c, k, (const float*)X, N, out_value, out_tangents);
}

// the handler id the interpreter dispatches `word` to (vsr::predecode)
int hostsim_predecode(vsr_insn_t word) { return (int)VSR_HANDLER(vsr::predecode(word)); }

// mean squared residual and its gradient w.r.t. the constants (dual numbers)
int hostsim_loss_grad(const vsr_insn_t* raw_prog, const double* imm, const double* c, int k,
                      const void* X, const void* y, long N, int dtype, int want_grad,
                      double* out_loss, double* out_grad) {
  const std::vector<vsr_insn_t> pd = predecoded(raw_prog);
  const vsr_insn_t* prog = pd.data();
  const int K = want_grad ? pick_K(k) : 0;
  if (K < 0) return -1;
  double s = 0.0, g[VSR_MAX_DUAL] = {0};
  int rc;
  if (dtype == VSR_F64)
    rc = sweep_dispatch<double>(K, prog, imm, c, k, (const double*)X, (const double*)y, N, &s, g);
  else
    rc = sweep_dispatch<float>(K, prog, imm, c, k, (const float*)X, (const float*)y, N, &s, g);
  if (rc) return rc;
  *out_loss = s / (double)N;
  if (want_grad)
    for (int i = 0; i < k; ++i) out_grad[i] = g[i] / (double)N;
  return 0;
}

// one BFGS run driven by the same state machine the fit kernel runs
int hostsim_fit(const vsr_insn_t* raw_prog, const double* imm, int k, const void* X, const void* y,
                long N, int dtype, const double* x0, int grad_mode, double loss_scale,
                double gtol, int maxiter_per_k, double* out_x, double* out_lastx,
                double* out_fun, int* out_status, int* out_nit, int* out_nfev) {
  const std::vector<vsr_insn_t> pd = predecoded(raw_prog);
  const vsr_insn_t* prog = pd.data();
  vsr::FitOpts O;
  O.gtol = gtol;
  O.c1 = 1e-4;
  O.c2 = 0.9;
  O.xrtol = 0.0;
  O.fd_eps = 1.4901161193847656e-08;
  O.penalty = 1e6;
  O.loss_scale = loss_scale;
  O.stop_time = 1e9;
  O.maxiter_per_k = maxiter_per_k;
  O.grad_mode = grad_mode;
  const int K = grad_mode == VSR_GRAD_DUAL ? pick_K(k) : 0;
  if (K < 0 || k > VSR_MAX_CONSTS || k < 1) return -1;
  std::vector<double> ws(vsr::fit_workspace_doubles(k));
  vsr::FitState S;
  vsr::fit_init(S, k, ws.data(), x0);
  while (vsr::fit_step(S, O) == vsr::VSR_NEED_EVAL) {
    double s = 0.0, g[VSR_MAX_DUAL] = {0};
    int rc;
    if (dtype == VSR_F64)
      rc = sweep_dispatch<double>(K, prog, imm, S.xe(), k, (const double*)X, (const double*)y, N, &s, g);
    else
      rc = sweep_dispatch<float>(K, prog, imm, S.xe(), k, (const float*)X, (const float*)y, N, &s, g);
    if (rc) return rc;
    double f = O.loss_scale * (s / (double)N);
    if (!std::isfinite(f)) {
      f = O.penalty;
      for (int i = 0; i < k; ++i) g[i] = 0.0;
    } else {
      for (int i = 0; i < k; ++i) {
        g[i] = O.loss_scale * (g[i] / (double)N);
        if (!std::isfinite(g[i])) g[i] = 0.0;
      }
    }
    S.rf = f;
    if (grad_mode == VSR_GRAD_DUAL)
      for (int i = 0; i < k; ++i) S.rg()[i] = g[i];
  }
  for (int i = 0; i < k; ++i) {
    out_x[i] = S.xk()[i];
    out_lastx[i] = S.lastx()[i];
  }
  *out_fun = S.old_fval;
  *out_status = S.status;
  *out_nit = S.it;
  *out_nfev = S.nfev;
  return 0;
}

}  // extern "C"
