// gram_twin.cpp -- TEST INFRASTRUCTURE ONLY: the CPU reference of vsr_gram.
//
// A g++ build of the kernels' interpreter (vsr_interp.h) with a serial loop over the points:
// sum r^2 and J^T J in fp64, point by point, through vsr::eval_points<double,K,1>.  The uncertainty
// tests (tests/_gram_ref.py compiles it into a temporary directory) compare it with sympy's exact
// Jacobian on the CPU and with the device's gram_kernel on the GPU; it shares no reduction code with
// the kernel.  Nothing in the product path links, loads or calls it.
#include <cmath>
#include <cstdint>
#include <vector>

#include "vsr_interp.h"

namespace {

template <typename T>
struct HostX {
  const T* X;  // column-major [d][N]
  long N;
  long i;
  T col(unsigned j, int) const { return X[(long)j * N + i]; }
};

std::vector<vsr_insn_t> predecoded(const vsr_insn_t* prog) {
  std::vector<vsr_insn_t> out;
  for (int i = 0;; ++i) {
    out.push_back(vsr::predecode(prog[i]));
    if (VSR_OP(prog[i]) == VSR_END) break;
  }
  out.push_back(0);  // pad word: the interpreter fetches one word ahead
  return out;
}

int pick_K(int k) {
  static const int ks[] = {0, 1, 2, 3, 4, 6, 8, 12, 16};
  for (int v : ks)
    if (v >= k) return v;
  return -1;
}

// fp32 points are widened to double as they are read, as the device's fp64 slot holds them
template <typename TX, int K>
void gram(const vsr_insn_t* prog, const double* imm, const double* c, int k, const TX* X, const TX* y,
          long N, double* out_rss, double* out_jtj) {
  double cst[VSR_MAX_CONSTS];
  for (int i = 0; i < k; ++i) cst[i] = c[i];
  double s = 0.0, g[K > 0 ? K * K : 1];
  for (int i = 0; i < (K > 0 ? K * K : 1); ++i) g[i] = 0.0;
  vsr::Stack<double, K, 1> stk;
  HostX<TX> xs{X, N, 0};
  for (long i = 0; i < N; ++i) {
    xs.i = i;
    vsr::Dual<double, K> acc[1];
    vsr::eval_points<double, K, 1>(prog, imm, cst, xs, acc, stk);
    const double r = acc[0].v - (double)y[i];
    s += r * r;
    for (int a = 0; a < K; ++a)
      for (int b = 0; b < K; ++b) g[a * K + b] += acc[0].d[a] * acc[0].d[b];
  }
  *out_rss = s;
  for (int a = 0; a < k && K > 0; ++a)
    for (int b = 0; b < k; ++b) out_jtj[a * k + b] = g[a * K + b];
}

template <typename TX>
int gram_dispatch(int K, const vsr_insn_t* prog, const double* imm, const double* c, int k, const void* X,
                  const void* y, long N, double* out_rss, double* out_jtj) {
  switch (K) {
#define C(KK) case KK: gram<TX, KK>(prog, imm, c, k, (const TX*)X, (const TX*)y, N, out_rss, out_jtj); return 0;
    C(0) C(1) C(2) C(3) C(4) C(6) C(8) C(12) C(16)
#undef C
  }
  return -1;
}

}  // namespace

extern "C" {

// out_rss = sum_i r_i^2, out_jtj[k][k] = J^T J (fp64 arithmetic for either dtype of the points);
// programs with k > VSR_MAX_DUAL: rss only, jtj nan
int gram_twin(const vsr_insn_t* raw_prog, const double* imm, const double* c, int k, const void* X,
              const void* y, long N, int dtype, double* out_rss, double* out_jtj) {
  const std::vector<vsr_insn_t> pd = predecoded(raw_prog);
  int K = pick_K(k);
  if (K < 0) {
    K = 0;
    for (int i = 0; i < k * k; ++i) out_jtj[i] = NAN;
  }
  return dtype == VSR_F32 ? gram_dispatch<float>(K, pd.data(), imm, c, k, X, y, N, out_rss, out_jtj)
                          : gram_dispatch<double>(K, pd.data(), imm, c, k, X, y, N, out_rss, out_jtj);
}

}  // extern "C"
