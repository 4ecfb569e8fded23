// vsr_interp.h -- the skeleton interpreter: evaluates one compiled skeleton at P
// points at once as forward-mode dual numbers with K tangents.
//
// Replaces the lambdified scalar loss of the reference
// (src/visymre/architectures/bfgs.py:104-112: one Python term per data point) and
// the per-restart lambdify over variables (bfgs.py:120-132).  Numeric semantics are
// numpy's (bfgs.py:38-40): a domain violation gives nan, overflow gives inf; the
// caller turns a non-finite loss into the 1e6 penalty.
//
// The same code is compiled by nvcc into the kernels and by g++ into the host
// simulator the CPU tests use to check the ISA semantics (oracle/hostsim); the
// product path only ever runs the CUDA build.
//
// Template parameters
//   T  float or double (arithmetic type of the point evaluation)
//   K  number of tangents carried (0 = value only)
//   P  points evaluated per call; the decode of each instruction is shared by the P
//      points, which amortises the interpreter overhead and gives the FP pipes P
//      independent dependency chains.
#ifndef VSR_INTERP_H_
#define VSR_INTERP_H_

#include "vsr_isa.h"

#if defined(__CUDACC__)
#define VSR_HD __host__ __device__ __forceinline__
// the heavy libm routines are kept OUT of line: the interpreter has ~60 handlers and P
// copies of each; inlining pow/sin/... into all of them made the kernels 300-500 KB of
// SASS, far beyond the instruction caches.  One copy per kernel, reached by a call.
#define VSR_MATH __host__ __device__ __noinline__ inline
#else
#include <cmath>
#define VSR_HD inline
#define VSR_MATH inline
#endif

namespace vsr {

// ---- scalar math, overloaded on float/double ------------------------------------
#define VSR_M1(Q, name, fd, ff)                 \
  Q double name(double x) { return fd(x); }     \
  Q float name(float x) { return ff(x); }
VSR_M1(VSR_HD, m_sqrt, ::sqrt, ::sqrtf)
VSR_M1(VSR_HD, m_abs, ::fabs, ::fabsf)
VSR_M1(VSR_MATH, m_exp, ::exp, ::expf)
VSR_M1(VSR_MATH, m_log, ::log, ::logf)
VSR_M1(VSR_MATH, m_sin, ::sin, ::sinf)
VSR_M1(VSR_MATH, m_cos, ::cos, ::cosf)
VSR_M1(VSR_MATH, m_tan, ::tan, ::tanf)
VSR_M1(VSR_MATH, m_asin, ::asin, ::asinf)
VSR_M1(VSR_MATH, m_acos, ::acos, ::acosf)
VSR_M1(VSR_MATH, m_atan, ::atan, ::atanf)
VSR_M1(VSR_MATH, m_sinh, ::sinh, ::sinhf)
VSR_M1(VSR_MATH, m_cosh, ::cosh, ::coshf)
VSR_M1(VSR_MATH, m_tanh, ::tanh, ::tanhf)
#undef VSR_M1
VSR_MATH double m_pow(double a, double b) { return ::pow(a, b); }
VSR_MATH float m_pow(float a, float b) { return ::powf(a, b); }
// a**b together with ln(a): exp(b ln a) for a > 0.  libm's pow carries ln(a) in double-double
// (~250 instructions in fp64); here ln a within L_log ulp and the rounding of b ln a put
// (2 L_log + 1) |b ln a| units of roundoff into the result, plus exp's own error: at most 2.4e-13
// relative in fp64 (|b ln a| < 708), inside the 1e-12 budget, and the tangent rules need ln(a)
// anyway.  libm's pow keeps its exact special cases: non-positive bases, 1**b, a**0 (exp(0 * ln a)
// is nan at a = inf), and |b ln a| from 708 (87 in fp32) on, where the result is next to overflow
// or underflow and exp(b ln a) could land on the other side of the threshold from the value-only
// path.
template <typename T>
VSR_HD T m_pow_log(T a, T b, T& lna) {
  lna = m_log(a);  // -inf at 0, nan below
  if (a > T(0) && a != T(1) && b != T(0)) {
    const T t = b * lna;
    if (m_abs(t) < (sizeof(T) == 8 ? T(708) : T(87))) return m_exp(t);
  }
  return m_pow(a, b);
}
// d(a**b)/da = b f / a for a != 0, f = a**b: b (f / a), or (b f) / a where f / a overflows but the
// derivative does not (a subnormal base and |b| < 1)
template <typename T>
VSR_HD T m_pow_grad(T a, T b, T f) {
  const T big = sizeof(T) == 8 ? (T)1.7976931348623157e308 : (T)3.4028234663852886e38;
  const T g = b * (f / a);
  return (m_abs(g) > big && m_abs(f) <= big) ? (b * f) / a : g;
}
VSR_MATH void m_sincos(double x, double* s, double* c) {
#if defined(__CUDA_ARCH__)
  ::sincos(x, s, c);
#else
  *s = ::sin(x);
  *c = ::cos(x);
#endif
}
VSR_MATH void m_sincos(float x, float* s, float* c) {
#if defined(__CUDA_ARCH__)
  ::sincosf(x, s, c);
#else
  *s = ::sinf(x);
  *c = ::cosf(x);
#endif
}
template <typename T>
VSR_HD T m_sign(T x) {
  return x > T(0) ? T(1) : (x < T(0) ? T(-1) : (x == T(0) ? T(0) : x));
}
// x**n for integer n >= 0 by binary powering (sympy Integer exponents)
template <typename T>
VSR_HD T m_powi(T x, int n) {
  T r = T(1);
  T b = x;
  while (n > 0) {
    if (n & 1) r *= b;
    n >>= 1;
    if (n) b *= b;
  }
  return r;
}
// multiply a tangent by a derivative that may be infinite while the tangent is an
// exact zero (sqrt at 0, asin at +-1): 0*inf must stay 0.
template <typename T>
VSR_HD T m_scale(T d, T fp) {
  return d == T(0) ? T(0) : d * fp;
}

// ---- dual numbers -----------------------------------------------------------------
template <typename T, int K>
struct Dual {
  T v;
  T d[K > 0 ? K : 1];
};

// Operand stack.  Only binary nodes whose two children are both non-leaf push, and
// the compiler orders children Sethi-Ullman style, so depth stays tiny; the array is
// dynamically indexed and therefore lives in (L1-resident) local memory on the GPU.
template <typename T, int K, int P>
struct Stack {
  T s[VSR_MAX_STACK][P][K + 1];
};

// One unary node applied to one dual number.  OP is a compile-time constant, so the
// switch folds away.  `n` is the POWI exponent.
template <int OP, typename T, int K>
VSR_HD void unary_apply(Dual<T, K>& x, unsigned am, int n) {
  const T a = x.v;
  const bool live = (K > 0) && am != 0u;
  T f = a, fp = T(1);
  bool guard = false;  // derivative may be infinite where the value is finite
  switch (OP) {
    case VSR_NEG:
      f = -a;
      fp = T(-1);
      break;
    case VSR_ABS:
      f = m_abs(a);
      fp = m_sign(a);
      break;
    case VSR_SIGN:
      f = m_sign(a);
      fp = T(0);
      break;
    case VSR_INV:
      f = T(1) / a;
      fp = -f * f;
      break;
    case VSR_SQRT:
      f = m_sqrt(a);
      fp = T(0.5) / f;
      guard = true;
      break;
    case VSR_EXP:
      f = m_exp(a);
      fp = f;
      break;
    case VSR_LOG:
      f = m_log(a);
      fp = T(1) / a;
      break;
    case VSR_SIN:
      if (live) {
        m_sincos(a, &f, &fp);
      } else {
        f = m_sin(a);
      }
      break;
    case VSR_COS:
      if (live) {
        T s;
        m_sincos(a, &s, &f);
        fp = -s;
      } else {
        f = m_cos(a);
      }
      break;
    case VSR_TAN:
      f = m_tan(a);
      fp = T(1) + f * f;
      break;
    // 1 - a^2 as (1 - a)(1 + a): 1 - a is exact for |a| >= 1/2, so the factor keeps its digits
    // next to +-1 where 1 - a*a cancels
    case VSR_ASIN:
      f = m_asin(a);
      if (live) fp = T(1) / m_sqrt((T(1) - a) * (T(1) + a));
      guard = true;
      break;
    case VSR_ACOS:
      f = m_acos(a);
      if (live) fp = T(-1) / m_sqrt((T(1) - a) * (T(1) + a));
      guard = true;
      break;
    case VSR_ATAN:
      f = m_atan(a);
      fp = T(1) / (T(1) + a * a);
      break;
    case VSR_SINH:
      f = m_sinh(a);
      if (live) fp = m_cosh(a);
      break;
    case VSR_COSH:
      f = m_cosh(a);
      if (live) fp = m_sinh(a);
      break;
    case VSR_TANH:
      f = m_tanh(a);
      // sech^2 a = 4e / (1 + e)^2 with e = exp(-2|a|): no cancellation, and it decays smoothly
      // to 0 in saturation where 1 - tanh^2 rounds to exactly 0
      if (live) {
        const T e = m_exp(T(-2) * m_abs(a));
        const T d = T(1) + e;
        fp = (T(4) * e) / (d * d);
      }
      break;
    case VSR_POWI: {
      const int m = n < 0 ? -n : n;
      const T pw = m_powi(a, m - 1);  // a^(|n|-1)
      const T full = pw * a;          // a^|n|
      if (n > 0) {
        f = full;
        fp = T(n) * pw;
      } else {
        f = T(1) / full;
        fp = T(n) * f / a;
      }
      break;
    }
    default:
      break;
  }
  x.v = f;
  if (K > 0) {
    if (guard) {  // sqrt at 0, asin/acos at +-1: an exact-zero tangent must stay zero
#pragma unroll
      for (int i = 0; i < K; ++i) x.d[i] = m_scale(x.d[i], fp);
    } else {      // dense: a dead tangent is an exact zero and stays one for finite fp
#pragma unroll
      for (int i = 0; i < K; ++i) x.d[i] *= fp;
    }
  }
}

// ---- instruction dispatch ------------------------------------------------------------------
// The interpreter dispatches on ONE dense handler id per instruction so the compiler emits a
// single jump table: (opcode, operand source) pairs for LOAD and the binary ops, the opcode
// alone for everything else.  Programs are "predecoded" (handler id written over the opcode
// byte) when they are copied into shared memory.
// ids are DENSE (0..63, no holes) so that the switch compiles to one indexed branch:
//   0 END, 1 PUSH, 2..37 (LOAD, ADD..RPOW) x 4 sources, 38..54 the unary ops,
//   55..118 LOAD / ADD / SUB / MUL with a FRESH fitted constant c_j as operand, one handler per
//   (op, j): the tangent of c_j is structurally dead in acc (every skeleton the compiler emits
//   names each constant once), so the one-hot operand tangent is WRITTEN into register slot j,
//   known at compile time, instead of being added through K selects (tangent registers cannot
//   be indexed at run time)
#define VSR_H_BINOP(op) ((op) == VSR_LOAD ? 0 : (op)-VSR_ADD + 1)          /* 0..8 */
#define VSR_H_BIN(op, src) (2 + ((VSR_H_BINOP(op)) << 2) + (src))          /* 2..37 */
#define VSR_H_UN(op) (38 + (op)-VSR_NEG)                                   /* 38..54 */
#define VSR_H_CFOP(op) ((op) == VSR_LOAD ? 0 : (op) == VSR_ADD ? 1 : (op) == VSR_SUB ? 2 : 3)
#define VSR_H_CF(op, j) (55 + VSR_H_CFOP(op) * VSR_MAX_DUAL + (j))          /* 55..118 */
#define VSR_H_END 0
#define VSR_H_PUSH 1
#define VSR_H_COUNT 119
#define VSR_HANDLER(w) ((unsigned)((w)&0xff))

VSR_HD vsr_insn_t predecode(vsr_insn_t w) {
  const unsigned op = VSR_OP(w);
  unsigned h;
  if (op == VSR_END)
    h = VSR_H_END;
  else if (op == VSR_PUSH)
    h = VSR_H_PUSH;
  else if ((op == VSR_LOAD || op == VSR_ADD || op == VSR_SUB || op == VSR_MUL) &&
           (VSR_SRC(w) & 3u) == VSR_SRC_CONST && VSR_IDX(w) < VSR_MAX_DUAL &&
           (op == VSR_LOAD || !((VSR_AMASK(w) >> VSR_IDX(w)) & 1u)))
    h = VSR_H_CF(op, VSR_IDX(w));
  else if (op <= VSR_RPOW)
    h = VSR_H_BIN(op, VSR_SRC(w) & 3u);
  else
    h = VSR_H_UN(op);
  return (w & ~(vsr_insn_t)0xff) | (vsr_insn_t)h;
}

// LOAD / binary node with its operand source known at compile time.
//   acc = acc (OP) b,  b = popped stack entry | column | fitted constant | literal
// Tangent arithmetic is dense over the K tangents wherever a dead (exactly zero) tangent
// stays zero for finite values; only stack operands and the guarded power rules consult
// the liveness masks.  (A tangent that turns nan where the value stays finite is dropped
// when the gradient is accumulated.)
template <int OP, int SRC, typename T, int K, int P, typename XSrc>
VSR_HD void binary_apply(Dual<T, K> (&acc)[P], Stack<T, K, P>& stk, int& sp, unsigned idx,
                         unsigned am, unsigned bm, const double* __restrict__ imm,
                         const T* __restrict__ cst, const XSrc& xs) {
  if (SRC == VSR_SRC_STACK) --sp;
  T ub = T(0);  // operand value when it is uniform over the points
  if (SRC == VSR_SRC_CONST) ub = cst[idx];
  if (SRC == VSR_SRC_IMM) ub = (T)imm[idx];
  const unsigned lm = am | bm;
#pragma unroll
  for (int p = 0; p < P; ++p) {
    T bv;
    if (SRC == VSR_SRC_STACK)
      bv = stk.s[sp][p][0];
    else if (SRC == VSR_SRC_VAR)
      bv = xs.col(idx, p);
    else
      bv = ub;
    Dual<T, K>& x = acc[p];
    // tangent i of the operand
#define VSR_TB(i)                                                                   \
  (SRC == VSR_SRC_STACK ? (((bm >> (i)) & 1u) ? stk.s[sp][p][(i) + 1] : T(0))      \
                        : (SRC == VSR_SRC_CONST ? ((i) == (int)idx ? T(1) : T(0)) : T(0)))
    switch (OP) {
      case VSR_LOAD:
        x.v = bv;
#pragma unroll
        for (int i = 0; i < K; ++i) x.d[i] = VSR_TB(i);
        break;
      case VSR_ADD:
        x.v += bv;
        if (SRC == VSR_SRC_STACK) {  // only the operand's live tangents exist on the stack
#pragma unroll
          for (int i = 0; i < K; ++i)
            if ((bm >> i) & 1u) x.d[i] += stk.s[sp][p][i + 1];
        } else if (SRC == VSR_SRC_CONST) {
#pragma unroll
          for (int i = 0; i < K; ++i) x.d[i] += VSR_TB(i);
        }
        break;
      case VSR_SUB:
        x.v -= bv;
        if (SRC == VSR_SRC_STACK) {
#pragma unroll
          for (int i = 0; i < K; ++i)
            if ((bm >> i) & 1u) x.d[i] -= stk.s[sp][p][i + 1];
        } else if (SRC == VSR_SRC_CONST) {
#pragma unroll
          for (int i = 0; i < K; ++i) x.d[i] -= VSR_TB(i);
        }
        break;
      case VSR_RSUB:
        x.v = bv - x.v;
#pragma unroll
        for (int i = 0; i < K; ++i) x.d[i] = VSR_TB(i) - x.d[i];
        break;
      case VSR_MUL: {
        const T a = x.v;
        x.v = a * bv;
        if (SRC == VSR_SRC_STACK) {
#pragma unroll
          for (int i = 0; i < K; ++i)
            if ((lm >> i) & 1u) x.d[i] = x.d[i] * bv + a * VSR_TB(i);
        } else if (SRC == VSR_SRC_CONST) {
#pragma unroll
          for (int i = 0; i < K; ++i) x.d[i] = x.d[i] * bv + (i == (int)idx ? a : T(0));
        } else {
#pragma unroll
          for (int i = 0; i < K; ++i) x.d[i] *= bv;
        }
        break;
      }
      case VSR_DIV: {  // acc / b
        const T inv = T(1) / bv;
        const T q = x.v / bv;
        if (SRC == VSR_SRC_STACK) {
#pragma unroll
          for (int i = 0; i < K; ++i)
            if ((lm >> i) & 1u) x.d[i] = (x.d[i] - q * VSR_TB(i)) * inv;
        } else if (SRC == VSR_SRC_CONST) {
#pragma unroll
          for (int i = 0; i < K; ++i) x.d[i] = (x.d[i] - (i == (int)idx ? q : T(0))) * inv;
        } else {
#pragma unroll
          for (int i = 0; i < K; ++i) x.d[i] *= inv;
        }
        x.v = q;
        break;
      }
      case VSR_RDIV: {  // b / acc
        const T a = x.v;
        const T inv = T(1) / a;
        const T q = bv / a;
        if (SRC == VSR_SRC_STACK) {
#pragma unroll
          for (int i = 0; i < K; ++i)
            if ((lm >> i) & 1u) x.d[i] = (VSR_TB(i) - q * x.d[i]) * inv;
        } else if (SRC == VSR_SRC_CONST) {
#pragma unroll
          for (int i = 0; i < K; ++i) x.d[i] = ((i == (int)idx ? T(1) : T(0)) - q * x.d[i]) * inv;
        } else {
          const T cf = -q * inv;
#pragma unroll
          for (int i = 0; i < K; ++i) x.d[i] *= cf;
        }
        x.v = q;
        break;
      }
      case VSR_POW: {  // acc ** b
        const T a = x.v;
        // value-only sweeps (forward-difference parity mode, final scores) keep libm's
        // pow: FD gradients amplify an error of 1e-13 in the loss by 1/1.5e-8
        T lna = T(0);
        const T f = (K == 0) ? m_pow(a, bv) : m_pow_log(a, bv, lna);
        if (K > 0 && lm) {
          // d/da = b a^(b-1) = b f / a (one division instead of a second pow; pow again
          // only at a == 0; 0 at b == 0, where f / a may overflow);  d/db = f ln a  (0 where
          // a == 0 and the power vanishes)
          const T fa = am ? (bv == T(0) ? T(0) : a != T(0) ? m_pow_grad(a, bv, f) : bv * m_pow(a, bv - T(1))) : T(0);
          T fb = T(0);
          if (bm) fb = (a == T(0) && f == T(0)) ? T(0) : f * lna;
#pragma unroll
          for (int i = 0; i < K; ++i)
            if ((lm >> i) & 1u) x.d[i] = m_scale(x.d[i], fa) + m_scale((T)VSR_TB(i), fb);
        }
        x.v = f;
        break;
      }
      case VSR_RPOW: {  // b ** acc
        const T a = x.v;
        T lnb = T(0);
        const T f = (K == 0) ? m_pow(bv, a) : m_pow_log(bv, a, lnb);
        if (K > 0 && lm) {
          T fa = T(0);
          if (am) fa = (bv == T(0) && f == T(0)) ? T(0) : f * lnb;
          const T fb = bm ? (a == T(0) ? T(0) : bv != T(0) ? m_pow_grad(bv, a, f) : a * m_pow(bv, a - T(1))) : T(0);
#pragma unroll
          for (int i = 0; i < K; ++i)
            if ((lm >> i) & 1u) x.d[i] = m_scale(x.d[i], fa) + m_scale((T)VSR_TB(i), fb);
        }
        x.v = f;
        break;
      }
      default:
        break;
    }
#undef VSR_TB
  }
}

// LOAD / ADD / SUB / MUL whose operand is the FRESH fitted constant c_J (its tangent is
// structurally dead in acc).  Same formulas as binary_apply<OP, VSR_SRC_CONST> with
// x.d[J] == 0; J is a compile-time register slot.
template <int OP, int J, typename T, int K, int P>
VSR_HD void const_fresh_apply(Dual<T, K> (&acc)[P], const T* __restrict__ cst) {
  constexpr int JJ = (K > 0 && J < K) ? J : 0;
  const T c = cst[J];
#pragma unroll
  for (int p = 0; p < P; ++p) {
    Dual<T, K>& x = acc[p];
    const T a = x.v;
    switch (OP) {
      case VSR_LOAD:
        x.v = c;
#pragma unroll
        for (int i = 0; i < K; ++i) x.d[i] = T(0);
        if (K > 0) x.d[JJ] = T(1);
        break;
      case VSR_ADD:
        x.v = a + c;
        if (K > 0) x.d[JJ] = T(1);
        break;
      case VSR_SUB:
        x.v = a - c;
        if (K > 0) x.d[JJ] = T(-1);
        break;
      case VSR_MUL:
        x.v = a * c;
#pragma unroll
        for (int i = 0; i < K; ++i)
          if (i != JJ) x.d[i] *= c;
        if (K > 0) x.d[JJ] = a;
        break;
      default:
        break;
    }
  }
}

// Where the points come from: col(j, p) returns x_{j+1} of the p-th point of this call.
// (a functor so the kernels can read global or shared memory and the host simulator a
// plain array.)  `prog` must be predecoded.
template <typename T, int K, int P, typename XSrc>
VSR_HD void eval_points(const vsr_insn_t* __restrict__ prog, const double* __restrict__ imm,
                        const T* __restrict__ cst, const XSrc& xs, Dual<T, K> (&acc)[P],
                        Stack<T, K, P>& stk) {
  int sp = 0;
#pragma unroll
  for (int p = 0; p < P; ++p) {
    acc[p].v = T(0);
#pragma unroll
    for (int i = 0; i < (K > 0 ? K : 1); ++i) acc[p].d[i] = T(0);
  }
  // the NEXT word is fetched before the current handler runs, so its shared-memory latency hides
  // behind the handler (every program is followed by a pad word, so the fetch past END is legal)
  vsr_insn_t w = prog[0];
  for (int pc = 1;; ++pc) {
    const unsigned hid = VSR_HANDLER(w);
    const unsigned idx = VSR_IDX(w);
    const unsigned am = VSR_AMASK(w);
    const unsigned bm = VSR_BMASK(w);
    w = prog[pc];  // consumed by the next trip (its latency overlaps the jump-table load)
    switch (hid) {
      case VSR_H_END:
        return;
      case VSR_H_PUSH:
#pragma unroll
        for (int p = 0; p < P; ++p) {
          stk.s[sp][p][0] = acc[p].v;
#pragma unroll
          for (int i = 0; i < K; ++i)
            if ((am >> i) & 1u) stk.s[sp][p][i + 1] = acc[p].d[i];
        }
        ++sp;
        break;
#define VSR_BCASE(OPC)                                                                          \
  case VSR_H_BIN(OPC, VSR_SRC_STACK):                                                           \
    binary_apply<OPC, VSR_SRC_STACK, T, K, P>(acc, stk, sp, idx, am, bm, imm, cst, xs);         \
    break;                                                                                      \
  case VSR_H_BIN(OPC, VSR_SRC_VAR):                                                             \
    binary_apply<OPC, VSR_SRC_VAR, T, K, P>(acc, stk, sp, idx, am, bm, imm, cst, xs);           \
    break;                                                                                      \
  case VSR_H_BIN(OPC, VSR_SRC_CONST):                                                           \
    binary_apply<OPC, VSR_SRC_CONST, T, K, P>(acc, stk, sp, idx, am, bm, imm, cst, xs);         \
    break;                                                                                      \
  case VSR_H_BIN(OPC, VSR_SRC_IMM):                                                             \
    binary_apply<OPC, VSR_SRC_IMM, T, K, P>(acc, stk, sp, idx, am, bm, imm, cst, xs);           \
    break;
        VSR_BCASE(VSR_LOAD)
        VSR_BCASE(VSR_ADD)
        VSR_BCASE(VSR_SUB)
        VSR_BCASE(VSR_RSUB)
        VSR_BCASE(VSR_MUL)
        VSR_BCASE(VSR_DIV)
        VSR_BCASE(VSR_RDIV)
        VSR_BCASE(VSR_POW)
        VSR_BCASE(VSR_RPOW)
#undef VSR_BCASE
#define VSR_CFCASE1(OPC, J)                                              \
  case VSR_H_CF(OPC, J):                                                 \
    if (J < K || K == 0) const_fresh_apply<OPC, J, T, K, P>(acc, cst);   \
    break;
#define VSR_CFCASE(OPC)                                                                          \
  VSR_CFCASE1(OPC, 0) VSR_CFCASE1(OPC, 1) VSR_CFCASE1(OPC, 2) VSR_CFCASE1(OPC, 3)                \
  VSR_CFCASE1(OPC, 4) VSR_CFCASE1(OPC, 5) VSR_CFCASE1(OPC, 6) VSR_CFCASE1(OPC, 7)                \
  VSR_CFCASE1(OPC, 8) VSR_CFCASE1(OPC, 9) VSR_CFCASE1(OPC, 10) VSR_CFCASE1(OPC, 11)              \
  VSR_CFCASE1(OPC, 12) VSR_CFCASE1(OPC, 13) VSR_CFCASE1(OPC, 14) VSR_CFCASE1(OPC, 15)
        VSR_CFCASE(VSR_LOAD)
        VSR_CFCASE(VSR_ADD)
        VSR_CFCASE(VSR_SUB)
        VSR_CFCASE(VSR_MUL)
#undef VSR_CFCASE
#undef VSR_CFCASE1
#define VSR_UCASE(OPC)                                                  \
  case VSR_H_UN(OPC):                                                   \
    _Pragma("unroll") for (int p = 0; p < P; ++p)                       \
        unary_apply<OPC, T, K>(acc[p], am, (int)(int16_t)idx);          \
    break;
        VSR_UCASE(VSR_NEG)
        VSR_UCASE(VSR_ABS)
        VSR_UCASE(VSR_SIGN)
        VSR_UCASE(VSR_INV)
        VSR_UCASE(VSR_SQRT)
        VSR_UCASE(VSR_EXP)
        VSR_UCASE(VSR_LOG)
        VSR_UCASE(VSR_SIN)
        VSR_UCASE(VSR_COS)
        VSR_UCASE(VSR_TAN)
        VSR_UCASE(VSR_ASIN)
        VSR_UCASE(VSR_ACOS)
        VSR_UCASE(VSR_ATAN)
        VSR_UCASE(VSR_SINH)
        VSR_UCASE(VSR_COSH)
        VSR_UCASE(VSR_TANH)
        VSR_UCASE(VSR_POWI)
#undef VSR_UCASE
      default:  // predecode() only emits the ids above (programs are validated at upload)
#if defined(__CUDA_ARCH__)
        __builtin_unreachable();
#else
        break;
#endif
    }
  }
}

}  // namespace vsr

#endif  // VSR_INTERP_H_
