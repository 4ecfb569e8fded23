// vsr_isa.h -- instruction set of the skeleton bytecode.
//
// One skeleton (a beam candidate with `c` placeholders, reference
// src/visymre/architectures/bfgs.py:65-71) is lowered on the host from its sympy
// tree to a short program for an accumulator machine: one accumulator `acc`, a
// small operand stack that only binary nodes with two non-leaf children ever touch,
// and four operand sources.  Every value is a forward-mode dual number
// (value + one tangent per fitted constant); each instruction carries the set of
// tangents that are structurally live so dead tangents cost nothing and never meet
// an infinite derivative (0*inf).
//
// This header is the single source of truth: the CUDA kernels, the g++ host
// simulator used by the CPU tests and the Python compiler (which parses the enums
// below, see src/visymre/engine/isa.py) all read it.
#ifndef VSR_ISA_H_
#define VSR_ISA_H_

#include <stdint.h>

// ---- instruction word (64 bit) --------------------------------------------------
//  bits  0.. 7  opcode            (VsrOp)
//  bits  8..15  operand source    (VsrSrc)       -- binary ops and LOAD only
//  bits 16..31  operand index     (column / constant slot / immediate slot),
//               or the signed 16-bit exponent of POWI
//  bits 32..47  amask: tangents live in acc BEFORE the instruction
//  bits 48..63  bmask: tangents live in the operand (1<<j for CONST j)
typedef uint64_t vsr_insn_t;

#define VSR_INSN(op, src, idx, amask, bmask)                                   \
  ((vsr_insn_t)((uint64_t)((op)&0xff) | ((uint64_t)((src)&0xff) << 8) |        \
                ((uint64_t)((idx)&0xffff) << 16) |                             \
                ((uint64_t)((amask)&0xffff) << 32) |                           \
                ((uint64_t)((bmask)&0xffff) << 48)))
#define VSR_OP(w) ((unsigned)((w)&0xff))
#define VSR_SRC(w) ((unsigned)(((w) >> 8) & 0xff))
#define VSR_IDX(w) ((unsigned)(((w) >> 16) & 0xffff))
#define VSR_AMASK(w) ((unsigned)(((w) >> 32) & 0xffff))
#define VSR_BMASK(w) ((unsigned)(((w) >> 48) & 0xffff))

enum VsrSrc {
  VSR_SRC_STACK = 0,  // pop the operand stack
  VSR_SRC_VAR = 1,    // column idx of X (0-based: x_1 -> 0)
  VSR_SRC_CONST = 2,  // fitted constant slot idx (c0, c1, ...)
  VSR_SRC_IMM = 3     // literal from the program's immediate pool (fp64)
};

enum VsrOp {
  VSR_END = 0,
  // data movement
  VSR_LOAD = 1,  // acc = operand
  VSR_PUSH = 2,  // stack.push(acc)
  // binary: acc = acc (op) operand, R* forms swap the roles
  VSR_ADD = 3,
  VSR_SUB = 4,   // acc - operand
  VSR_RSUB = 5,  // operand - acc
  VSR_MUL = 6,
  VSR_DIV = 7,   // acc / operand
  VSR_RDIV = 8,  // operand / acc
  VSR_POW = 9,   // acc ** operand
  VSR_RPOW = 10, // operand ** acc
  // unary on acc
  VSR_NEG = 11,
  VSR_ABS = 12,
  VSR_INV = 13,  // 1/acc
  VSR_SQRT = 14,
  VSR_EXP = 15,
  VSR_LOG = 16,
  VSR_SIN = 17,
  VSR_COS = 18,
  VSR_TAN = 19,
  VSR_ASIN = 20,
  VSR_ACOS = 21,
  VSR_ATAN = 22,
  VSR_SINH = 23,
  VSR_COSH = 24,
  VSR_TANH = 25,
  VSR_POWI = 26,  // acc ** n, n = (int16) idx, |n| >= 2
  VSR_SIGN = 27,
  VSR_OP_COUNT = 28
};

// ---- static limits ---------------------------------------------------------------
#define VSR_MAX_VARS 10      // total_variables x_1..x_10 (metadata.h5)
#define VSR_MAX_DUAL 16      // widest tangent kernel; more constants -> FD-gradient mode
#define VSR_MAX_CONSTS 32    // hard cap on constants per skeleton (any mode)
#define VSR_MAX_STACK 8      // operand stack slots (Sethi-Ullman ordered programs)
#define VSR_MAX_INSNS 256    // instructions per program, END included
#define VSR_MAX_IMMS 64      // immediate pool entries per program

// ---- fit status codes (out_status of vsr_fit), scipy OptimizeResult.status -------
enum VsrFitStatus {
  VSR_FIT_SUCCESS = 0,     // gradient norm <= gtol
  VSR_FIT_MAXITER = 1,     // iteration cap (200*k) reached
  VSR_FIT_PRECLOSS = 2,    // line search failed / precision loss
  VSR_FIT_NAN = 3,         // nan in gnorm / fval / x
  VSR_FIT_NOT_RUN = 255    // k == 0: nothing to optimise (bfgs.py:117-118)
};

// gradient modes of vsr_fit
enum VsrGradMode {
  VSR_GRAD_DUAL = 0,  // forward-mode dual numbers, one pass per (f, grad)
  VSR_GRAD_FD = 1     // scipy '2-point' forward differences, k+1 passes (parity mode)
};

// element types of the uploaded points
enum VsrDtype { VSR_F64 = 0, VSR_F32 = 1 };

// robust losses of vsr_set_loss: scipy.optimize.least_squares' `loss` (rho of z = w r^2 / f_scale^2)
enum VsrLoss {
  VSR_LOSS_LINEAR = 0,   // rho(z) = z: the (weighted) sum of squares
  VSR_LOSS_SOFT_L1 = 1,  // 2 ((1 + z)^(1/2) - 1)
  VSR_LOSS_HUBER = 2,    // z if z <= 1, else 2 z^(1/2) - 1
  VSR_LOSS_CAUCHY = 3,   // log1p(z)
  VSR_LOSS_ARCTAN = 4    // arctan(z)
};

#endif  // VSR_ISA_H_
