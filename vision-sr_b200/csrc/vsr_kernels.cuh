// vsr_kernels.cuh -- sm_100a kernels of the refinement engine.
//
//   fit_kernel<T,K,P>   PERSISTENT thread-block clusters that keep several (candidate, restart)
//                       runs in flight each ("seats").  A pass of a run is a dataflow of messages
//                       through distributed shared memory: the seat's optimiser warp (leader CTA)
//                       advances the BFGS state machine (vsr_bfgs.h) and sends the next request;
//                       every other warp of the cluster sweeps its part of the points -- TMA-staged
//                       once into shared memory -- through the interpreter (vsr_interp.h) and the
//                       CTAs' partial sums travel back.  Replaces minimize(safe_loss, x0, 'BFGS') +
//                       the lambdified loss (reference bfgs.py:102-118).
//   eval_kernel<T,K,P>  batched loss (+ gradient) of (program, constants) pairs; grid.y
//                       splits the points.  Replaces bfgs.py:106-112 and :120-132.
//   eval_tile_kernel    the same over chunks of the points that all pairs of a launch share (N >= 5e5).
//   eval_finalize       deterministic fixed-order sum of the split partials.
//   gram_kernel<K,P>    fp64 sum r^2 and J^T J of (program, constants) pairs (Gauss-Newton statistics
//                       for the covariance of fitted constants); gram_finalize sums its splits.
//   predict_kernel<T,K,P> per-point values of (program, constants) pairs and, with a covariance, the
//                       fp64 delta-method variance g^T C g of each point (prediction bands).
//
// Work mapping: lanes stride over points (coalesced column reads), P points per thread
// share one instruction decode; per-thread partial sums are fp64 and parked in shared memory, then
// summed over the warp by shuffles (fit_kernel: warp_totals) or per component by one warp
// (eval kernels: block_totals); fixed order throughout, so results are reproducible run to run.
#ifndef VSR_KERNELS_CUH_
#define VSR_KERNELS_CUH_

#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "vsr_bfgs.h"
#include "vsr_interp.h"
#include "vsr_isa.h"

namespace vsr {

struct ProgramTable {
  const vsr_insn_t* insns;
  const int32_t* insn_off;  // [C+1]
  const double* imms;
  const int32_t* imm_off;  // [C+1]
  const int32_t* k;        // [C]
};

struct Points {
  const void* X;  // column-major, column stride ldx elements
  const void* y;
  int64_t n;
  int64_t ldx;
};

// ---- hand-over of runs between the clusters of a launch ----------------------------------------------
// When the launch's queues have drained, the clusters that run dry would exit while others still
// carry several long runs each, which share their cluster's sweeps.  Instead, the last seat of a
// cluster to run dry takes a TICKET and waits; a cluster with two or more runs in flight answers a
// ticket by handing one of its runs over: the optimiser state goes through global memory into the
// ticket's slot, the run continues in the waiting cluster (the slices are the same in every cluster
// of a launch, and a run's result does not depend on where it runs).  `live` counts the runs that are
// seated or being pulled; the waiting clusters leave when it reaches zero with the queues drained.
constexpr int kHandoverSlots = 64;       // tickets per launch (a waiting cluster takes one at a time)
constexpr unsigned long long kHandoverWaitNs = 300000ull;  // how long a dry cluster waits for a run
constexpr int kHandoverHead = 4;         // doubles in front of a slot's state: (flag, slot) (prog, k) t0 n_pass
struct Handover {
  int32_t requests;                       // tickets taken by waiting clusters
  int32_t offers;                         // tickets answered (claimed by CAS: offers < requests)
  int32_t live;                           // runs seated or being pulled
  int32_t pad;
  double slots[1];                        // kHandoverSlots slots of FitArgs::handover_slot_d doubles:
                                          // head | FitState (kFitStateDoubles) | workspace
};

constexpr int kMaxSeats = 8;  // runs a cluster can work on at a time
constexpr int kMaxQueues = 4;  // run queues a launch pulls from: its own and up to three narrower groups'

struct FitArgs {
  ProgramTable pt;
  Points pts;
  // Runs of ALL width groups of the vsr_fit call, group after group in launch order (widest
  // first).  The clusters of this launch pull from queue[0] (their own group) until it is drained,
  // then from the queues of the next narrower groups: a K-wide kernel evaluates any k <= K, and a
  // seat that would otherwise stay empty behind a long run takes work the narrower launches are
  // still waiting for SMs to start on.
  const int32_t* run_prog;  // [all runs]
  const int32_t* run_slot;  // [all runs]
  int32_t n_queues;         // queues this launch may pull from (own group first), <= kMaxQueues
  int32_t q_begin[kMaxQueues], q_end[kMaxQueues];  // their ranges in run_prog / run_slot
  int32_t kstride;
  const double* x0;
  double* out_consts;
  double* out_lastx;
  double* out_loss;
  int32_t* out_info;
  int32_t resident;      // 1: every CTA stages its slice of the points into shared memory
  int32_t tma_ok;        // 1: column starts and strides are 16-byte aligned (bulk copies)
  int32_t slice_stride;  // elements between columns of the staged slice
  int32_t seats;         // runs in flight per cluster (<= kMaxSeats)
  int32_t reserved;      // warps of the leader CTA that run optimiser turns and never sweep (0: the
                         // optimiser warps sweep as well), see choose_geometry
  // seat layout in doubles, computed once on the host (fit_seat_layout): the kernel would
  // otherwise re-derive it from (kmax, K, cluster size, ...) at every use
  int32_t seat_d, off_cred, off_ctrl, off_insn;
  int32_t kmax, max_insn, max_imm;  // maxima over this launch's programs (size the seat areas)
  int32_t n_cols;                   // columns of X this launch's programs read
  int32_t col_of_var[VSR_MAX_VARS]; // slice column of variable j (-1: unused)
  int32_t hold_passes;      // a seat retires instead of taking a run while two other seats of its cluster hold
                            // runs with at least this many passes behind them (0: never)
  Handover* handover;       // run hand-over between this launch's clusters (nullptr: off)
  int32_t handover_slot_d;  // doubles per hand-over slot
  int32_t* queue;           // [n_queues] next run of each queue, relative to q_begin (zeroed by the host)
  long long* phase_cycles;  // optional [n_slots][8]: cycles of the run's optimiser lane 0: [0] optimiser turns
                            // ([1] taking in the totals, [2] the BFGS step, [4] publishing the request),
                            // [3] everything else while seated, [5] / [6] %globaltimer when the run was seated /
                            // finished, [7] passes
  FitOpts O;
};

struct EvalArgs {
  ProgramTable pt;
  Points pts;
  const int32_t* pair_prog;  // [n_pairs]
  const int32_t* pair_row;   // [n_pairs] row of `consts`
  const int32_t* pair_out;   // [n_pairs] row of the outputs
  int32_t n_pairs;
  int32_t kstride;
  const double* consts;
  double* partial;  // [n_pairs][nsplit][K+1]
  int32_t nsplit;
  int32_t nan_to_num;  // 1: predictions pass through numpy's nan_to_num before the residual (vsr_score)
};

// Robust loss of a point slot (vsr_set_loss): kind (VsrLoss), C^2 and 1/C^2 of f_scale C.
struct RobustLoss {
  int32_t kind;
  double c2, inv_c2;
};

// The point objective a fit, eval, eval-tile or Gram kernel is compiled for: sum r^2 (kLinear), sum w r^2
// with per-point weights w_i (kWeighted), or a robust loss sum C^2 rho(w r^2 / C^2) (kRobust, weights
// optional at run time).
enum class LossMode { kLinear, kWeighted, kRobust };

// Kernel arguments of a launch of mode M: the argument struct A, then the slot's weights (the slot's
// element type, like y) and then its loss, so that every member of A keeps its parameter offset.
template <typename A, LossMode M>
struct LaunchArgs : A {  // kRobust
  const void* w;         // nullptr: unweighted
  RobustLoss loss;
};
template <typename A>
struct LaunchArgs<A, LossMode::kWeighted> : A {
  const void* w;
};
template <typename A>
struct LaunchArgs<A, LossMode::kLinear> : A {};

// Per-point factors of a robust loss at z = w r^2 / C^2 (finite, >= 0), scipy's least_squares
// definitions: q = rho(z) / z (the cost ratio, q(0) = 1), g = rho'(z), s = rho'(z) + 2 z rho''(z).  q is
// formed directly, never as z / z, so huber's z <= 1 branch gives q = g = s = 1 exactly.  fp64 throughout.
__device__ __forceinline__ void robust_factors(int kind, double z, double& q, double& g, double& s) {
  switch (kind) {
    case VSR_LOSS_SOFT_L1: {
      const double t = 1.0 + z, st = sqrt(t);
      q = 2.0 / (1.0 + st);  // 2 (sqrt(1+z) - 1) / z without the cancellation
      g = 1.0 / st;
      s = g / t;
      return;
    }
    case VSR_LOSS_HUBER:
      if (z <= 1.0) {
        q = g = s = 1.0;
      } else {
        const double sz = sqrt(z);
        q = (2.0 * sz - 1.0) / z;
        g = 1.0 / sz;
        s = 0.0;
      }
      return;
    case VSR_LOSS_CAUCHY:
      q = z == 0.0 ? 1.0 : log1p(z) / z;
      g = 1.0 / (1.0 + z);
      s = (1.0 - z) * g * g;
      return;
    case VSR_LOSS_ARCTAN:
      q = z == 0.0 ? 1.0 : atan(z) / z;
      g = 1.0 / (1.0 + z * z);
      s = (1.0 - 3.0 * z * z) * g * g;  // nan past z ~ 1e154 (inf * 0): the clamp to eps takes it
      return;
    default:
      q = g = s = 1.0;
  }
}

// scipy's rho at z = +inf, where z overflowed from a finite residual: C^2 pi / 2 for arctan, +inf otherwise
__device__ __forceinline__ double robust_cost_inf(const RobustLoss& L) {
  return L.kind == VSR_LOSS_ARCTAN ? L.c2 * 1.5707963267948966 : __longlong_as_double(0x7ff0000000000000ll);
}

// Residual step of a robust sweep (kRobust): adds cost = C^2 rho(z) to ps as (rw * q) * r and rho'(z) rw d_t to
// pg[t], with rw = w r (r without weights).  A non-finite r contributes the linear terms rw r and rw d_t
// (the penalty rule); a z that overflows from a finite r contributes scipy's rho(inf) and no gradient.  With
// q = g = 1 the products are the linear step's, so huber with every z <= 1 gives its sums bit for bit.
template <typename T, int K>
__device__ __forceinline__ void robust_step(const RobustLoss& L, double r, double rw, const Dual<T, K>& d,
                                            double& ps, double* pg) {
  double q = 1.0, g = 1.0, s;
  bool add = true;
  if (fabs(r) <= 1.7976931348623157e308) {
    const double z = rw * r * L.inv_c2;
    if (z <= 1.7976931348623157e308) {
      robust_factors(L.kind, z, q, g, s);
    } else {
      ps += robust_cost_inf(L);
      g = 0.0;
      add = false;
    }
  }
  if (add) ps += (rw * q) * r;
  const double rg = g * rw;
#pragma unroll
  for (int t = 0; t < K; ++t) {
    const double gt = rg * (double)d.d[t];
    if (fabs(gt) <= 1.7976931348623157e308) pg[t] += gt;
  }
}

// ---- point source: coalesced global loads (read-only path) --------------------------
template <typename T, int P>
struct GlobalPoints {
  const T* X;
  int64_t ldx;
  int64_t idx[P];
  __device__ __forceinline__ T col(unsigned j, int p) const {
    return __ldg(X + (int64_t)j * ldx + idx[p]);
  }
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}

// keeps a value in a register: without it the compiler re-derives point indices and thread
// ranks from %tid inside every handler that needs them (it rematerialises rather than spend one
// of the 96 registers)
__device__ __forceinline__ void keep_in_register(int& v) { asm volatile("" : "+r"(v)); }

// One pass over points [n0, n1).  The thread's partial sums  sum r^2  and  sum r * d f/d c_t  go
// straight into its slots of the reduction scratch ([(K+1)][nt] doubles, see block_totals): no
// accumulator is live across the interpreter (they used to be spilled around it).
// Every thread runs the same number of iterations (tail lanes are masked), so the warp stays
// converged for the reduction that follows.
// NTN: the prediction passes through numpy's nan_to_num (nan -> 0, +-inf -> +-largest finite
// value of T) before the residual is taken: the drivers' scoring rule (Feynman_test.py:87).
// M (LossMode): kWeighted: per-point weights w (fp64 arithmetic): sum w r^2 and sum w r df/dc_t.  rw = w * r
// is formed once and every product is the linear one with r replaced by rw, so w = 1.0 gives the linear sums
// bit for bit.  kRobust: robust loss L (robust_step), weights optional (w = nullptr: rw = r).
template <typename T, int K, int P, bool NTN = false, LossMode M = LossMode::kLinear>
__device__ __forceinline__ void sweep_points(const vsr_insn_t* prog, const double* imm,
                                             const T* cst, const T* __restrict__ X,
                                             const T* __restrict__ y, int64_t ldx, int64_t n0,
                                             int64_t n1, double* scratch, int tid, int nt,
                                             const T* __restrict__ w = nullptr, RobustLoss L = {}) {
  // tid / nt: index of this thread among the nt threads that take part in the sweep
  Stack<T, K, P> stk;
  GlobalPoints<T, P> xs;
  xs.X = X;
  xs.ldx = ldx;
  bool first = true;
  for (int64_t base = n0; base < n1; base += (int64_t)nt * P) {
    bool valid[P];
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const int64_t i = base + (int64_t)p * nt + tid;
      valid[p] = i < n1;
      xs.idx[p] = valid[p] ? i : (n1 - 1);
    }
    Dual<T, K> acc[P];
    eval_points<T, K, P>(prog, imm, cst, xs, acc, stk);
    double ps = 0.0, pg[K > 0 ? K : 1];
#pragma unroll
    for (int t = 0; t < (K > 0 ? K : 1); ++t) pg[t] = 0.0;
#pragma unroll
    for (int p = 0; p < P; ++p) {
      if (valid[p]) {
        T pv = acc[p].v;
        if (NTN) {
          const T big = sizeof(T) == 8 ? (T)1.7976931348623157e308 : (T)3.4028234663852886e38;
          pv = pv != pv ? T(0) : (pv > big ? big : (pv < -big ? -big : pv));
        }
        const double r = (double)pv - (double)__ldg(y + xs.idx[p]);
        if constexpr (M == LossMode::kRobust) {
          robust_step<T, K>(L, r, w ? (double)__ldg(w + xs.idx[p]) * r : r, acc[p], ps, pg);
        } else if constexpr (M == LossMode::kWeighted) {
          const double rw = (double)__ldg(w + xs.idx[p]) * r;
          ps += rw * r;
#pragma unroll
          for (int t = 0; t < K; ++t) {
            const double gt = rw * (double)acc[p].d[t];
            if (fabs(gt) <= 1.7976931348623157e308) pg[t] += gt;
          }
        } else {
          ps += r * r;
#pragma unroll
          for (int t = 0; t < K; ++t) {
            const double gt = r * (double)acc[p].d[t];
            // a tangent that blew up where the value stayed finite (exp(-exp(x)) ...) counts 0
            // (one compare and a predicated add; nan fails the compare)
            if (fabs(gt) <= 1.7976931348623157e308) pg[t] += gt;
          }
        }
      }
    }
    if (first) {
      scratch[tid] = ps;
#pragma unroll
      for (int t = 0; t < K; ++t) scratch[(1 + t) * nt + tid] = pg[t];
      first = false;
    } else {
      scratch[tid] += ps;
#pragma unroll
      for (int t = 0; t < K; ++t) scratch[(1 + t) * nt + tid] += pg[t];
    }
  }
  if (first) {  // no points at all
    scratch[tid] = 0.0;
#pragma unroll
    for (int t = 0; t < K; ++t) scratch[(1 + t) * nt + tid] = 0.0;
  }
}

// named barrier over the `count` threads that take part in a sweep (count: multiple of 32)
__device__ __forceinline__ void sweep_barrier(int count) {
  asm volatile("bar.sync 1, %0;" ::"r"(count) : "memory");
}

// Totals of (sum r^2, sum r df/dc_t) over the `snt` threads that took part in a sweep, stored to
// out[0..K].  The sweep parked every thread's partial sums in shared memory (scratch:
// [(K+1)][snt] doubles, column per component); component c is summed by warp c % nw: each lane adds its strided share in
// index order, a lane butterfly finishes.  Fixed order, so results are reproducible and depend on
// snt only.  4x fewer instructions than a butterfly over K+1 values in every warp followed by a
// cross-warp stage (the shuffles were 7 % of the kernel's instructions).  Only the taking-part
// threads may call it (named barrier, so the optimiser warps of the leader CTA can stay out).
template <int K>
__device__ __forceinline__ void block_totals(double* scratch, int stid, int snt, double* out) {
  const int lane = stid & 31, warp = stid >> 5, nw = snt >> 5;
  sweep_barrier(snt);  // every thread's partial sums are parked (by the sweep)
  for (int c = warp; c <= K; c += nw) {
    const double* col = scratch + c * snt;
    double acc = 0.0;
    for (int j = lane; j < snt; j += 32) acc += col[j];
    acc = warp_sum(acc);
    if (lane == 0) out[c] = acc;
  }
  sweep_barrier(snt);  // the scratch may be rewritten
}

// cooperative copy of one program into shared memory
__device__ __forceinline__ void load_program(const ProgramTable& pt, int prog, vsr_insn_t* s_insn,
                                             double* s_imm, int& n_insn, int& n_imm) {
  const int i0 = pt.insn_off[prog], i1 = pt.insn_off[prog + 1];
  const int m0 = pt.imm_off[prog], m1 = pt.imm_off[prog + 1];
  n_insn = i1 - i0;
  n_imm = m1 - m0;
  for (int i = threadIdx.x; i < n_insn; i += blockDim.x) s_insn[i] = pt.insns[i0 + i];
  for (int i = threadIdx.x; i < n_imm; i += blockDim.x) s_imm[i] = pt.imms[m0 + i];
}

__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// ---- TMA (bulk async copy), mbarrier and cluster async-store primitives, sm_90+ PTX -----------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
// blocks until the phase with the given parity has completed (hardware-suspended wait, SASS SYNCS...TRYWAIT)
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "VSR_MBAR_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra VSR_MBAR_DONE;\n"
      "bra VSR_MBAR_WAIT;\n"
      "VSR_MBAR_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// non-blocking probe of a phase
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// global -> this CTA's shared memory, completion counted in bytes on `bar` (SASS: UBLKCP)
__device__ __forceinline__ void tma_bulk_load(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                              uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
// shared::cluster address of this CTA's shared-memory address `a` in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t a, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
  return r;
}
// one arrival + `bytes` more expected transaction bytes on a barrier of ANY CTA of the cluster
__device__ __forceinline__ void mbar_expect_tx_cluster(uint32_t bar_cluster_addr, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(bar_cluster_addr), "r"(bytes)
               : "memory");
}
// asynchronous store into the shared memory of a CTA of the cluster; the store's bytes are counted
// on a barrier of the SAME CTA, whose waiters see the data once the phase completes
__device__ __forceinline__ void st_async_b64(uint32_t dst_cluster_addr, uint64_t v, uint32_t bar_cluster_addr) {
  asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];" ::"r"(dst_cluster_addr),
               "l"(v), "r"(bar_cluster_addr)
               : "memory");
}
__device__ __forceinline__ void st_async_b32(uint32_t dst_cluster_addr, uint32_t v, uint32_t bar_cluster_addr) {
  asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(dst_cluster_addr),
               "r"(v), "r"(bar_cluster_addr)
               : "memory");
}
__device__ __forceinline__ void st_async_val(uint32_t dst, double v, uint32_t bar) {
  st_async_b64(dst, (uint64_t)__double_as_longlong(v), bar);
}
__device__ __forceinline__ void st_async_val(uint32_t dst, float v, uint32_t bar) {
  st_async_b32(dst, __float_as_uint(v), bar);
}

// ---- point source: this CTA's slice, resident in shared memory ----------------------------------
// VAR operands of the shared-memory copy of the program are rewritten to column SLOTS of
// the slice, so col(j, p) is one LDS.
template <typename T, int P>
struct SlicePoints {
  const T* base;  // [n_slots][stride]
  int stride;
  int idx[P];
  __device__ __forceinline__ T col(unsigned j, int p) const { return base[j * stride + idx[p]]; }
};

// One pass over the resident slice (cnt points); partial sums parked like sweep_points does.
// The weights (kWeighted, kRobust) are staged like y (ws, cnt values); same residual rule as sweep_points.
template <typename T, int K, int P, bool NTN = false, LossMode M = LossMode::kLinear>
__device__ __forceinline__ void sweep_slice(const vsr_insn_t* prog, const double* imm, const T* cst,
                                            const T* xs, const T* ys, int stride, int cnt, double* scratch,
                                            int tid, int nt, const T* ws = nullptr, RobustLoss L = {}) {
  Stack<T, K, P> stk;
  SlicePoints<T, P> src;
  src.base = xs;
  src.stride = stride;
  bool first = true;
  for (int base = 0; base < cnt; base += nt * P) {
    bool valid[P];
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const int i = base + p * nt + tid;
      valid[p] = i < cnt;
      src.idx[p] = valid[p] ? i : (cnt - 1);
      keep_in_register(src.idx[p]);
    }
    Dual<T, K> acc[P];
    eval_points<T, K, P>(prog, imm, cst, src, acc, stk);
    double ps = 0.0, pg[K > 0 ? K : 1];
#pragma unroll
    for (int t = 0; t < (K > 0 ? K : 1); ++t) pg[t] = 0.0;
#pragma unroll
    for (int p = 0; p < P; ++p) {
      if (src.idx[p] == base + p * nt + tid) {  // valid[p], from the kept index
        T pv = acc[p].v;
        if (NTN) {  // numpy's nan_to_num on the prediction (the drivers' scoring rule, see sweep_points)
          const T big = sizeof(T) == 8 ? (T)1.7976931348623157e308 : (T)3.4028234663852886e38;
          pv = pv != pv ? T(0) : (pv > big ? big : (pv < -big ? -big : pv));
        }
        const double r = (double)pv - (double)ys[src.idx[p]];
        if constexpr (M == LossMode::kRobust) {
          robust_step<T, K>(L, r, ws ? (double)ws[src.idx[p]] * r : r, acc[p], ps, pg);
        } else if constexpr (M == LossMode::kWeighted) {
          const double rw = (double)ws[src.idx[p]] * r;
          ps += rw * r;
#pragma unroll
          for (int t = 0; t < K; ++t) {
            const double gt = rw * (double)acc[p].d[t];
            if (fabs(gt) <= 1.7976931348623157e308) pg[t] += gt;
          }
        } else {
          ps += r * r;
#pragma unroll
          for (int t = 0; t < K; ++t) {
            const double gt = r * (double)acc[p].d[t];
            if (fabs(gt) <= 1.7976931348623157e308) pg[t] += gt;
          }
        }
      }
    }
    if (first) {
      scratch[tid] = ps;
#pragma unroll
      for (int t = 0; t < K; ++t) scratch[(1 + t) * nt + tid] = pg[t];
      first = false;
    } else {
      scratch[tid] += ps;
#pragma unroll
      for (int t = 0; t < K; ++t) scratch[(1 + t) * nt + tid] += pg[t];
    }
  }
  if (first) {  // no points in this CTA's slice
    scratch[tid] = 0.0;
#pragma unroll
    for (int t = 0; t < K; ++t) scratch[(1 + t) * nt + tid] = 0.0;
  }
}

// ---- warp reduction of NC values per lane --------------------------------------------------------
// Recursive halving: at the level with lane distance m, the lanes with (lane & m) == 0 keep the
// first half of their values and receive the partner's copy of them, the others the second half.
// After log2(n) levels each lane holds ONE value; the remaining levels are a plain butterfly.
// n + (5 - log2 n) double shuffles instead of 5 n.  Fixed order: the result depends on nothing
// but the values.  On return v[0] of every lane is the total of component reduce_comp<N>(lane).
template <int N>  // N: power of two, 1..32
__device__ __forceinline__ void warp_reduce_pow2(double (&v)[N], int lane) {
  int m = 16;
#pragma unroll
  for (int n = N; n > 1; n >>= 1) {
    const bool upper = (lane & m) != 0;
#pragma unroll
    for (int i = 0; i < n / 2; ++i) {
      const double send = upper ? v[i] : v[i + n / 2];
      const double keep = upper ? v[i + n / 2] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, m);
    }
    m >>= 1;
  }
#pragma unroll
  for (; m > 0; m >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], m);
}
template <int N>
__device__ __forceinline__ int reduce_comp(int lane) {
  int c = 0, m = 16;
#pragma unroll
  for (int n = N; n > 1; n >>= 1) {
    if (lane & m) c += n / 2;
    m >>= 1;
  }
  return c;
}
__host__ __device__ constexpr int pow2_floor(int n) { return n >= 32 ? 32 : n >= 16 ? 16 : n >= 8 ? 8 : n >= 4 ? 4 : n >= 2 ? 2 : 1; }
__host__ __device__ constexpr int pow2_ceil(int n) { return n > 16 ? 32 : n > 8 ? 16 : n > 4 ? 8 : n > 2 ? 4 : n > 1 ? 2 : 1; }

// Sums the K+1 per-thread partial sums of a sweep (scratch: [(K+1)][snt], this thread's column
// stid) over the warp and stores the warp's totals to out[0..K].
template <int K>
__device__ __forceinline__ void warp_totals(const double* scratch, int stid, int snt, int lane, double* out) {
  constexpr int NC = K + 1;
  // NC = 2^j + 1 (2, 3, 5, 9, 17): the 2^j block by halving, the odd one out by a plain butterfly;
  // otherwise pad to the next power of two
  constexpr bool odd_one = NC > 1 && pow2_floor(NC) + 1 == NC;
  constexpr int NB = odd_one ? pow2_floor(NC) : pow2_ceil(NC);
  double v[NB];
#pragma unroll
  for (int c = 0; c < NB; ++c) v[c] = c < NC ? scratch[c * snt + stid] : 0.0;
  warp_reduce_pow2<NB>(v, lane);
  const int comp = reduce_comp<NB>(lane);
  constexpr int low = 32 / NB - 1;  // lanes that share a component differ in these bits
  if ((lane & low) == 0 && comp < NC) out[comp] = v[0];
  if (odd_one) {
    double w = scratch[(NC - 1) * snt + stid];
    w = warp_sum(w);
    if (lane == 0) out[NC - 1] = w;
  }
}

// ---- fit kernel ------------------------------------------------------------------------------------
// PERSISTENT thread-block clusters, each working on `seats` (candidate, restart) runs at a time, as a
// DATAFLOW of point-to-point messages through distributed shared memory -- no cluster-wide or
// CTA-wide barrier between the one that starts the kernel and the one that ends it.
//
// A pass of one run is: optimiser turn (one warp: take in the totals, advance the BFGS state machine
// to its next request) -> sweep of all points through the interpreter (every sweeper warp of every CTA)
// -> reduction.  The run of seat g moves through these stations by messages:
//
//   REQUEST  the seat's optimiser warp (leader CTA) writes (program id, k, trial constants -- and the
//            predecoded program itself when the run is new) into the seat area of EVERY CTA with
//            st.async; the bytes are counted on that CTA's request barrier req_bar[g], so a sweeper
//            warp that sees the phase complete sees the whole request.
//   SWEEP    every sweeper warp polls the request barriers of the seats; a warp that finds a request
//            evaluates ITS points for it, reduces its K+1 partial sums over the warp (shuffles) and
//            parks them; the last warp of the CTA to finish (a shared-memory ticket) adds the warps'
//            partials in warp order and sends the CTA's K+1 sums to the leader with st.async, counted
//            on the leader's part_bar[g].
//   TOTALS   the optimiser warp wakes when all CTAs have reported, adds them in rank order, and
//            runs its turn.
//
// Warps never wait for each other: while one seat's optimiser turn runs (5-20 k cycles of dependent
// scalar work) the sweepers serve the other seats, and a warp that finishes a sweep early starts the
// next seat's.  A seat whose run finishes takes the next run from the launch's queue (one atomic)
// inside the same turn; when the queue is drained the seat's optimiser sends a last request with
// program id -1 and the sweepers stop polling it.  The last long runs then have the cluster to
// themselves and a pass costs: turn + two DSMEM hops + one sweep.
//
// The points are split in contiguous slices, one per CTA.  When a slice fits, the columns the
// launch's programs read and y are staged ONCE per cluster into shared memory by TMA bulk copies and
// stay there for every pass of every run the cluster handles.  Reduction order is fixed (lanes,
// warps, CTA rank), so a run's result does not depend on its seat, its cluster or the other runs.
//
// dynamic shared memory (doubles):
//   per seat [ FitState | ws | cred[cs*(K+1)] | ctrl (16 B) | cst | imm | insn ]
//   then wpart [seats][warps][K+1], the per-thread scratch [(K+1)][threads], then the slice
//   (n_cols + 1) * stride * sizeof(T), one column more in a weighted launch (the weights, after X's).
// FitState / ws / cred are used in the leader CTA only; the layout is the same in every CTA so that
// one offset addresses the same thing cluster-wide (mapa).
constexpr int kFitStateDoubles = (int)((sizeof(FitState) + 15) / 16 * 2);
// The code area of a seat is  ctrl[2] | cst[kSeatCstDoubles] | imm[VSR_MAX_IMMS] | insn[...]  with FIXED
// sizes in front of the instructions, so that the interpreter addresses constants, literals and
// instruction words at compile-time offsets from ONE register (see the sweep call site).
constexpr int kSeatCstDoubles = VSR_MAX_CONSTS + 2;
constexpr int kSeatCtrlDoubles = 2;

__host__ __device__ inline size_t fit_seat_doubles(int kmax, int K, int cs, int max_insn) {
  size_t d = kFitStateDoubles + (size_t)fit_workspace_doubles(kmax) + (size_t)cs * (K + 1) + kSeatCtrlDoubles +
             kSeatCstDoubles + VSR_MAX_IMMS + max_insn + 1;  // + pad word after END
  return (d + 1) & ~(size_t)1;  // 16-byte multiple
}
// offsets (in doubles) of the parts of a seat, and the seat's size
struct SeatLayout {
  int seat_d, off_ws, off_cred, off_ctrl, off_cst, off_imm, off_insn;
};
__host__ __device__ inline SeatLayout fit_seat_layout(int kmax, int K, int cs, int max_insn) {
  SeatLayout L;
  L.off_ws = kFitStateDoubles;
  L.off_cred = L.off_ws + fit_workspace_doubles(kmax);
  L.off_ctrl = L.off_cred + cs * (K + 1);
  L.off_cst = L.off_ctrl + kSeatCtrlDoubles;
  L.off_imm = L.off_cst + kSeatCstDoubles;
  L.off_insn = L.off_imm + VSR_MAX_IMMS;
  L.seat_d = (int)fit_seat_doubles(kmax, K, cs, max_insn);
  return L;
}

__host__ __device__ inline size_t fit_smem_bytes(int seats, int kmax, int K, int nwarps, int cs, int max_insn,
                                                 int n_cols, int stride, int elem) {
  return (size_t)seats * fit_seat_doubles(kmax, K, cs, max_insn) * 8 +
         (size_t)seats * nwarps * (K + 1) * 8 +  // wpart
         (size_t)(K + 1) * nwarps * 32 * 8 +     // per-thread scratch of the sweeps
         (n_cols >= 0 ? (size_t)(n_cols + 1) * stride * elem : 0);
}

// Widest CTA the fit kernel is compiled for: ONE CTA of 640 threads (20 warps at <= 96
// registers) per SM, so a cluster owns its SMs.
#if !defined(VSR_FIT_THREADS)
#define VSR_FIT_THREADS 640
#define VSR_FIT_MINCTAS 1
#endif
template <typename T, int K>
__host__ __device__ constexpr int fit_max_threads() {
  return (sizeof(T) == 8 && K > 8) ? 256 : VSR_FIT_THREADS;
}
template <typename T, int K>
__host__ __device__ constexpr int fit_min_ctas() {
  return (sizeof(T) == 8 && K > 8) ? 1 : VSR_FIT_MINCTAS;
}
// lanes that own vector elements in the optimiser turn of a width-K kernel (k <= K; the width-0
// kernel also runs the forward-difference mode, any k <= 32)
template <int K>
__host__ __device__ constexpr int fit_lanes() {
  return K == 0 ? 32 : (K <= 8 ? 8 : 16);
}

// The optimiser step, out of line: its register and stack needs stay out of the sweep's
// allocation (the sweep is the hot loop; this runs on one warp per seat between sweeps).
template <int W>
static __device__ __noinline__ int fit_step_call(FitState& S, const FitOpts& O) {
  return fit_step<W>(S, O);
}

// request header of a seat, 16 bytes, written by the seat's optimiser into every CTA
struct SeatCtrl {
  int prog;  // program of the seated run, -1: the seat is closed (queue drained)
  int k;     // its number of constants
  int n_insn;
  int age;   // passes the run has behind it: the sweepers serve the oldest ready request first
};

// what the optimiser warp of a seat carries from one turn to the next (leader CTA only)
struct SeatBook {
  int slot;  // output row of the seated run
  int prog;  // its program, -1: seat empty
  int k;
  int pad;
  unsigned long long t0;  // TimedFun clock (bfgs.py:29-33)
  double rf;              // scratch: lane 0 -> all lanes
  long long t_logic, t_seated, n_pass, t_take, t_step, t_pub, ns_seated;  // phase_cycles bookkeeping
};

// Sends the request of seat `seat` to every CTA of the cluster.  `fresh`: the program goes along
// (predecoded, VAR operands rewritten to slice columns when the slices are resident).
template <typename T>
__device__ __forceinline__ void publish_request(const FitArgs& a, int cs, int lane, int prog, int k, bool fresh, int age,
                                                const double* xe, uint32_t ctrl_addr, uint32_t req_bar_addr) {
  int i0 = 0, ni = 0, m0 = 0, nm = 0;
  if (prog >= 0 && fresh) {
    i0 = a.pt.insn_off[prog];
    ni = a.pt.insn_off[prog + 1] - i0;
    m0 = a.pt.imm_off[prog];
    nm = a.pt.imm_off[prog + 1] - m0;
  }
  const uint32_t bytes = 16u + (prog >= 0 ? (uint32_t)k * (uint32_t)sizeof(T) : 0u) +
                         (fresh && prog >= 0 ? (uint32_t)(nm + ni + 1) * 8u : 0u);
  for (int r = lane; r < cs; r += 32) mbar_expect_tx_cluster(mapa_u32(req_bar_addr, r), bytes);
  // header words and trial constants (in the sweep's arithmetic type): one (CTA, item) pair per lane;
  // cs is a power of two
  const uint32_t cst_addr = ctrl_addr + 8u * kSeatCtrlDoubles;
  {
    const int n_items = 2 + (prog >= 0 ? k : 0);
    const int sh = __ffs(cs) - 1;
    for (int idx = lane; idx < (n_items << sh); idx += 32) {
      const int r = idx & (cs - 1), it = idx >> sh;
      const uint32_t bar = mapa_u32(req_bar_addr, r);
      if (it < 2) {
        const uint64_t w = it == 0 ? ((uint64_t)(uint32_t)prog | ((uint64_t)(uint32_t)k << 32))
                                   : ((uint64_t)(uint32_t)ni | ((uint64_t)(uint32_t)age << 32));
        st_async_b64(mapa_u32(ctrl_addr + 8u * it, r), w, bar);
      } else {
        st_async_val(mapa_u32(cst_addr + (uint32_t)(it - 2) * (uint32_t)sizeof(T), r), (T)xe[it - 2], bar);
      }
    }
  }
  if (prog < 0) return;
  if (!fresh) return;
  const uint32_t imm_addr = cst_addr + 8u * kSeatCstDoubles;
  const uint32_t insn_addr = imm_addr + 8u * VSR_MAX_IMMS;
  for (int i = lane; i < nm; i += 32) {
    const double v = a.pt.imms[m0 + i];
    for (int r = 0; r < cs; ++r) st_async_val(mapa_u32(imm_addr + 8u * i, r), v, mapa_u32(req_bar_addr, r));
  }
  for (int i = lane; i <= ni; i += 32) {
    vsr_insn_t w = 0;  // pad word after END
    if (i < ni) {
      w = a.pt.insns[i0 + i];
      const unsigned op = VSR_OP(w);
      if (a.resident && op >= VSR_LOAD && op <= VSR_RPOW && op != VSR_PUSH && VSR_SRC(w) == VSR_SRC_VAR)
        w = (w & ~((vsr_insn_t)0xffff << 16)) | ((vsr_insn_t)a.col_of_var[VSR_IDX(w)] << 16);
      w = predecode(w);
    }
    for (int r = 0; r < cs; ++r) st_async_b64(mapa_u32(insn_addr + 8u * i, r), w, mapa_u32(req_bar_addr, r));
  }
}

// One optimiser turn of seat `seat`, run by ONE warp of the leader CTA: take in the totals of the
// sweep that served the seat's last request (if there was one), advance the run to its next
// request, and when it finishes write its results and seat the next run of the launch's queue.
// Ends by publishing the seat's next request.  Returns false when the seat is closed (queue
// drained; the closing request has been sent).
template <typename T, int K>
__device__ __forceinline__ bool seat_turn(const FitArgs& a, int lane, int cs, FitState& S, double* ws,
                                          const double* cred, SeatBook& book, volatile int* s_qcur, uint64_t* part_bar,
                                          uint32_t ctrl_addr, uint32_t req_bar_addr, const SeatBook* books, int* s_open,
                                          int* s_running) {
  constexpr int W = fit_lanes<K>();
  const bool timing = a.phase_cycles != nullptr && lane == 0;
  long long ta = timing ? clock64() : 0;
  int my_prog = book.prog, my_k = book.k;
  if (my_prog >= 0) {
    // component `lane` of (sum r^2, sum r df/dc_t) over the CTAs of the cluster in rank order;
    // lane 0 applies the penalty rule, lanes 1..k scale the gradient
    const double inv_n = 1.0 / (double)a.pts.n;
    double tot = 0.0;
    if (lane <= K) {
#pragma unroll 8
      for (int r = 0; r < cs; ++r) tot += cred[r * (K + 1) + lane];
    }
    const double f = a.O.loss_scale * (__shfl_sync(0xffffffffu, tot, 0) * inv_n);
    bool bad = !isfinite(f);
    if (a.O.stop_time < 1e8) {  // TimedFun: the clock starts at the first call
      int late = 0;
      if (lane == 0) {
        const unsigned long long now = global_ns();
        if (book.t0 == 0ull)
          book.t0 = now;
        else if ((double)(now - book.t0) * 1e-9 >= a.O.stop_time)
          late = 1;
      }
      if (__shfl_sync(0xffffffffu, late, 0)) bad = true;
    }
    if (lane >= 1 && lane <= K && lane - 1 < my_k) {
      const double gv = a.O.loss_scale * (2.0 * tot * inv_n);
      ws[my_k + lane - 1] = (bad || !isfinite(gv)) ? 0.0 : gv;  // S.rg()
    }
    if (lane == 0) {
      S.rf = bad ? a.O.penalty : f;
      book.n_pass += 1;
      if (timing) book.t_take += clock64() - ta;
    }
    __syncwarp();
  }
  bool fresh = false;
  for (;;) {
    if (my_prog < 0) {  // empty seat: take the next run of the launch
      int r = -1;
      // ... unless the cluster already carries two OLD runs (on their way to the iteration cap: each
      // advances at the cluster's sweep rate divided by its live seats, and the launch ends when the
      // slowest of them does): then this seat retires and the run goes to a cluster with room.  Two
      // seats of every cluster always stay open, so the queues drain whatever the rule decides.
      if (a.hold_passes > 0) {
        int hold = 0;
        if (lane == 0) {
          int n_old = 0;
          for (int g2 = 0; g2 < a.seats; ++g2)
            if (&books[g2] != &book && books[g2].prog >= 0 && books[g2].n_pass >= a.hold_passes) ++n_old;
          if (n_old >= 2) {
            if (atomicSub(s_open, 1) > 2)
              hold = 1;
            else
              atomicAdd(s_open, 1);
          }
        }
        if (__shfl_sync(0xffffffffu, hold, 0)) break;
      }
      Handover* const ho = a.handover;
      if (ho != nullptr && lane == 0) atomicAdd(&ho->live, 1);  // counted BEFORE the pull: `live` never under-counts
      for (;;) {
        // ONE read per trip: another seat's warp may advance s_qcur at any time, and a second read
        // could return n_queues -- the counter of a group this launch must not touch (its run would
        // be skipped by the launch that owns it)
        const int q = *s_qcur;
        if (q >= a.n_queues) break;
        if (lane == 0) r = atomicAdd(a.queue + q, 1) + a.q_begin[q];
        r = __shfl_sync(0xffffffffu, r, 0);
        if (r < a.q_end[q]) break;
        __syncwarp();
        if (lane == 0 && *s_qcur == q) *s_qcur = q + 1;  // drained (another seat's warp may have said so already)
        __syncwarp();
        r = -1;
      }
      if (r < 0) {
        // the launch's queues are drained
        if (ho == nullptr) break;
        int ticket = -1;
        if (lane == 0) {
          atomicSub(&ho->live, 1);
          // the last seat of the cluster to run dry waits for a run of a cluster that carries several
          if (*(volatile int*)s_running == 0) ticket = atomicAdd(&ho->requests, 1);
        }
        ticket = __shfl_sync(0xffffffffu, ticket, 0);
        if (ticket < 0 || ticket >= kHandoverSlots) break;
        double* hs = ho->slots + (size_t)ticket * a.handover_slot_d;
        // Waits at most kHandoverWaitNs: a cluster with several runs answers at the next turn of one of
        // its seats, and no cluster gains runs once the queues are drained -- when nobody answers
        // within a few turns nobody will.  Leaving is a CAS on the slot's flag (0 -> 2); an answer is the
        // other CAS (0 -> 1): exactly one of them wins, so a run is never handed to a cluster that left.
        int got = 0;  // 1: a run arrived, 2: nothing to take over
        const unsigned long long t_wait0 = global_ns();
        while (got == 0) {
          if (lane == 0) {
            int flag;
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(flag) : "l"(hs) : "memory");
            if (flag == 1) {
              got = 1;
            } else {
              int live;
              asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(live) : "l"(&ho->live) : "memory");
              if (live == 0 || global_ns() - t_wait0 > kHandoverWaitNs) {
                got = atomicCAS(reinterpret_cast<int*>(hs), 0, 2) == 0 ? 2 : 1;
                if (got == 1) __threadfence();
              } else {
                __nanosleep(400);
              }
            }
          }
          got = __shfl_sync(0xffffffffu, got, 0);
        }
        if (got == 2) break;
        // take the run over: FitState and workspace from the slot, the workspace pointer re-aimed
        {
          const int* hi = reinterpret_cast<const int*>(hs);
          const int h_slot = hi[1], h_prog = hi[2], h_k = hi[3];
          double* dst = reinterpret_cast<double*>(&S);
          for (int i = lane; i < kFitStateDoubles; i += 32) dst[i] = hs[kHandoverHead + i];
          const int nws = fit_workspace_doubles(h_k);
          for (int i = lane; i < nws; i += 32) ws[i] = hs[kHandoverHead + kFitStateDoubles + i];
          __syncwarp();
          if (lane == 0) {
            S.ws = ws;
            book.slot = h_slot;
            book.t0 = *reinterpret_cast<const unsigned long long*>(hs + 2);
            book.n_pass = *reinterpret_cast<const long long*>(hs + 3);
            if (timing) book.t_seated = clock64(), book.t_logic = 0, book.t_take = book.t_step = book.t_pub = 0, book.ns_seated = (long long)global_ns();
            atomicAdd(s_running, 1);
          }
          __syncwarp();
          my_prog = h_prog;
          my_k = h_k;
          fresh = true;  // the program goes round with the request
        }
        break;  // the run was about to publish its request: do that
      }
      const int prog = a.run_prog[r];
      const int slot = a.run_slot[r];
      const int k = a.pt.k[prog];
      if (k == 0) {  // nothing to optimise (reference bfgs.py:117-118)
        if (lane == 0) {
          int32_t* info = a.out_info + (int64_t)slot * 4;
          info[0] = VSR_FIT_NOT_RUN;
          info[1] = 0;
          info[2] = 0;
          info[3] = 0;
          a.out_loss[slot] = 0.0;
          if (ho != nullptr) atomicSub(&ho->live, 1);
        }
        continue;
      }
      my_prog = prog;
      my_k = k;
      fresh = true;
      fit_init<W>(S, k, ws, a.x0 + (int64_t)slot * a.kstride);
      if (lane == 0) {
        atomicAdd(s_running, 1);
        book.slot = slot;
        book.t0 = 0ull;
        book.n_pass = 0;
        if (timing) book.t_seated = clock64(), book.t_logic = 0, book.t_take = book.t_step = book.t_pub = 0, book.ns_seated = (long long)global_ns();
      }
      __syncwarp();
    }
    const long long tb = timing ? clock64() : 0;
    const int act = fit_step_call<W>(S, a.O);
    __syncwarp();  // the state written back by the step is visible to every lane
    if (timing) book.t_step += clock64() - tb;
    if (act == VSR_NEED_EVAL) {
      // a cluster that carries several runs answers the ticket of a waiting one with THIS run
      Handover* const ho = a.handover;
      if (ho == nullptr) break;
      int o = -1;
      if (lane == 0 && *(volatile int*)s_running >= 2) {
        int req, off;
        asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(req) : "l"(&ho->requests) : "memory");
        asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(off) : "l"(&ho->offers) : "memory");
        while (off < req && off < kHandoverSlots) {
          const int old = atomicCAS(&ho->offers, off, off + 1);
          if (old == off) {
            o = off;
            break;
          }
          off = old;
        }
      }
      o = __shfl_sync(0xffffffffu, o, 0);
      if (o < 0) break;
      double* hs = ho->slots + (size_t)o * a.handover_slot_d;
      const double* src = reinterpret_cast<const double*>(&S);
      for (int i = lane; i < kFitStateDoubles; i += 32) hs[kHandoverHead + i] = src[i];
      const int nws = fit_workspace_doubles(my_k);
      for (int i = lane; i < nws; i += 32) hs[kHandoverHead + kFitStateDoubles + i] = ws[i];
      __threadfence();
      __syncwarp();
      if (lane == 0) {
        int* hi = reinterpret_cast<int*>(hs);
        hi[1] = book.slot;
        hi[2] = my_prog;
        hi[3] = my_k;
        *reinterpret_cast<unsigned long long*>(hs + 2) = book.t0;
        *reinterpret_cast<long long*>(hs + 3) = book.n_pass;
        __threadfence();
        // the waiting cluster may have given up (flag 2): then the run stays here
        o = atomicCAS(reinterpret_cast<int*>(hs), 0, 1) == 0 ? o : -1;
        if (o >= 0) atomicSub(s_running, 1);
      }
      o = __shfl_sync(0xffffffffu, o, 0);
      if (o < 0) break;
      my_prog = -1;  // the run lives on elsewhere (it stays counted in `live`)
      fresh = false;
      continue;
    }
    // finished: results out, seat free, try to seat another run in this same turn
    if (lane == 0) {
      if (a.handover != nullptr) atomicSub(&a.handover->live, 1);
      atomicSub(s_running, 1);
      const int slot = book.slot;
      double* oc = a.out_consts + (int64_t)slot * a.kstride;
      double* ol = a.out_lastx + (int64_t)slot * a.kstride;
      const double* xk = ws + 5 * my_k;
      const double* lastx = ws + 4 * my_k;
      for (int i = 0; i < my_k; ++i) {
        oc[i] = xk[i];
        ol[i] = lastx[i];
      }
      a.out_loss[slot] = S.old_fval;
      int32_t* info = a.out_info + (int64_t)slot * 4;
      info[0] = S.status;
      info[1] = S.it;
      info[2] = S.nfev;
      // with the phase buffer on (probes): the cluster that ran it; otherwise reserved (0)
      info[3] = a.phase_cycles != nullptr ? (int32_t)(blockIdx.x / (unsigned)cs) : 0;
      if (timing) {
        const long long now = clock64();
        book.t_logic += now - ta;
        ta = now;
        long long* ph = a.phase_cycles + (int64_t)slot * 8;
        ph[0] += book.t_logic;
        ph[1] += book.t_take;
        ph[2] += book.t_step;
        ph[4] += book.t_pub;
        ph[3] += (now - book.t_seated) - book.t_logic;
        ph[5] = book.ns_seated;
        ph[6] = (long long)global_ns();
        ph[7] += book.n_pass;
      }
    }
    __syncwarp();
    my_prog = -1;
    fresh = false;
  }
  if (lane == 0) {
    book.prog = my_prog;
    book.k = my_k;
    // the totals of the request that goes out now: cs CTAs x (K + 1) doubles
    if (my_prog >= 0) mbar_expect_tx(part_bar, (uint32_t)cs * (uint32_t)(K + 1) * 8u);
  }
  __syncwarp();
  const long long tp = timing ? clock64() : 0;
  publish_request<T>(a, cs, lane, my_prog, my_k, fresh, (int)book.n_pass, ws /* S.xe() */, ctrl_addr, req_bar_addr);
  if (timing && my_prog >= 0) book.t_logic += clock64() - ta, book.t_pub += clock64() - tp;
  return my_prog >= 0;
}

// kWeighted (a.w: per-point weights of the slot of T): a resident slice stages the weight column after the
// n_cols columns of X.  kRobust (a.loss), weighted when a.w is set: it stages exactly what the weighted or
// linear launch stages.
template <typename T, int K, int P, LossMode M>
__global__ void __launch_bounds__((fit_max_threads<T, K>()), (fit_min_ctas<T, K>()))
    fit_kernel(const LaunchArgs<FitArgs, M> a) {
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  extern __shared__ __align__(16) double smem[];
  __shared__ SeatBook s_book[kMaxSeats];
  __shared__ __align__(8) uint64_t s_req_bar[kMaxSeats];   // request of seat g has arrived (every CTA)
  __shared__ __align__(8) uint64_t s_part_bar[kMaxSeats];  // totals of seat g's request have arrived (leader)
  __shared__ __align__(8) uint64_t s_bar;                  // TMA staging of the slice
  __shared__ int s_ticket[kMaxSeats];                      // sweeper warps of this CTA that finished seat g's requests
  __shared__ int s_qcur;  // first queue of this launch that is not drained yet
  __shared__ int s_open;  // seats of this cluster that still take runs (leader CTA)
  __shared__ int s_running;  // seats of this cluster that hold a run (leader CTA)

  const int cs = (int)cluster.num_blocks();
  const int crank = (int)cluster.block_rank();
  const int nw = (blockDim.x + 31) >> 5;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const int G = a.seats;
  const int seat_d = a.seat_d;
#define VSR_SEAT_STATE(g) (smem + (size_t)(g)*seat_d)

  // ---- this CTA's slice of the points ----
  // CTAs 1..cs-1 take `per` points each, the leader (rank 0) takes what is left at the end: its
  // reserved warps never sweep, and the host sizes `per` so that the leader's remainder fits its
  // remaining warps.
  const int64_t N = a.pts.n;
  const int64_t per = a.slice_stride;
  int64_t n0 = crank == 0 ? (int64_t)(cs - 1) * per : (int64_t)(crank - 1) * per;
  int64_t n1 = crank == 0 ? N : n0 + per;
  n0 = n0 < N ? n0 : N;
  n1 = n1 < N ? n1 : N;
  const int cnt = (int)(n1 - n0);
  const T* X = static_cast<const T*>(a.pts.X);
  const T* y = static_cast<const T*>(a.pts.y);
  const T* rb_w = nullptr;  // the weights of a robust launch (nullptr: unweighted)
  if constexpr (M == LossMode::kRobust) rb_w = static_cast<const T*>(a.w);

  double* wpart = smem + (size_t)G * seat_d;                      // [G][nw][K+1]
  double* scratch = wpart + (size_t)G * nw * (K + 1);             // [(K+1)][threads]
  T* xs = nullptr;
  T* ys = nullptr;
  const int stride = a.slice_stride;
  if (tid == 0) {
    for (int g = 0; g < kMaxSeats; ++g) {
      mbar_init(&s_req_bar[g], 1);
      mbar_init(&s_part_bar[g], 1);
      s_ticket[g] = 0;
    }
    mbar_init(&s_bar, 1);
    mbar_fence_init();
    s_qcur = 0;
    s_open = a.seats;
    s_running = 0;
  }
  if (tid < kMaxSeats) {
    s_book[tid].prog = -1;
    s_book[tid].k = 0;
    s_book[tid].t0 = 0ull;
    s_book[tid].t_logic = s_book[tid].t_seated = s_book[tid].n_pass = 0;
    s_book[tid].t_take = s_book[tid].t_step = s_book[tid].t_pub = 0;
  }
  __syncthreads();
  if (a.resident) {
    ys = reinterpret_cast<T*>(scratch + (size_t)(K + 1) * blockDim.x);
    xs = ys + stride;
    constexpr int kAlign = 16 / (int)sizeof(T);
    const int full = cnt & ~(kAlign - 1);  // elements per column that move as 16-byte units
    const bool use_tma = a.tma_ok && full > 0;
    if (tid == 0 && use_tma) {
      const uint32_t bytes = (uint32_t)full * (uint32_t)sizeof(T);
      mbar_expect_tx(&s_bar, bytes * (uint32_t)(a.n_cols + 1 + (M == LossMode::kWeighted || rb_w ? 1 : 0)));
      tma_bulk_load(ys, y + n0, bytes, &s_bar);
      for (int j = 0; j < VSR_MAX_VARS; ++j)
        if (a.col_of_var[j] >= 0)
          tma_bulk_load(xs + (size_t)a.col_of_var[j] * stride, X + (int64_t)j * a.pts.ldx + n0, bytes, &s_bar);
      if constexpr (M == LossMode::kWeighted)
        tma_bulk_load(xs + (size_t)a.n_cols * stride, static_cast<const T*>(a.w) + n0, bytes, &s_bar);
      if (rb_w) tma_bulk_load(xs + (size_t)a.n_cols * stride, rb_w + n0, bytes, &s_bar);
    }
    {
      // everything TMA does not move (all of it when the caller's memory is unaligned): coalesced loads
      const int first = use_tma ? full : 0;
      for (int i = first + tid; i < cnt; i += blockDim.x) ys[i] = y[n0 + i];
      if constexpr (M == LossMode::kWeighted) {
        T* wsl = xs + (size_t)a.n_cols * stride;
        for (int i = first + tid; i < cnt; i += blockDim.x) wsl[i] = static_cast<const T*>(a.w)[n0 + i];
      }
      if (rb_w) {
        T* wsl = xs + (size_t)a.n_cols * stride;
        for (int i = first + tid; i < cnt; i += blockDim.x) wsl[i] = rb_w[n0 + i];
      }
      for (int j = 0; j < VSR_MAX_VARS; ++j) {
        const int sj = a.col_of_var[j];
        if (sj < 0) continue;
        for (int i = first + tid; i < cnt; i += blockDim.x)
          xs[(size_t)sj * stride + i] = X[(int64_t)j * a.pts.ldx + n0 + i];
      }
    }
    if (use_tma) mbar_wait(&s_bar, 0);  // every thread observes the completed transaction
    __syncthreads();                    // ... and the plain stores of the others
  }

  // every CTA of the cluster is running and has initialised its barriers before any DSMEM access
  cluster.sync();

  // ---- roles ----
  // Optimiser warps: the LAST n_opt warps of the leader CTA (the warp scheduler prefers higher warp
  // ids, and a turn is the latency-critical part of a pass); optimiser warp j serves seats j,
  // j + n_opt, ...  With reserved warps (a.reserved > 0, see choose_geometry) they never sweep and
  // the leader's slice is sized for the remaining warps; without (small CTAs) they sweep as well.
  const int reserved = crank == 0 ? a.reserved : 0;
  const int n_opt = a.reserved > 0 ? a.reserved : (G < nw ? G : nw);
  const bool is_opt = crank == 0 && warp >= nw - n_opt;
  const bool sweeper = warp < nw - reserved;
  const int nsw = nw - reserved;  // sweeper warps of this CTA
  int stid = warp * 32 + lane, snt = nsw * 32;
  keep_in_register(stid);
  keep_in_register(snt);

  uint32_t req_phase = 0, live = sweeper ? ((1u << G) - 1u) : 0u;
  uint32_t part_phase = 0, opt_wait = 0, opt_live = 0;
  if (is_opt)
    for (int g = warp - (nw - n_opt); g < G; g += n_opt) opt_live |= 1u << g;
  const uint32_t ctrl0 = smem_u32(smem) + 8u * (uint32_t)a.off_ctrl;

  while (live | opt_live) {
    bool progress = false;
    // ---- optimiser turns of my seats whose totals have arrived ----
    if (opt_live) {
      const bool only = !live && (opt_live & (opt_live - 1)) == 0;  // nothing else to do: block
      for (int g = 0; g < G; ++g) {
        if (!((opt_live >> g) & 1u)) continue;
        if ((opt_wait >> g) & 1u) {
          const uint32_t par = (part_phase >> g) & 1u;
          if (only)
            mbar_wait(&s_part_bar[g], par);
          else if (!mbar_test(&s_part_bar[g], par))
            continue;
          part_phase ^= 1u << g;
        }
        double* seat = VSR_SEAT_STATE(g);
        const bool open = seat_turn<T, K>(a, lane, cs, *reinterpret_cast<FitState*>(seat), seat + kFitStateDoubles,
                                          seat + a.off_cred, s_book[g], &s_qcur, &s_part_bar[g],
                                          ctrl0 + 8u * (uint32_t)(g * seat_d), smem_u32(&s_req_bar[g]), s_book, &s_open,
                                          &s_running);
        if (open)
          opt_wait |= 1u << g;
        else
          opt_live &= ~(1u << g);
        progress = true;
      }
    }
    // ---- one sweep: of the ready requests, the one of the OLDEST run ----
    // (a run that has many passes behind it is probably on its way to the iteration cap, and the
    // launch ends when the longest run does: it must not queue behind the young runs of its cluster)
    if (live) {
      int g = -1;
      if (!opt_live && (live & (live - 1)) == 0) {  // nothing else to do: block on the one live seat
        g = __ffs(live) - 1;
        mbar_wait(&s_req_bar[g], (req_phase >> g) & 1u);
      } else {
        int best_age = -1;
        for (int q = 0; q < G; ++q) {
          if (!((live >> q) & 1u) || !mbar_test(&s_req_bar[q], (req_phase >> q) & 1u)) continue;
          const SeatCtrl* c = reinterpret_cast<const SeatCtrl*>(smem + (size_t)q * seat_d + a.off_ctrl);
          const int age = c->prog < 0 ? 0x7fffffff : c->age;  // a closing request costs nothing: first
          if (age > best_age) best_age = age, g = q;
        }
      }
      if (g >= 0) {
        req_phase ^= 1u << g;
        progress = true;
        // the seat's code area through ONE opaque byte offset: without the asm the compiler
        // re-derives the pointers from (g, seat_d, ...) for every bytecode instruction instead
        // of spending registers on them
        unsigned code_off = (unsigned)((g * seat_d + a.off_insn) * 8);
        asm volatile("" : "+r"(code_off));
        const vsr_insn_t* c_insn = reinterpret_cast<const vsr_insn_t*>(reinterpret_cast<char*>(smem) + code_off);
        const double* c_imm = reinterpret_cast<const double*>(c_insn) - VSR_MAX_IMMS;
        const T* c_cst = reinterpret_cast<const T*>(c_imm - kSeatCstDoubles);
        const SeatCtrl c = *reinterpret_cast<const SeatCtrl*>(c_imm - kSeatCstDoubles - kSeatCtrlDoubles);
        if (c.prog < 0) {  // the seat is closed
          live &= ~(1u << g);
        } else {
          if constexpr (M == LossMode::kRobust) {
            if (a.resident)
              sweep_slice<T, K, P, false, M>(c_insn, c_imm, c_cst, xs, ys, stride, cnt, scratch, stid, snt,
                                                       rb_w ? xs + (size_t)a.n_cols * stride : nullptr, a.loss);
            else
              sweep_points<T, K, P, false, M>(c_insn, c_imm, c_cst, X, y, a.pts.ldx, n0, n1, scratch, stid,
                                                        snt, rb_w, a.loss);
          } else if constexpr (M == LossMode::kWeighted) {
            if (a.resident)
              sweep_slice<T, K, P, false, M>(c_insn, c_imm, c_cst, xs, ys, stride, cnt, scratch, stid, snt,
                                                xs + (size_t)a.n_cols * stride);
            else
              sweep_points<T, K, P, false, M>(c_insn, c_imm, c_cst, X, y, a.pts.ldx, n0, n1, scratch, stid, snt,
                                                 static_cast<const T*>(a.w));
          } else {
            if (a.resident)
              sweep_slice<T, K, P>(c_insn, c_imm, c_cst, xs, ys, stride, cnt, scratch, stid, snt);
            else
              sweep_points<T, K, P>(c_insn, c_imm, c_cst, X, y, a.pts.ldx, n0, n1, scratch, stid, snt);
          }
          double* mine = wpart + ((size_t)g * nw + warp) * (K + 1);
          warp_totals<K>(scratch, stid, snt, lane, mine);
          __syncwarp();
          int t = 0;
          if (lane == 0) {
            __threadfence_block();
            t = atomicAdd(&s_ticket[g], 1);
          }
          t = __shfl_sync(0xffffffffu, t, 0);
          if ((t + 1) % nsw == 0) {
            // last warp of this CTA for this request: the CTA's sums in warp order, to the leader
            __threadfence_block();
            if (lane <= K) {
              const double* col = wpart + (size_t)g * nw * (K + 1) + lane;
              double acc = 0.0;
              for (int w = 0; w < nsw; ++w) acc += col[w * (K + 1)];
              const uint32_t dst = smem_u32(VSR_SEAT_STATE(g) + a.off_cred + crank * (K + 1) + lane);
              st_async_val(mapa_u32(dst, 0), acc, mapa_u32(smem_u32(&s_part_bar[g]), 0));
            }
          }
        }
      }
    }
    if (!progress) __nanosleep(40);
  }
#undef VSR_SEAT_STATE
  // no CTA may exit while another can still write to (or wait on) its shared memory
  cluster.sync();
}

// dynamic shared memory of eval_kernel, in doubles: red[(K+1)*threads] | cst[k] | imm | insn
// kWeighted: weighted sums (a.w, read from global memory like y).  kRobust: robust sums (a.loss), weighted
// when a.w is set.
template <typename T, int K, int P, LossMode M>
__global__ void __launch_bounds__(256) eval_kernel(const LaunchArgs<EvalArgs, M> a) {
  extern __shared__ double smem[];
  const int pair = blockIdx.x;
  const int split = blockIdx.y;
  if (pair >= a.n_pairs) return;
  const int prog = a.pair_prog[pair];
  const int k = a.pt.k[prog];
  double* red = smem;  // reduction scratch of block_totals: [(K+1)][blockDim.x]
  const int n_red = (K + 1) * (int)blockDim.x;
  T* cst = reinterpret_cast<T*>(red + n_red);
  double* s_imm = red + n_red + k + 1;
  const int m_imm = a.pt.imm_off[prog + 1] - a.pt.imm_off[prog];
  vsr_insn_t* s_insn = reinterpret_cast<vsr_insn_t*>(s_imm + m_imm);
  int n_insn, n_imm;
  load_program(a.pt, prog, s_insn, s_imm, n_insn, n_imm);
  const double* c = a.consts + (int64_t)a.pair_row[pair] * a.kstride;
  for (int i = threadIdx.x; i < k; i += blockDim.x) cst[i] = (T)c[i];
  __syncthreads();
  for (int i = threadIdx.x; i < n_insn; i += blockDim.x) s_insn[i] = predecode(s_insn[i]);
  __syncthreads();

  const int64_t N = a.pts.n;
  // split the points in chunks that are multiples of the CTA tile so every split but the
  // last is full
  const int64_t tile = (int64_t)blockDim.x * P;
  const int64_t tiles = (N + tile - 1) / tile;
  const int64_t per = (tiles + a.nsplit - 1) / a.nsplit;
  int64_t n0 = (int64_t)split * per * tile;
  int64_t n1 = (int64_t)(split + 1) * per * tile;
  n0 = n0 < N ? n0 : N;
  n1 = n1 < N ? n1 : N;

  if constexpr (M == LossMode::kRobust)  // (nor robust)
    sweep_points<T, K, P, false, M>(s_insn, s_imm, cst, static_cast<const T*>(a.pts.X),
                                              static_cast<const T*>(a.pts.y), a.pts.ldx, n0, n1, red,
                                              (int)threadIdx.x, (int)blockDim.x, static_cast<const T*>(a.w), a.loss);
  else if constexpr (M == LossMode::kWeighted)  // (vsr_score, the nan_to_num rule, is never weighted)
    sweep_points<T, K, P, false, M>(s_insn, s_imm, cst, static_cast<const T*>(a.pts.X),
                                       static_cast<const T*>(a.pts.y), a.pts.ldx, n0, n1, red, (int)threadIdx.x,
                                       (int)blockDim.x, static_cast<const T*>(a.w));
  else if (K == 0 && a.nan_to_num)  // scoring rule of the drivers, value only
    sweep_points<T, K, P, true>(s_insn, s_imm, cst, static_cast<const T*>(a.pts.X),
                                static_cast<const T*>(a.pts.y), a.pts.ldx, n0, n1, red, (int)threadIdx.x,
                                (int)blockDim.x);
  else
    sweep_points<T, K, P>(s_insn, s_imm, cst, static_cast<const T*>(a.pts.X),
                          static_cast<const T*>(a.pts.y), a.pts.ldx, n0, n1, red, (int)threadIdx.x,
                          (int)blockDim.x);
  block_totals<K>(red, (int)threadIdx.x, (int)blockDim.x,
                  a.partial + ((int64_t)pair * a.nsplit + split) * (K + 1));
}

// ---- batched evaluation over SHARED tiles (large N) ------------------------------------------------
// eval_kernel gives every (pair, split) CTA its own pass over the columns: at N = 1e7 and 1024 pairs
// the launch requests ~1000x the data set from L2 / HBM.  Here a CTA owns one CHUNK of the points,
// stages its columns and y ONCE into shared memory (TMA bulk copies, like fit_kernel's resident
// slices) and then runs EVERY pair over that chunk: the points cross HBM once per launch, whatever
// the number of pairs.  Partial sums go to partial[pair][chunk][K+1]; eval_finalize adds the chunks
// in index order (deterministic).
struct EvalTileArgs {
  EvalArgs e;        // e.nsplit = number of chunks = gridDim.x
  int32_t chunk;     // points per CTA (multiple of 32)
  int32_t stride;    // elements between columns of the staged chunk
  int32_t n_cols;    // columns staged
  int32_t tma_ok;
  int32_t max_insn;  // longest program of the launch (sizes the code area)
  int32_t col_of_var[VSR_MAX_VARS];
};

template <int K>
__host__ __device__ constexpr int eval_tile_threads() {
  return K <= 2 ? 1024 : 512;
}

// dynamic shared memory, in doubles: red[(K+1)*threads] | cst[kSeatCstDoubles] | imm[VSR_MAX_IMMS] |
// insn[max_insn + 1] | chunk ((n_cols + 1) * stride * sizeof(T))
__host__ __device__ inline size_t eval_tile_fixed_doubles(int K, int threads, int max_insn) {
  size_t d = (size_t)(K + 1) * threads + kSeatCstDoubles + VSR_MAX_IMMS + max_insn + 1;
  return (d + 1) & ~(size_t)1;
}

// kWeighted: weighted sums.  The weights are read from global memory (a.w, like y in eval_kernel), not
// staged: the chunks are those of the linear launch, so the partial sums are formed in the same order and
// w = 1 gives the linear result bit for bit.  kRobust: robust sums (a.loss), weights as in kWeighted when
// a.w is set.
template <typename T, int K, int P, LossMode M>
__global__ void __launch_bounds__((eval_tile_threads<K>()), 1)
    eval_tile_kernel(const LaunchArgs<EvalTileArgs, M> a) {
  extern __shared__ __align__(16) double smem[];
  __shared__ __align__(8) uint64_t s_bar;
  const int tid = threadIdx.x, nt = blockDim.x;
  double* red = smem;
  T* cst = reinterpret_cast<T*>(red + (size_t)(K + 1) * nt);
  double* s_imm = reinterpret_cast<double*>(cst) + kSeatCstDoubles;
  vsr_insn_t* s_insn = reinterpret_cast<vsr_insn_t*>(s_imm + VSR_MAX_IMMS);
  T* ys = reinterpret_cast<T*>(smem + eval_tile_fixed_doubles(K, nt, a.max_insn));
  T* xs = ys + a.stride;
  const int64_t N = a.e.pts.n;
  const int64_t n0 = (int64_t)blockIdx.x * a.chunk;
  const int cnt = (int)((n0 + a.chunk <= N ? a.chunk : (N > n0 ? N - n0 : 0)));
  const T* X = static_cast<const T*>(a.e.pts.X);
  const T* y = static_cast<const T*>(a.e.pts.y);
  // ---- stage the chunk ----
  if (tid == 0) {
    mbar_init(&s_bar, 1);
    mbar_fence_init();
  }
  __syncthreads();
  {
    constexpr int kAlign = 16 / (int)sizeof(T);
    const int full = cnt & ~(kAlign - 1);
    const bool use_tma = a.tma_ok && full > 0;
    if (tid == 0 && use_tma) {
      const uint32_t bytes = (uint32_t)full * (uint32_t)sizeof(T);
      mbar_expect_tx(&s_bar, bytes * (uint32_t)(a.n_cols + 1));
      tma_bulk_load(ys, y + n0, bytes, &s_bar);
      for (int j = 0; j < VSR_MAX_VARS; ++j)
        if (a.col_of_var[j] >= 0)
          tma_bulk_load(xs + (size_t)a.col_of_var[j] * a.stride, X + (int64_t)j * a.e.pts.ldx + n0, bytes, &s_bar);
    }
    const int first = use_tma ? full : 0;
    for (int i = first + tid; i < cnt; i += nt) ys[i] = y[n0 + i];
    for (int j = 0; j < VSR_MAX_VARS; ++j) {
      const int sj = a.col_of_var[j];
      if (sj < 0) continue;
      for (int i = first + tid; i < cnt; i += nt) xs[(size_t)sj * a.stride + i] = X[(int64_t)j * a.e.pts.ldx + n0 + i];
    }
    if (use_tma) mbar_wait(&s_bar, 0);
    __syncthreads();
  }
  // ---- every pair over the staged chunk ----
  // The program, literals and constants of pair p+1 are FETCHED (global -> registers, one word per
  // thread: programs have at most VSR_MAX_INSNS <= blockDim words) before the sweep of pair p and
  // stored to the code area after it, so their L2 latency hides behind the sweep.
  vsr_insn_t nx_w = 0;
  double nx_imm = 0.0, nx_c = 0.0;
  int nx_ni = 0, nx_nm = 0, nx_k = 0;
  auto fetch = [&](int pair) {
    const int prog = a.e.pair_prog[pair];
    nx_k = a.e.pt.k[prog];
    const int i0 = a.e.pt.insn_off[prog], m0 = a.e.pt.imm_off[prog];
    nx_ni = a.e.pt.insn_off[prog + 1] - i0;
    nx_nm = a.e.pt.imm_off[prog + 1] - m0;
    nx_w = tid < nx_ni ? a.e.pt.insns[i0 + tid] : (vsr_insn_t)0;
    nx_imm = tid < nx_nm ? a.e.pt.imms[m0 + tid] : 0.0;
    nx_c = tid < nx_k ? a.e.consts[(int64_t)a.e.pair_row[pair] * a.e.kstride + tid] : 0.0;
  };
  auto commit = [&]() {
    if (tid <= nx_ni) {
      vsr_insn_t w = 0;  // pad word after END
      if (tid < nx_ni) {
        w = nx_w;
        const unsigned op = VSR_OP(w);
        if (op >= VSR_LOAD && op <= VSR_RPOW && op != VSR_PUSH && VSR_SRC(w) == VSR_SRC_VAR)
          w = (w & ~((vsr_insn_t)0xffff << 16)) | ((vsr_insn_t)a.col_of_var[VSR_IDX(w)] << 16);
        w = predecode(w);
      }
      s_insn[tid] = w;
    }
    if (tid < nx_nm) s_imm[tid] = nx_imm;
    if (tid < nx_k) cst[tid] = (T)nx_c;
  };
  if (a.e.n_pairs > 0) fetch(0);
  for (int pair = 0; pair < a.e.n_pairs; ++pair) {
    commit();
    __syncthreads();
    if (pair + 1 < a.e.n_pairs) fetch(pair + 1);
    if constexpr (M == LossMode::kRobust)
      sweep_slice<T, K, P, false, M>(s_insn, s_imm, cst, xs, ys, a.stride, cnt, red, tid, nt,
                                               a.w ? static_cast<const T*>(a.w) + n0 : nullptr, a.loss);
    else if constexpr (M == LossMode::kWeighted)
      sweep_slice<T, K, P, false, M>(s_insn, s_imm, cst, xs, ys, a.stride, cnt, red, tid, nt,
                                        static_cast<const T*>(a.w) + n0);
    else if (K == 0 && a.e.nan_to_num)
      sweep_slice<T, K, P, true>(s_insn, s_imm, cst, xs, ys, a.stride, cnt, red, tid, nt);
    else
      sweep_slice<T, K, P>(s_insn, s_imm, cst, xs, ys, a.stride, cnt, red, tid, nt);
    // (block_totals ends with a barrier over all threads: the code area may be rewritten after it)
    block_totals<K>(red, tid, nt, a.e.partial + ((int64_t)pair * a.e.nsplit + blockIdx.x) * (K + 1));
  }
}

// ---- Gauss-Newton statistics of (program, constants) pairs -----------------------------------------
// For each pair, over all N points, in fp64 from the fp64 point slot:
//   rss = sum_i r_i^2,   jtj[a][b] = sum_i J_ia J_ib   (a <= b < K),
// r_i = f(x_i; c) - y_i and J_ia the tangent of constant a.  The grid is (pairs x point splits) like
// eval_kernel's.  A CTA interprets one tile of blockDim.x * P points at a time, parks r and J of the
// tile's points in shared memory, and after one barrier thread t adds ITS entry of the upper triangle
// (t = 0: rss) over the tile's points in point order, into a register carried from tile to tile.  The
// split count is a function of N alone (gram_nsplit) and every sum runs in a fixed order, so a pair's
// result does not depend on the other pairs of the call or on its place in the list.  Non-finite
// values propagate (no penalty rule): a point where f is not real makes the outputs nan.
// partial[pair][split][gram_entries(K)] in the order rss, (0,0), (0,1) .. (0,K-1), (1,1) ..
struct GramArgs {
  ProgramTable pt;
  Points pts;  // the fp64 slot
  const int32_t* pair_prog;  // [n_pairs]
  const int32_t* pair_row;   // [n_pairs] row of `consts`
  int32_t n_pairs;
  int32_t kstride;
  const double* consts;
  double* partial;  // [n_pairs][nsplit][gram_entries(K)]
  int32_t nsplit;
};

constexpr int kGramThreads = 256;
__host__ __device__ constexpr int gram_entries(int K) { return 1 + K * (K + 1) / 2; }
static_assert(gram_entries(VSR_MAX_DUAL) <= kGramThreads, "one thread per Gram entry");
// splits of the points: at least 16 tiles each, at most 128 splits (a function of N only)
__host__ __device__ inline int gram_nsplit(int64_t N, int64_t tile) {
  const int64_t tiles = (N + tile - 1) / tile;
  const int64_t s = tiles / 16;
  return (int)(s < 1 ? 1 : (s > 128 ? 128 : s));
}
// column stride (doubles) of the tile's values in shared memory: odd, so that the lanes of a warp,
// which read the same point of different tangent columns, hit different banks
__host__ __device__ constexpr int gram_col_stride(int tile) { return tile + 1; }

// dynamic shared memory of gram_kernel, in doubles: tile[(K+1) * gram_col_stride] | cst[k] | imm | insn
// kWeighted: weighted sums rss = sum w r^2, jtj[a][b] = sum w J_a J_b (J^T W J).  The tile gets one column more, the
// weights, and every term is fma(col_a * w, col_b, acc): w = 1.0 gives the unweighted sums bit for bit.
// kRobust: curve_fit's statistics under a robust loss (a.loss, weighted when a.w is set): rss = sum C^2 rho(z),
// jtj[a][b] = sum w s J_a J_b with s = max(rho' + 2 z rho'', 2^-52) (least_squares' scaled Jacobian).  The
// tile gets two factor columns where kWeighted parks w: w q (q = rho(z)/z) for rss and w s for the J entries, so the
// terms are fma(r * wq, r, acc) and fma(J_a * ws, J_b, acc), the unweighted / weighted sums when q = s = 1.
// A non-finite r gets q = s = 1 (the outputs become non-finite, as in the linear kernel); a z that overflows
// from a finite r parks r = 1 and wq = rho(inf) C^2, and s = 2^-52.
template <int K, int P, LossMode M>
__global__ void __launch_bounds__(kGramThreads) gram_kernel(const LaunchArgs<GramArgs, M> a) {
  extern __shared__ double smem[];
  const int pair = blockIdx.x;
  const int split = blockIdx.y;
  const int tid = threadIdx.x;
  constexpr int kTile = kGramThreads * P;
  constexpr int kLd = gram_col_stride(kTile);
  constexpr int kEnt = gram_entries(K);
  const int prog = a.pair_prog[pair];
  const int k = a.pt.k[prog];
  double* s_val = smem;  // [K+1][kLd]: r, then J[0..K) (then w when kWeighted, wq and ws when kRobust)
  double* cst = s_val + (K + 1 + (M == LossMode::kWeighted ? 1 : 0) + (M == LossMode::kRobust ? 2 : 0)) * kLd;
  double* s_imm = cst + k + 1;
  const int m_imm = a.pt.imm_off[prog + 1] - a.pt.imm_off[prog];
  vsr_insn_t* s_insn = reinterpret_cast<vsr_insn_t*>(s_imm + m_imm);
  int n_insn, n_imm;
  load_program(a.pt, prog, s_insn, s_imm, n_insn, n_imm);
  const double* c = a.consts + (int64_t)a.pair_row[pair] * a.kstride;
  for (int i = tid; i < k; i += kGramThreads) cst[i] = c[i];
  __syncthreads();
  for (int i = tid; i < n_insn; i += kGramThreads) s_insn[i] = predecode(s_insn[i]);
  __syncthreads();

  // the entry this thread owns: 0 = rss, else (ea, eb) of the upper triangle
  int ea = 0, eb = 0;
  if (tid > 0 && tid < kEnt) {
    int t = tid - 1;
    while (t >= K - ea) t -= K - ea++;
    eb = ea + t;
  }
  const double* col_a = s_val + (tid == 0 ? 0 : 1 + ea) * kLd;
  const double* col_b = s_val + (tid == 0 ? 0 : 1 + eb) * kLd;

  const int64_t N = a.pts.n;
  const int64_t tiles = (N + kTile - 1) / kTile;
  const int64_t per = (tiles + a.nsplit - 1) / a.nsplit;
  const int64_t n0 = min((int64_t)split * per * kTile, N);
  const int64_t n1 = min((int64_t)(split + 1) * per * kTile, N);
  const double* X = static_cast<const double*>(a.pts.X);
  const double* y = static_cast<const double*>(a.pts.y);
  Stack<double, K, P> stk;
  GlobalPoints<double, P> xs;
  xs.X = X;
  xs.ldx = a.pts.ldx;
  double acc = 0.0;
  for (int64_t base = n0; base < n1; base += kTile) {
    const int cnt = (int)min((int64_t)kTile, n1 - base);
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const int64_t i = base + (int64_t)p * kGramThreads + tid;
      xs.idx[p] = i < n1 ? i : (n1 - 1);
    }
    Dual<double, K> v[P];
    eval_points<double, K, P>(s_insn, s_imm, cst, xs, v, stk);
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const int j = p * kGramThreads + tid;  // = point index - base
      if (j < cnt) {
        s_val[j] = v[p].v - __ldg(y + xs.idx[p]);
#pragma unroll
        for (int t = 0; t < K; ++t) s_val[(1 + t) * kLd + j] = v[p].d[t];
        if constexpr (M == LossMode::kWeighted) s_val[(K + 1) * kLd + j] = __ldg(static_cast<const double*>(a.w) + xs.idx[p]);
        if constexpr (M == LossMode::kRobust) {
          const double r = s_val[j];
          const double w = a.w ? __ldg(static_cast<const double*>(a.w) + xs.idx[p]) : 1.0;
          double q = 1.0, g, s = 1.0, wq;
          bool over = false;
          if (fabs(r) <= 1.7976931348623157e308) {
            const double z = w * r * r * a.loss.inv_c2;
            if (z <= 1.7976931348623157e308) {
              robust_factors(a.loss.kind, z, q, g, s);
            } else {
              over = true;
              s_val[j] = 1.0;
              s = 0.0;
            }
          }
          wq = over ? robust_cost_inf(a.loss) : w * q;
          s_val[(K + 1) * kLd + j] = wq;
          s_val[(K + 2) * kLd + j] = w * (s > 0x1p-52 ? s : 0x1p-52);  // (nan fails the compare)
        }
      }
    }
    __syncthreads();
    if constexpr (M == LossMode::kRobust) {
      const double* col_f = s_val + (K + (tid == 0 ? 1 : 2)) * kLd;
      if (tid < kEnt)
        for (int j = 0; j < cnt; ++j) acc = fma(col_a[j] * col_f[j], col_b[j], acc);
    } else if constexpr (M == LossMode::kWeighted) {
      const double* col_w = s_val + (K + 1) * kLd;
      if (tid < kEnt)
        for (int j = 0; j < cnt; ++j) acc = fma(col_a[j] * col_w[j], col_b[j], acc);
    } else {
      if (tid < kEnt)
        for (int j = 0; j < cnt; ++j) acc = fma(col_a[j], col_b[j], acc);
    }
    __syncthreads();  // the tile's values may be overwritten
  }
  if (tid < kEnt) a.partial[((int64_t)pair * a.nsplit + split) * kEnt + tid] = acc;
}

// ---- per-point values and delta-method variances of (program, constants) pairs ---------------------
// For each pair and every point i of the slot of T:
//   out_value[row][i] = f(x_i; c)                     stored as f64; numpy's semantics, no nan_to_num
//   out_var[row][i]   = sum_a sum_b g_a C_ab g_b       g = d f / d c at x_i, C the pair's k x k block
// The variance is fp64 whatever T (the tangents are widened first) and runs over a, then b, in index
// order.  The grid is (pairs x point splits) like eval_kernel's; thread tid handles point
// base + p * kPredictThreads + tid of each tile, so a warp's stores are coalesced.  Nothing is summed
// across points, so a point's outputs depend only on its program, constants, covariance and the point:
// not on the grid or on the other pairs of the call.  Width 0 serves the value-only pairs; with
// out_var it writes 0 for k == 0 and nan for k > VSR_MAX_DUAL (no tangents).  All offsets are int64.
struct PredictArgs {
  ProgramTable pt;
  Points pts;                // the slot of T
  const int32_t* pair_prog;  // [n_pairs]
  const int32_t* pair_row;   // [n_pairs] row of `consts` and of `cov`
  const int32_t* pair_out;   // [n_pairs] row of the outputs
  int32_t n_pairs;
  int32_t kstride;
  const double* consts;  // [rows][kstride]
  const double* cov;     // [rows][kstride][kstride]; nullptr iff out_var is
  double* out_value;     // [..][ld_out]
  double* out_var;       // [..][ld_out] or nullptr
  int64_t ld_out;
  int32_t nsplit;
};

constexpr int kPredictThreads = 256;

// dynamic shared memory of predict_kernel, in doubles: cov[K * K] | cst[k] | imm | insn
template <typename T, int K, int P>
__global__ void __launch_bounds__(kPredictThreads) predict_kernel(const PredictArgs a) {
  extern __shared__ double smem[];
  const int pair = blockIdx.x;
  const int split = blockIdx.y;
  const int tid = threadIdx.x;
  constexpr int kTile = kPredictThreads * P;
  const int prog = a.pair_prog[pair];
  const int k = a.pt.k[prog];
  const int64_t row = a.pair_row[pair];
  double* s_cov = smem;  // [K][K], zero past k
  T* cst = reinterpret_cast<T*>(s_cov + K * K);
  double* s_imm = s_cov + K * K + k + 1;
  const int m_imm = a.pt.imm_off[prog + 1] - a.pt.imm_off[prog];
  vsr_insn_t* s_insn = reinterpret_cast<vsr_insn_t*>(s_imm + m_imm);
  int n_insn, n_imm;
  load_program(a.pt, prog, s_insn, s_imm, n_insn, n_imm);
  const double* c = a.consts + row * a.kstride;
  for (int i = tid; i < k; i += kPredictThreads) cst[i] = (T)c[i];
  if (K > 0) {
    const double* C = a.cov + row * a.kstride * a.kstride;
    for (int e = tid; e < K * K; e += kPredictThreads) {
      const int r = e / (K > 0 ? K : 1), q = e - r * K;
      s_cov[e] = (r < k && q < k) ? C[(int64_t)r * a.kstride + q] : 0.0;
    }
  }
  __syncthreads();
  for (int i = tid; i < n_insn; i += kPredictThreads) s_insn[i] = predecode(s_insn[i]);
  __syncthreads();

  const int64_t N = a.pts.n;
  const int64_t tiles = (N + kTile - 1) / kTile;
  const int64_t per = (tiles + a.nsplit - 1) / a.nsplit;
  const int64_t n0 = min((int64_t)split * per * kTile, N);
  const int64_t n1 = min((int64_t)(split + 1) * per * kTile, N);
  const int64_t out_row = (int64_t)a.pair_out[pair] * a.ld_out;
  double* val = a.out_value + out_row;
  double* var = a.out_var ? a.out_var + out_row : nullptr;
  // value-only pairs with a variance row: none to carry (k == 0) or no tangents for it (k > K)
  const double var0 = k == 0 ? 0.0 : __longlong_as_double(0x7ff8000000000000ll);
  Stack<T, K, P> stk;
  GlobalPoints<T, P> xs;
  xs.X = static_cast<const T*>(a.pts.X);
  xs.ldx = a.pts.ldx;
  for (int64_t base = n0; base < n1; base += kTile) {
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const int64_t i = base + (int64_t)p * kPredictThreads + tid;
      xs.idx[p] = i < n1 ? i : (n1 - 1);
    }
    Dual<T, K> v[P];
    eval_points<T, K, P>(s_insn, s_imm, cst, xs, v, stk);
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const int64_t i = base + (int64_t)p * kPredictThreads + tid;
      if (i >= n1) continue;
      val[i] = (double)v[p].v;
      if (K > 0) {
        // tangents past the program's k are not constants of it: they are 0 unless an overflow made
        // them nan (inf * 0 in a product rule), which must not reach the form through C's zero padding
        double g[K > 0 ? K : 1];
#pragma unroll
        for (int t = 0; t < K; ++t) g[t] = t < k ? (double)v[p].d[t] : 0.0;
        double q = 0.0;
#pragma unroll
        for (int r = 0; r < K; ++r) {
          double cg = 0.0;
#pragma unroll
          for (int t = 0; t < K; ++t) cg = fma(s_cov[r * K + t], g[t], cg);
          q = fma(g[r], cg, q);
        }
        var[i] = q;
      } else if (var) {
        var[i] = var0;
      }
    }
  }
}

#if defined(VSR_API_TU)  // plain kernels: defined once, in the API translation unit
// out_loss[row] = sum_splits partial / N ; out_grad[row][t] = 2 * sum / N  (t < k, else 0)
__global__ void eval_finalize(const double* partial, const int32_t* pair_prog,
                              const int32_t* pair_out, const int32_t* prog_k, int n_pairs,
                              int nsplit, int K, int kstride, double inv_n, double* out_loss,
                              double* out_grad) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int pair = idx / (K + 1);
  const int comp = idx - pair * (K + 1);
  if (pair >= n_pairs) return;
  double acc = 0.0;
  for (int sidx = 0; sidx < nsplit; ++sidx)
    acc += partial[((int64_t)pair * nsplit + sidx) * (K + 1) + comp];
  const int row = pair_out[pair];
  if (comp == 0) {
    out_loss[row] = acc * inv_n;
  } else if (out_grad != nullptr) {
    const int t = comp - 1;
    if (t < kstride) out_grad[(int64_t)row * kstride + t] = t < prog_k[pair_prog[pair]] ? 2.0 * acc * inv_n : 0.0;
  }
}

// out_rss[row] = sum_splits partial[rss]; out_jtj[row][a][b] = sum_splits partial[(min, max)] for a, b < k,
// splits added in index order (both triangles from the same sum, so the matrix is exactly symmetric).
// A pair whose program has more constants than the group's width K (k > VSR_MAX_DUAL, value-only
// group) gets nan for its k x k entries.
__global__ void gram_finalize(const double* partial, const int32_t* pair_prog, const int32_t* pair_out,
                              const int32_t* prog_k, int n_pairs, int nsplit, int K, int kstride,
                              double* out_rss, double* out_jtj) {
  const int per = 1 + kstride * kstride;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int pair = (int)(idx / per);
  const int e = (int)(idx - (int64_t)pair * per);
  if (pair >= n_pairs) return;
  const int k = prog_k[pair_prog[pair]];
  const int row = pair_out[pair];
  const int n_ent = 1 + K * (K + 1) / 2;
  int ent = 0;
  if (e > 0) {
    const int r = (e - 1) / kstride, c = (e - 1) % kstride;
    if (r >= k || c >= k) return;
    if (k > K) {
      out_jtj[((int64_t)row * kstride + r) * kstride + c] = __longlong_as_double(0x7ff8000000000000ll);
      return;
    }
    const int lo = r < c ? r : c, hi = r < c ? c : r;
    ent = 1 + lo * K - lo * (lo - 1) / 2 + (hi - lo);
  }
  double acc = 0.0;
  for (int s = 0; s < nsplit; ++s) acc += partial[((int64_t)pair * nsplit + s) * n_ent + ent];
  if (e == 0)
    out_rss[row] = acc;
  else
    out_jtj[((int64_t)row * kstride + (e - 1) / kstride) * kstride + (e - 1) % kstride] = acc;
}

// fill rows of a [n][kstride] f64 array with nan (gradients of pairs too wide for duals)
__global__ void fill_nan_rows(const int32_t* rows, int n_rows, int kstride, double* out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_rows * kstride) return;
  out[(int64_t)rows[idx / kstride] * kstride + idx % kstride] = __longlong_as_double(0x7ff8000000000000ll);
}

#endif  // VSR_API_TU

}  // namespace vsr

#endif  // VSR_KERNELS_CUH_
