// vsr_api.cu -- C ABI of libvsr.so (declared in include/vsr.h): handle, uploads, launch
// logic.  No torch types, no host synchronisation except in the *_host entry points.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <mutex>
#include <vector>

#include "../../include/vsr.h"
#define VSR_API_TU 1
#include "vsr_launch.h"

namespace {

constexpr int kWidths[] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 12, 16};
constexpr int kNumWidths = sizeof(kWidths) / sizeof(kWidths[0]);

int pick_width(int k) {
  for (int w : kWidths)
    if (w >= k) return w;
  return -1;
}

std::string g_create_error;

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);  // synchronises: nothing in flight can still use the old block
    p = nullptr;
    cap = 0;
    // generous first size and doubling: a cudaFree synchronises the whole device, which stalls a
    // caller that overlaps this handle's work with another handle's running fit
    size_t want = std::max(bytes * 2, (size_t)256 * 1024);
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

struct PinnedBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaEvent_t done = nullptr;  // last async copy that read from this buffer
  cudaError_t reserve(size_t bytes) {
    if (done) cudaEventSynchronize(done);
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    size_t want = std::max(bytes, (size_t)4096) * 2;
    cudaError_t e = cudaMallocHost(&p, want);
    if (e == cudaSuccess) cap = want;
    if (!done) cudaEventCreateWithFlags(&done, cudaEventDisableTiming);
    return e;
  }
  void release() {
    if (done) {
      cudaEventSynchronize(done);
      cudaEventDestroy(done);
    }
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    done = nullptr;
  }
};

struct PointSlot {
  const void* X = nullptr;
  const void* y = nullptr;
  const void* w = nullptr;  // per-point weights (vsr_set_weights), nullptr: unweighted
  int64_t n = 0, ldx = 0;
  int n_vars = 0;
  DevBuf ownX, ownY;
};

}  // namespace

// Side streams of the width-group launches: ONE pool per device, shared by the handles.  Every handle
// used to own eight streams; a process with many handles (bench.py keeps one per resident beam) then
// holds hundreds, which alias on the device's hardware queues (CUDA_DEVICE_MAX_CONNECTIONS, 8 by default
// and 32 at most): two launches of one fit landing in the same queue run one AFTER the other, and with
// persistent kernels the group tails add up (one beam of the bench: 65-75 ms alone, 95-160 ms in the
// bench process).  A handle takes a window of the pool at an offset of its own, so the handles that fit
// at the same time (refine_hypotheses stages a beam over up to four) do not meet.
constexpr int kPoolStreams = 32;
constexpr int kHandleStride = 8;   // side streams per handle (+ the caller's stream: nine groups at once; more groups share)
constexpr int kMaxGroups = 16;
struct StreamPool {
  std::mutex mu;
  std::vector<cudaStream_t> streams;  // created on first use, never destroyed (process lifetime)
  int next_base = 0;
};
StreamPool& pool_of(int device) {
  static StreamPool pools[64];
  return pools[device & 63];
}

struct vsr_handle {
  int device = 0;
  int stream_base = 0;  // this handle's window of the device's side-stream pool
  int num_sms = 148;
  std::string err;
  PointSlot pts[2];
  // programs
  DevBuf d_insns, d_insn_off, d_imms, d_imm_off, d_k;
  std::vector<int32_t> h_k, h_ninsn, h_nimm, h_nvars;
  std::vector<uint32_t> h_varmask;
  std::vector<cudaStream_t> side_streams;
  cudaEvent_t ev_fork = nullptr;
  std::vector<cudaEvent_t> ev_join;
  int n_programs = 0;
  // scratch
  DevBuf d_lists;    // grouped run / pair lists
  DevBuf d_partial;  // eval partial sums
  DevBuf d_stage;    // device staging of the *_host entry points
  DevBuf d_queue;    // one run counter per launch group (persistent clusters pull runs from it)
  DevBuf d_handover; // hand-over boards of the launch groups (vsr::Handover)
  PinnedBuf h_lists;
  int64_t launches = 0;
  int hook[4] = {0, 0, 0, 0};  // VSR_GEOMETRY measurement hook, read once in vsr_create
  int tile_smem_kb = 200;            // shared memory of an eval_tile_kernel CTA (fixed part + staged chunk)
  int64_t tile_min_points = 500000;  // vsr_eval / vsr_score share staged chunks between the pairs from this N on
  int steal_span = 3;          // a launch takes runs of groups up to this many tangent widths narrower
  int latency_k = 0;
  bool queue_by_candidate = false;
  bool handover = true;        // run hand-over to clusters that ran dry (VSR_HANDOVER=0: off)
  int hold_passes = 500;       // see FitArgs::hold_passes (VSR_HOLD_PASSES; 0 / 200 / 500 / 1000: 1044-1077 / 1040-1093 / 1011-1029 / 1028-1053 ms over 27 beams)
  // measurement hooks
  bool profiling = false;
  long long* phase_cycles = nullptr;  // optional device buffer [n_slots][8], see vsr_set_phase_buffer
  struct Span {
    cudaEvent_t a, b;
    int kind, n;
  };
  std::vector<Span> spans;
  std::vector<cudaEvent_t> event_pool;
};

namespace {

int fail(vsr_handle* h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (h)
    h->err = buf;
  else
    g_create_error = buf;
  return code;
}

cudaEvent_t take_event(vsr_handle* h) {
  if (!h->event_pool.empty()) {
    cudaEvent_t e = h->event_pool.back();
    h->event_pool.pop_back();
    return e;
  }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}

#define VSR_CUDA(h, expr)                                                              \
  do {                                                                                 \
    cudaError_t e_ = (expr);                                                           \
    if (e_ != cudaSuccess)                                                             \
      return fail(h, VSR_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), \
                  __FILE__, __LINE__);                                                 \
  } while (0)

vsr::ProgramTable table_of(const vsr_handle* h) {
  vsr::ProgramTable t;
  t.insns = (const vsr_insn_t*)h->d_insns.p;
  t.insn_off = (const int32_t*)h->d_insn_off.p;
  t.imms = (const double*)h->d_imms.p;
  t.imm_off = (const int32_t*)h->d_imm_off.p;
  t.k = (const int32_t*)h->d_k.p;
  return t;
}

vsr::Points points_of(const PointSlot& s) {
  vsr::Points p;
  p.X = s.X;
  p.y = s.y;
  p.n = s.n;
  p.ldx = s.ldx;
  return p;
}

using vsr::points_per_thread;

// the kernels are instantiated one (type, width) pair per translation unit (vsr_inst.cu) so the
// library builds in parallel; here only the dispatch over the runtime width
template <typename T>
cudaError_t launch_fit(int K, const vsr::FitArgs& a, int threads, int cs, size_t smem, int clusters, cudaStream_t st,
                       const void* w) {
  switch (K) {
#define C(KK) case KK: return vsr::launch_fit_T<T, KK>(a, threads, cs, smem, clusters, st, w);
    C(0) C(1) C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(12) C(16)
#undef C
  }
  return cudaErrorInvalidValue;
}

template <typename T>
int fit_threads_cap(int K) {
  switch (K) {
#define C(KK) case KK: return vsr::fit_max_threads<T, KK>();
    C(0) C(1) C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(12) C(16)
#undef C
  }
  return 256;
}

template <typename T>
cudaError_t launch_eval(int K, const vsr::EvalArgs& a, int threads, size_t smem, cudaStream_t st, const void* w) {
  switch (K) {
#define C(KK) case KK: return vsr::launch_eval_T<T, KK>(a, threads, smem, st, w);
    C(0) C(1) C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(12) C(16)
#undef C
  }
  return cudaErrorInvalidValue;
}

template <typename T>
cudaError_t launch_eval_tile(int K, const vsr::EvalTileArgs& a, size_t smem, cudaStream_t st, const void* w) {
  switch (K) {
#define C(KK) case KK: return vsr::launch_eval_tile_T<T, KK>(a, smem, st, w);
    C(0) C(1) C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(12) C(16)
#undef C
  }
  return cudaErrorInvalidValue;
}

template <typename T>
cudaError_t launch_predict(int K, const vsr::PredictArgs& a, size_t smem, cudaStream_t st) {
  switch (K) {
#define C(KK) case KK: return vsr::launch_predict_T<T, KK>(a, smem, st);
    C(0) C(1) C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(12) C(16)
#undef C
  }
  return cudaErrorInvalidValue;
}

cudaError_t launch_gram(int K, const vsr::GramArgs& a, size_t smem, cudaStream_t st, const void* w) {
  switch (K) {
#define C(KK) case KK: return vsr::launch_gram_K<KK>(a, smem, st, w);
    C(0) C(1) C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(12) C(16)
#undef C
  }
  return cudaErrorInvalidValue;
}

int eval_tile_threads_of(int K) {
  switch (K) {
#define C(KK) case KK: return vsr::eval_tile_threads<KK>();
    C(0) C(1) C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(12) C(16)
#undef C
  }
  return 512;
}

int next_pow2(int64_t v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// Geometry of a launch: persistent clusters of `cs` CTAs of `threads` threads, each cluster
// working on `seats` runs at a time, each CTA owning a contiguous slice of `stride` points.
// Aim: a sweep over the points is one or two tile iterations per thread (the critical path of a
// long run is passes x latency per pass), and the slice fits the CTA's shared memory so the
// points are read from HBM once per cluster.
struct Geometry {
  int cs, threads, stride, resident, seats, reserved;
  size_t smem;
};

constexpr int kMaxCluster = 16;             // 16 needs the non-portable cluster size opt-in
constexpr int kDefaultSeats = 4;            // runs in flight per cluster
constexpr size_t kSmemBudget = (VSR_FIT_MINCTAS == 1 ? 200 : 100) * 1024;  // per CTA, so that all co-resident CTAs keep their slices

// want_reserved: optimiser warps of the leader CTA that never sweep; 0 = default (a function of
// the CTA width), < 0 = none
Geometry choose_geometry(int64_t N, int P, int cap_threads, int forced_warps, int kmax, int K, int max_insn,
                         int n_cols, int elem, int max_cluster, int seats, int want_reserved) {
  Geometry g;
  const int64_t per_iter = (int64_t)cap_threads * P;
  int cs = 1;
  while (cs < max_cluster && (N + cs - 1) / cs > per_iter) cs <<= 1;
  int64_t per = (N + cs - 1) / cs;
  per = (per + 31) & ~(int64_t)31;
  int threads = (int)std::min<int64_t>(cap_threads, ((per + P - 1) / P + 31) & ~(int64_t)31);
  if (forced_warps > 0) threads = std::min(cap_threads, 32 * forced_warps);
  threads = std::max(32, threads);
  int nw = threads / 32;
  g.cs = cs;
  g.seats = std::max(1, std::min(seats, (int)vsr::kMaxSeats));
  // Optimiser warps.  A CTA wide enough gives the last `res` warps of the cluster's leader to the
  // optimiser turns for good (one per seat at the default width): they never sweep, so a turn never
  // holds a sweep up.  The leader's slice is sized for its remaining warps: CTAs 1..cs-1 take
  // `per` points, the leader the remainder.  The layout and the set of sweeping warps are functions
  // of (N, cluster size, CTA width) only, so a run's result does not depend on the number of seats,
  // on the queue order or on the other runs of the launch.
  g.reserved = 0;
  int res = want_reserved > 0 ? want_reserved : (want_reserved < 0 ? 0 : (nw >= 16 ? 4 : (nw >= 6 ? 2 : 0)));
  if (forced_warps > 0) res = 0;
  if (res > 0 && cs == 1 && threads + 32 * res <= cap_threads) {
    // a single CTA: the optimiser warps come on top of the warps the points need
    threads += 32 * res;
    nw = threads / 32;
    g.reserved = res;
  } else {
    // as many of the wanted warps as the points leave room for (N = 10 000 on 8 x 640 threads x 2
    // points leaves 240 point slots: three warps)
    for (; res > 0 && g.reserved == 0; --res) {
      if (nw <= res) continue;
      const int64_t denom = (int64_t)(cs - 1) * nw + (nw - res);
      int64_t per2 = (N * nw + denom - 1) / denom;
      per2 = (per2 + 31) & ~(int64_t)31;
      const int64_t lead = N - (int64_t)(cs - 1) * per2;
      // accept only if nobody needs more tile iterations than with equal slices
      const int64_t tile = (int64_t)threads * P, tile_lead = (int64_t)(nw - res) * 32 * P;
      const int64_t it0 = (per + tile - 1) / tile;
      const int64_t it_others = (per2 + tile - 1) / tile;
      const int64_t it_lead = lead > 0 ? (lead + tile_lead - 1) / tile_lead : 0;
      if (it_others <= it0 && it_lead <= it0 && lead <= per2 && lead >= 0) {
        per = per2;
        g.reserved = res;
      }
    }
  }
  g.threads = threads;
  g.stride = (int)per;
  const size_t with = vsr::fit_smem_bytes(g.seats, kmax, K, nw, cs, max_insn, n_cols, (int)per, elem);
  g.resident = with <= kSmemBudget && per < (1 << 30);
  g.smem = g.resident ? with : vsr::fit_smem_bytes(g.seats, kmax, K, nw, cs, max_insn, -1, 0, elem);
  return g;
}

struct Group {
  int K;
  int grad_mode;
  std::vector<int32_t> prog, slot;
  int kmax = 0, max_insn = 0, max_imm = 0;
  unsigned var_mask = 0;  // variables any of the group's programs reads
};

// copies host int32 lists into the handle's device list buffer at `offset` (in ints)
int stage_lists(vsr_handle* h, const std::vector<int32_t>& all, cudaStream_t st) {
  const size_t bytes = all.size() * sizeof(int32_t);
  VSR_CUDA(h, h->h_lists.reserve(bytes));
  VSR_CUDA(h, h->d_lists.reserve(bytes));
  std::memcpy(h->h_lists.p, all.data(), bytes);
  VSR_CUDA(h, cudaMemcpyAsync(h->d_lists.p, h->h_lists.p, bytes, cudaMemcpyHostToDevice, st));
  VSR_CUDA(h, cudaEventRecord(h->h_lists.done, st));
  return VSR_OK;
}

// eval over explicit (prog, row, out) triples, all of one tangent width
int run_eval_group(vsr_handle* h, int K, int dtype, const int32_t* d_prog, const int32_t* d_row,
                   const int32_t* d_out, int n_pairs, int kmax, int max_insn, int max_imm,
                   const double* consts, int kstride, double* out_loss, double* out_grad,
                   cudaStream_t st, int nan_to_num = 0, unsigned var_mask = 0, const void* w = nullptr) {
  // w: the slot's weights for a weighted loss and gradient (nullptr: unweighted)
  const PointSlot& ps = h->pts[dtype];
  const int P = points_per_thread(K);
  const int64_t N = ps.n;
  // Large N and several pairs: chunks of the points staged once per CTA and shared by all pairs
  // (eval_tile_kernel).  The choice is a function of (N, number of pairs, columns) only.
  if (N >= h->tile_min_points && n_pairs >= 8) {
    const int elem = dtype == VSR_F64 ? 8 : 4;
    if (var_mask == 0) var_mask = ps.n_vars >= 32 ? 0xffffffffu : ((1u << ps.n_vars) - 1u);
    vsr::EvalTileArgs t;
    t.n_cols = 0;
    for (int j = 0; j < VSR_MAX_VARS; ++j) t.col_of_var[j] = (((var_mask >> j) & 1u) && j < ps.n_vars) ? t.n_cols++ : -1;
    const int threads = eval_tile_threads_of(K);
    const size_t fixed = vsr::eval_tile_fixed_doubles(K, threads, max_insn) * 8;
    const size_t budget = (size_t)h->tile_smem_kb * 1024;
    if (fixed + (size_t)(t.n_cols + 1) * 1024 * elem <= budget) {
      int64_t cap = (int64_t)((budget - fixed) / ((size_t)(t.n_cols + 1) * elem));  // points a CTA can hold
      cap &= ~(int64_t)127;
      int64_t chunks = (N + cap - 1) / cap;
      chunks = (chunks + h->num_sms - 1) / h->num_sms * h->num_sms;  // whole waves of one CTA per SM
      int64_t chunk = (N + chunks - 1) / chunks;
      chunk = (chunk + 127) & ~(int64_t)127;
      chunks = (N + chunk - 1) / chunk;
      VSR_CUDA(h, h->d_partial.reserve((size_t)n_pairs * chunks * (K + 1) * sizeof(double)));
      t.e.pt = table_of(h);
      t.e.pts = points_of(ps);
      t.e.pair_prog = d_prog;
      t.e.pair_row = d_row;
      t.e.pair_out = d_out;
      t.e.n_pairs = n_pairs;
      t.e.kstride = kstride;
      t.e.consts = consts;
      t.e.partial = (double*)h->d_partial.p;
      t.e.nsplit = (int)chunks;
      t.e.nan_to_num = nan_to_num;
      t.chunk = (int)chunk;
      t.stride = (int)chunk;
      t.tma_ok = (((uintptr_t)ps.X % 16 == 0) && ((uintptr_t)ps.y % 16 == 0) && ((ps.ldx * elem) % 16 == 0)) ? 1 : 0;
      t.max_insn = max_insn;
      // (a weighted launch reads the weights from global memory: the same chunks, so w = 1 gives the
      // unweighted sums bit for bit)
      const size_t smem = fixed + (size_t)(t.n_cols + 1) * chunk * elem;
      cudaError_t e = dtype == VSR_F64 ? launch_eval_tile<double>(K, t, smem, st, w) : launch_eval_tile<float>(K, t, smem, st, w);
      if (e != cudaSuccess) return fail(h, VSR_ECUDA, "eval tile kernel launch failed (smem %zu): %s", smem, cudaGetErrorString(e));
      const int total = n_pairs * (K + 1);
      vsr::eval_finalize<<<(total + 127) / 128, 128, 0, st>>>(t.e.partial, d_prog, d_out, t.e.pt.k, n_pairs, (int)chunks, K,
                                                               kstride, 1.0 / (double)N, out_loss, out_grad);
      VSR_CUDA(h, cudaGetLastError());
      h->launches += 2;
      return VSR_OK;
    }
  }
  int threads = 32 * std::min<int64_t>(8, std::max<int64_t>(1, next_pow2((N + 32 * P * 4 - 1) / (32 * P * 4))));
  const int64_t tile = (int64_t)threads * P;
  const int64_t tiles = (N + tile - 1) / tile;
  // split the points when there are too few pairs to fill the machine
  int nsplit = 1;
  const int64_t target = (int64_t)h->num_sms * 8;
  if (n_pairs < target) nsplit = (int)std::min<int64_t>(std::max<int64_t>(1, tiles / 8), (target + n_pairs - 1) / n_pairs);
  nsplit = std::max(1, std::min(nsplit, 65535));
  VSR_CUDA(h, h->d_partial.reserve((size_t)n_pairs * nsplit * (K + 1) * sizeof(double)));
  vsr::EvalArgs a;
  a.pt = table_of(h);
  a.pts = points_of(ps);
  a.pair_prog = d_prog;
  a.pair_row = d_row;
  a.pair_out = d_out;
  a.n_pairs = n_pairs;
  a.kstride = kstride;
  a.consts = consts;
  a.partial = (double*)h->d_partial.p;
  a.nsplit = nsplit;
  a.nan_to_num = nan_to_num;
  const size_t smem = sizeof(double) * (size_t)((K + 1) * threads + kmax + 2 + max_imm + max_insn + 1);  // + pad word
  cudaError_t e = dtype == VSR_F64 ? launch_eval<double>(K, a, threads, smem, st, w)
                                   : launch_eval<float>(K, a, threads, smem, st, w);
  if (e != cudaSuccess) return fail(h, VSR_ECUDA, "eval kernel launch failed: %s", cudaGetErrorString(e));
  const int total = n_pairs * (K + 1);
  vsr::eval_finalize<<<(total + 127) / 128, 128, 0, st>>>(
      a.partial, d_prog, d_out, a.pt.k, n_pairs, nsplit, K, kstride, 1.0 / (double)N, out_loss,
      out_grad);
  VSR_CUDA(h, cudaGetLastError());
  h->launches += 2;
  return VSR_OK;
}

// a program that reads x_j with j >= the uploaded n_vars would read past the last column
int check_vars(vsr_handle* h, int prog, int dtype) {
  const int nv = h->pts[dtype].n_vars;
  if (nv < VSR_MAX_VARS && (h->h_varmask[prog] >> nv) != 0u)
    return fail(h, VSR_EINVAL, "program %d reads a variable beyond the %d uploaded columns (dtype %d)", prog, nv, dtype);
  return VSR_OK;
}

int check_ready(vsr_handle* h, int dtype) {
  if (!h) return VSR_EINVAL;
  if (dtype != VSR_F64 && dtype != VSR_F32) return fail(h, VSR_EINVAL, "dtype must be VSR_F64 or VSR_F32");
  if (h->n_programs <= 0) return fail(h, VSR_ESTATE, "no programs uploaded");
  if (!h->pts[dtype].X || h->pts[dtype].n <= 0)
    return fail(h, VSR_ESTATE, "no points uploaded for dtype %d", dtype);
  return VSR_OK;
}

}  // namespace

extern "C" {

int vsr_abi_version(void) { return VSR_ABI_VERSION; }

void vsr_fit_opts_default(vsr_fit_opts* o) {
  if (!o) return;
  o->gtol = 1e-5;
  o->c1 = 1e-4;
  o->c2 = 0.9;
  o->xrtol = 0.0;
  o->fd_eps = 1.4901161193847656e-08;
  o->penalty = 1e6;
  o->loss_scale = 1.0;
  o->stop_time = 1e9;
  o->maxiter_per_k = 200;
  o->grad_mode = VSR_GRAD_DUAL;
  o->eval_dtype = VSR_F64;
  o->score_dtype = VSR_F64;
  o->warps_per_run = 0;
  o->reserved = 0;
}

int vsr_create(int device, vsr_handle** out) {
  if (!out) return VSR_EINVAL;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0)
    return fail(nullptr, VSR_ECUDA, "no CUDA device (%s); libvsr has no CPU path",
                e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
  if (device < 0 || device >= count) return fail(nullptr, VSR_EINVAL, "device %d out of range [0,%d)", device, count);
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(nullptr, VSR_ECUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return fail(nullptr, VSR_ECUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, VSR_ECUDA, "device %d is sm_%d%d; libvsr is built for sm_100a only", device,
                prop.major, prop.minor);
  // Load every kernel instantiation now (CUDA loads modules lazily: the first launch of each of
  // the 44 kernels would otherwise stall a fit by milliseconds), once per process and device.
  static bool preloaded[64] = {false};
  if (device < 64 && !preloaded[device]) {
#define C(KK)                                                        \
  if (e == cudaSuccess) e = vsr::preload_T<double, KK>();            \
  if (e == cudaSuccess) e = vsr::preload_T<float, KK>();
    C(0) C(1) C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(12) C(16)
#undef C
    if (e != cudaSuccess) return fail(nullptr, VSR_ECUDA, "loading the kernels: %s", cudaGetErrorString(e));
    preloaded[device] = true;
  }
  vsr_handle* h = new (std::nothrow) vsr_handle();
  if (!h) return fail(nullptr, VSR_ENOMEM, "out of host memory");
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  if (const char* env = getenv("VSR_GEOMETRY")) sscanf(env, "%d:%d:%d:%d", &h->hook[0], &h->hook[1], &h->hook[2], &h->hook[3]);
  if (const char* env = getenv("VSR_STEAL_SPAN")) h->steal_span = atoi(env);
  if (const char* env = getenv("VSR_TILE_MIN_POINTS")) h->tile_min_points = atoll(env);  // measurement / test hook
  if (const char* env = getenv("VSR_TILE_SMEM_KB")) h->tile_smem_kb = std::max(48, std::min(220, atoi(env)));
  if (const char* env = getenv("VSR_LATENCY_K")) h->latency_k = atoi(env);
  h->queue_by_candidate = getenv("VSR_QUEUE_BY_CANDIDATE") != nullptr;
  if (const char* env = getenv("VSR_HOLD_PASSES")) h->hold_passes = atoi(env);
  if (const char* env = getenv("VSR_HANDOVER")) h->handover = atoi(env) != 0;
  // scratch every fit needs, allocated here rather than inside the first fit: run lists (pinned
  // + device), run counters, eval partials, the side streams and their events
  e = h->h_lists.reserve(256 << 10);
  if (e == cudaSuccess) e = h->d_lists.reserve(256 << 10);
  if (e == cudaSuccess) e = h->d_queue.reserve(64 * sizeof(int32_t));
  if (e == cudaSuccess) e = h->d_partial.reserve(1 << 20);
  if (e == cudaSuccess) e = h->d_handover.reserve(2 << 20);
  {
    StreamPool& sp = pool_of(device);
    std::lock_guard<std::mutex> lock(sp.mu);
    while ((int)sp.streams.size() < kPoolStreams && e == cudaSuccess) {
      cudaStream_t s2;
      e = cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking);
      if (e == cudaSuccess) sp.streams.push_back(s2);
    }
    h->stream_base = sp.next_base;
    sp.next_base = (sp.next_base + kHandleStride) % kPoolStreams;
    for (int i = 0; i < kHandleStride; ++i) h->side_streams.push_back(sp.streams[(h->stream_base + i) % kPoolStreams]);
    for (int i = 0; i < kMaxGroups && e == cudaSuccess; ++i) {
      cudaEvent_t e2;
      e = cudaEventCreateWithFlags(&e2, cudaEventDisableTiming);
      if (e == cudaSuccess) h->ev_join.push_back(e2);
    }
  }
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
  if (e != cudaSuccess) {
    fail(nullptr, VSR_ECUDA, "allocating the handle's scratch: %s", cudaGetErrorString(e));
    vsr_destroy(h);
    return VSR_ECUDA;
  }
  *out = h;
  return VSR_OK;
}

void vsr_destroy(vsr_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  for (auto& s : h->pts) {
    s.ownX.release();
    s.ownY.release();
  }
  h->d_insns.release();
  h->d_insn_off.release();
  h->d_imms.release();
  h->d_imm_off.release();
  h->d_k.release();
  h->d_lists.release();
  h->d_partial.release();
  h->d_stage.release();
  h->d_queue.release();
  h->d_handover.release();
  h->h_lists.release();
  for (auto e2 : h->ev_join) cudaEventDestroy(e2);  // (the side streams belong to the device's pool)
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  for (auto& sp : h->spans) {
    if (sp.kind == 0) h->event_pool.push_back(sp.a);
    h->event_pool.push_back(sp.b);
  }
  for (auto e : h->event_pool) cudaEventDestroy(e);
  delete h;
}

const char* vsr_last_error(const vsr_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int64_t vsr_launch_count(const vsr_handle* h) { return h ? h->launches : 0; }

int vsr_set_phase_buffer(vsr_handle* h, void* dev_i64_nslots_by_8) {
  if (!h) return VSR_EINVAL;
  h->phase_cycles = (long long*)dev_i64_nslots_by_8;
  return VSR_OK;
}

int vsr_set_geometry(vsr_handle* h, int32_t cluster, int32_t threads, int32_t seats, int32_t opt_warps) {
  if (!h) return VSR_EINVAL;
  h->hook[0] = cluster;
  h->hook[1] = threads;
  h->hook[2] = seats;
  h->hook[3] = opt_warps;
  return VSR_OK;
}

int vsr_set_profiling(vsr_handle* h, int32_t on) {
  if (!h) return VSR_EINVAL;
  h->profiling = on != 0;
  return VSR_OK;
}

int vsr_read_profile(vsr_handle* h, double out[4]) {
  if (!h || !out) return VSR_EINVAL;
  out[0] = out[1] = out[2] = out[3] = 0.0;
  // spans come in (fit, score) pairs sharing the middle event; ev_c closes the pair
  for (size_t i = 0; i < h->spans.size(); ++i) {
    auto& sp = h->spans[i];
    VSR_CUDA(h, cudaEventSynchronize(sp.b));
    float ms = 0.f;
    VSR_CUDA(h, cudaEventElapsedTime(&ms, sp.a, sp.b));
    out[sp.kind * 2] += ms;
    out[sp.kind * 2 + 1] += sp.n;
  }
  for (size_t i = 0; i < h->spans.size(); ++i) {
    if (h->spans[i].kind == 0) h->event_pool.push_back(h->spans[i].a);
    h->event_pool.push_back(h->spans[i].b);
  }
  h->spans.clear();
  return VSR_OK;
}

int vsr_set_points(vsr_handle* h, const void* X_dev, const void* y_dev, int64_t n_points,
                   int64_t ldx, int32_t n_vars, int32_t dtype) {
  if (!h) return VSR_EINVAL;
  if (dtype != VSR_F64 && dtype != VSR_F32) return fail(h, VSR_EINVAL, "bad dtype %d", dtype);
  if (!X_dev || !y_dev || n_points <= 0 || ldx < n_points || n_vars < 1 || n_vars > VSR_MAX_VARS)
    return fail(h, VSR_EINVAL, "bad points: n=%lld ldx=%lld n_vars=%d", (long long)n_points,
                (long long)ldx, n_vars);
  PointSlot& s = h->pts[dtype];
  s.X = X_dev;
  s.y = y_dev;
  s.w = nullptr;
  s.n = n_points;
  s.ldx = ldx;
  s.n_vars = n_vars;
  return VSR_OK;
}

int vsr_upload_points(vsr_handle* h, const void* X_host, const void* y_host, int64_t n_points,
                      int64_t ldx, int32_t n_vars, int32_t dtype, void* stream) {
  if (!h) return VSR_EINVAL;
  if (dtype != VSR_F64 && dtype != VSR_F32) return fail(h, VSR_EINVAL, "bad dtype %d", dtype);
  if (!X_host || !y_host || n_points <= 0 || ldx < n_points || n_vars < 1 || n_vars > VSR_MAX_VARS)
    return fail(h, VSR_EINVAL, "bad points: n=%lld ldx=%lld n_vars=%d", (long long)n_points,
                (long long)ldx, n_vars);
  cudaStream_t st = (cudaStream_t)stream;
  VSR_CUDA(h, cudaSetDevice(h->device));
  const size_t es = dtype == VSR_F64 ? 8 : 4;
  PointSlot& s = h->pts[dtype];
  // device copy keeps columns 16-byte aligned: pad the column stride to a multiple of 4
  const int64_t dld = (n_points + 3) & ~(int64_t)3;
  VSR_CUDA(h, s.ownX.reserve((size_t)dld * n_vars * es));
  VSR_CUDA(h, s.ownY.reserve((size_t)dld * es));
  VSR_CUDA(h, cudaMemcpy2DAsync(s.ownX.p, dld * es, X_host, ldx * es, n_points * es, n_vars,
                                cudaMemcpyHostToDevice, st));
  VSR_CUDA(h, cudaMemcpyAsync(s.ownY.p, y_host, n_points * es, cudaMemcpyHostToDevice, st));
  s.X = s.ownX.p;
  s.y = s.ownY.p;
  s.w = nullptr;
  s.n = n_points;
  s.ldx = dld;
  s.n_vars = n_vars;
  return VSR_OK;
}

int vsr_set_weights(vsr_handle* h, const void* w_dev, int64_t n_points, int32_t dtype) {
  if (!h) return VSR_EINVAL;
  if (dtype != VSR_F64 && dtype != VSR_F32) return fail(h, VSR_EINVAL, "bad dtype %d", dtype);
  PointSlot& s = h->pts[dtype];
  if (!s.X || s.n <= 0) return fail(h, VSR_ESTATE, "no points uploaded for dtype %d", dtype);
  if (w_dev && n_points != s.n)
    return fail(h, VSR_EINVAL, "%lld weights for %lld points (dtype %d)", (long long)n_points, (long long)s.n, dtype);
  s.w = w_dev;
  return VSR_OK;
}

int vsr_upload_programs(vsr_handle* h, const uint64_t* insns, const int32_t* insn_off,
                        const double* imms, const int32_t* imm_off, const int32_t* k,
                        int32_t n_programs, void* stream) {
  if (!h) return VSR_EINVAL;
  if (!insns || !insn_off || !imms || !imm_off || !k || n_programs <= 0)
    return fail(h, VSR_EINVAL, "bad program table");
  cudaStream_t st = (cudaStream_t)stream;
  VSR_CUDA(h, cudaSetDevice(h->device));
  h->n_programs = 0;
  h->h_k.assign(k, k + n_programs);
  h->h_ninsn.resize(n_programs);
  h->h_nimm.resize(n_programs);
  h->h_nvars.assign(n_programs, 0);
  h->h_varmask.assign(n_programs, 0u);
  for (int c = 0; c < n_programs; ++c) {
    const int ni = insn_off[c + 1] - insn_off[c];
    const int nm = imm_off[c + 1] - imm_off[c];
    if (ni < 1 || ni > VSR_MAX_INSNS || nm < 0 || nm > VSR_MAX_IMMS || k[c] < 0 || k[c] > VSR_MAX_CONSTS)
      return fail(h, VSR_ELIMIT, "program %d: %d insns, %d literals, %d constants", c, ni, nm, k[c]);
    if (VSR_OP(insns[insn_off[c + 1] - 1]) != VSR_END)
      return fail(h, VSR_EINVAL, "program %d does not end in END", c);
    // static check of operand indices and stack discipline: the kernels trust the table
    int sp = 0;
    unsigned var_mask = 0;
    for (int i = insn_off[c]; i < insn_off[c + 1]; ++i) {
      const unsigned op = VSR_OP(insns[i]), src = VSR_SRC(insns[i]), idx = VSR_IDX(insns[i]);
      if (op >= VSR_OP_COUNT) return fail(h, VSR_EINVAL, "program %d: bad opcode %u", c, op);
      if (op == VSR_PUSH && ++sp > VSR_MAX_STACK) return fail(h, VSR_ELIMIT, "program %d: stack too deep", c);
      if (op >= VSR_LOAD && op <= VSR_RPOW && op != VSR_PUSH) {
        if (src == VSR_SRC_STACK) {
          if (--sp < 0) return fail(h, VSR_EINVAL, "program %d: stack underflow", c);
        } else if (src == VSR_SRC_VAR) {
          if (idx >= VSR_MAX_VARS) return fail(h, VSR_EINVAL, "program %d: variable %u", c, idx);
          var_mask |= 1u << idx;
        } else if (src == VSR_SRC_CONST) {
          if ((int)idx >= k[c]) return fail(h, VSR_EINVAL, "program %d: constant %u of %d", c, idx, k[c]);
        } else if (src == VSR_SRC_IMM) {
          if ((int)idx >= nm) return fail(h, VSR_EINVAL, "program %d: literal %u of %d", c, idx, nm);
        } else {
          return fail(h, VSR_EINVAL, "program %d: bad operand source %u", c, src);
        }
      }
    }
    h->h_ninsn[c] = ni;
    h->h_nimm[c] = nm;
    h->h_nvars[c] = __builtin_popcount(var_mask);
    h->h_varmask[c] = var_mask;
  }
  const size_t nins = insn_off[n_programs], nimm = std::max(1, imm_off[n_programs]);
  VSR_CUDA(h, h->d_insns.reserve(nins * sizeof(uint64_t)));
  VSR_CUDA(h, h->d_insn_off.reserve((n_programs + 1) * sizeof(int32_t)));
  VSR_CUDA(h, h->d_imms.reserve(nimm * sizeof(double)));
  VSR_CUDA(h, h->d_imm_off.reserve((n_programs + 1) * sizeof(int32_t)));
  VSR_CUDA(h, h->d_k.reserve(n_programs * sizeof(int32_t)));
  // pageable sources: cudaMemcpyAsync stages them before returning
  VSR_CUDA(h, cudaMemcpyAsync(h->d_insns.p, insns, nins * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
  VSR_CUDA(h, cudaMemcpyAsync(h->d_insn_off.p, insn_off, (n_programs + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  if (imm_off[n_programs] > 0)
    VSR_CUDA(h, cudaMemcpyAsync(h->d_imms.p, imms, imm_off[n_programs] * sizeof(double), cudaMemcpyHostToDevice, st));
  VSR_CUDA(h, cudaMemcpyAsync(h->d_imm_off.p, imm_off, (n_programs + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  VSR_CUDA(h, cudaMemcpyAsync(h->d_k.p, k, n_programs * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  h->n_programs = n_programs;
  return VSR_OK;
}

int vsr_eval(vsr_handle* h, const int32_t* prog_idx, const int32_t* const_row, int32_t n_pairs,
             const double* consts, int32_t kstride, int32_t dtype, double* out_loss,
             double* out_grad, void* stream) {
  int rc = check_ready(h, dtype);
  if (rc) return rc;
  if (!prog_idx || n_pairs <= 0 || !out_loss || kstride < 0 || (!consts && kstride > 0))
    return fail(h, VSR_EINVAL, "bad eval arguments");
  cudaStream_t st = (cudaStream_t)stream;
  VSR_CUDA(h, cudaSetDevice(h->device));
  // group pairs by tangent width (value only: one group of width 0)
  std::vector<Group> groups(kNumWidths + 1);
  for (int i = 0; i < kNumWidths; ++i) groups[i].K = kWidths[i];
  Group& toowide = groups[kNumWidths];
  for (int p = 0; p < n_pairs; ++p) {
    const int c = prog_idx[p];
    if (c < 0 || c >= h->n_programs) return fail(h, VSR_EINVAL, "pair %d: program %d out of range", p, c);
    const int k = h->h_k[c];
    if (k > kstride) return fail(h, VSR_EINVAL, "pair %d: %d constants > kstride %d", p, k, kstride);
    if ((rc = check_vars(h, c, dtype))) return rc;
    int gi = 0;
    if (out_grad) {
      const int w = pick_width(k);
      if (w < 0) {
        toowide.prog.push_back(p);
        gi = 0;  // value through the width-0 kernel, gradient row = nan
      } else {
        gi = (int)(std::find(kWidths, kWidths + kNumWidths, w) - kWidths);
      }
    }
    Group& g = groups[gi];
    g.prog.push_back(c);
    g.slot.push_back(const_row ? const_row[p] : p);  // row of consts
    g.kmax = std::max(g.kmax, k);
    g.max_insn = std::max(g.max_insn, h->h_ninsn[c]);
    g.max_imm = std::max(g.max_imm, h->h_nimm[c]);
    g.var_mask |= h->h_varmask[c];
  }
  // lists: for each group prog | row | out
  std::vector<int32_t> all;
  std::vector<size_t> off(kNumWidths + 1, 0);
  std::vector<std::vector<int32_t>> outs(kNumWidths);
  {
    // recompute output rows per group in the same order as above
    std::vector<int> cursor(kNumWidths, 0);
    for (auto& o : outs) o.clear();
    for (int p = 0; p < n_pairs; ++p) {
      const int k = h->h_k[prog_idx[p]];
      int gi = 0;
      if (out_grad) {
        const int w = pick_width(k);
        if (w >= 0) gi = (int)(std::find(kWidths, kWidths + kNumWidths, w) - kWidths);
      }
      outs[gi].push_back(p);
    }
  }
  for (int gi = 0; gi < kNumWidths; ++gi) {
    off[gi] = all.size();
    Group& g = groups[gi];
    all.insert(all.end(), g.prog.begin(), g.prog.end());
    all.insert(all.end(), g.slot.begin(), g.slot.end());
    all.insert(all.end(), outs[gi].begin(), outs[gi].end());
  }
  off[kNumWidths] = all.size();
  all.insert(all.end(), toowide.prog.begin(), toowide.prog.end());
  rc = stage_lists(h, all, st);
  if (rc) return rc;
  const int32_t* dl = (const int32_t*)h->d_lists.p;
  for (int gi = 0; gi < kNumWidths; ++gi) {
    Group& g = groups[gi];
    const int n = (int)g.prog.size();
    if (!n) continue;
    rc = run_eval_group(h, g.K, dtype, dl + off[gi], dl + off[gi] + n, dl + off[gi] + 2 * n, n,
                        g.kmax, g.max_insn, g.max_imm, consts, kstride, out_loss,
                        g.K > 0 ? out_grad : nullptr, st, 0, g.var_mask, h->pts[dtype].w);
    if (rc) return rc;
  }
  if (out_grad && !toowide.prog.empty()) {
    const int n = (int)toowide.prog.size();
    vsr::fill_nan_rows<<<(n * kstride + 127) / 128, 128, 0, st>>>(dl + off[kNumWidths], n, kstride, out_grad);
    VSR_CUDA(h, cudaGetLastError());
    h->launches += 1;
  }
  if (out_grad) {
    // width-0 pairs (k == 0) have no gradient entries to write
  }
  return VSR_OK;
}

int vsr_gram(vsr_handle* h, const int32_t* prog_idx, const int32_t* const_row, int32_t n_pairs,
             const double* consts, int32_t kstride, double* out_rss, double* out_jtj, void* stream) {
  int rc = check_ready(h, VSR_F64);
  if (rc) return rc;
  if (!prog_idx || n_pairs <= 0 || !out_rss || kstride < 0 || ((!consts || !out_jtj) && kstride > 0))
    return fail(h, VSR_EINVAL, "bad gram arguments");
  cudaStream_t st = (cudaStream_t)stream;
  VSR_CUDA(h, cudaSetDevice(h->device));
  // group pairs by tangent width; programs wider than VSR_MAX_DUAL go with the width-0 group (rss
  // only, gram_finalize writes their jtj as nan)
  std::vector<Group> groups(kNumWidths);
  std::vector<std::vector<int32_t>> outs(kNumWidths);
  for (int i = 0; i < kNumWidths; ++i) groups[i].K = kWidths[i];
  for (int p = 0; p < n_pairs; ++p) {
    const int c = prog_idx[p];
    if (c < 0 || c >= h->n_programs) return fail(h, VSR_EINVAL, "pair %d: program %d out of range", p, c);
    const int k = h->h_k[c];
    if (k > kstride) return fail(h, VSR_EINVAL, "pair %d: %d constants > kstride %d", p, k, kstride);
    if ((rc = check_vars(h, c, VSR_F64))) return rc;
    const int w = pick_width(k);
    const int gi = w < 0 ? 0 : (int)(std::find(kWidths, kWidths + kNumWidths, w) - kWidths);
    Group& g = groups[gi];
    g.prog.push_back(c);
    g.slot.push_back(const_row ? const_row[p] : p);
    g.kmax = std::max(g.kmax, k);
    g.max_insn = std::max(g.max_insn, h->h_ninsn[c]);
    g.max_imm = std::max(g.max_imm, h->h_nimm[c]);
    outs[gi].push_back(p);
  }
  std::vector<int32_t> all;
  std::vector<size_t> off(kNumWidths, 0);
  for (int gi = 0; gi < kNumWidths; ++gi) {
    off[gi] = all.size();
    all.insert(all.end(), groups[gi].prog.begin(), groups[gi].prog.end());
    all.insert(all.end(), groups[gi].slot.begin(), groups[gi].slot.end());
    all.insert(all.end(), outs[gi].begin(), outs[gi].end());
  }
  rc = stage_lists(h, all, st);
  if (rc) return rc;
  const int32_t* dl = (const int32_t*)h->d_lists.p;
  const PointSlot& ps = h->pts[VSR_F64];
  // the groups share the partial buffer: size it for all of them at once, so that a reserve (which
  // frees the old block) never happens while an earlier group's partials are still to be summed
  size_t need = 0;
  for (int gi = 0; gi < kNumWidths; ++gi) {
    const int K = groups[gi].K;
    const int nsplit = vsr::gram_nsplit(ps.n, (int64_t)vsr::kGramThreads * points_per_thread(K));
    need += groups[gi].prog.size() * (size_t)nsplit * vsr::gram_entries(K);
  }
  VSR_CUDA(h, h->d_partial.reserve(need * sizeof(double)));
  double* partial = (double*)h->d_partial.p;
  for (int gi = 0; gi < kNumWidths; ++gi) {
    const Group& g = groups[gi];
    const int n = (int)g.prog.size();
    if (!n) continue;
    const int K = g.K;
    const int tile = vsr::kGramThreads * points_per_thread(K);
    vsr::GramArgs a;
    a.pt = table_of(h);
    a.pts = points_of(ps);
    a.pair_prog = dl + off[gi];
    a.pair_row = dl + off[gi] + n;
    a.n_pairs = n;
    a.kstride = kstride;
    a.consts = consts;
    a.partial = partial;
    a.nsplit = vsr::gram_nsplit(ps.n, tile);
    const size_t cols = (size_t)(K + 1) + (ps.w ? 1 : 0);  // r, J (and w)
    const size_t smem = sizeof(double) * (cols * vsr::gram_col_stride(tile) + g.kmax + 1 + g.max_imm) +
                        sizeof(vsr_insn_t) * (g.max_insn + 1);
    cudaError_t e = launch_gram(K, a, smem, st, ps.w);
    if (e != cudaSuccess) return fail(h, VSR_ECUDA, "gram kernel launch failed: %s", cudaGetErrorString(e));
    const int64_t total = (int64_t)n * (1 + (int64_t)kstride * kstride);
    vsr::gram_finalize<<<(unsigned)((total + 127) / 128), 128, 0, st>>>(partial, a.pair_prog, dl + off[gi] + 2 * n,
                                                                         a.pt.k, n, a.nsplit, K, kstride, out_rss,
                                                                         out_jtj);
    VSR_CUDA(h, cudaGetLastError());
    h->launches += 2;
    partial += (size_t)n * a.nsplit * vsr::gram_entries(K);
  }
  return VSR_OK;
}

int vsr_predict(vsr_handle* h, const int32_t* prog_idx, const int32_t* const_row, int32_t n_pairs,
                const double* consts, int32_t kstride, const double* cov, int32_t dtype,
                double* out_value, double* out_var, int64_t ld_out, void* stream) {
  int rc = check_ready(h, dtype);
  if (rc) return rc;
  const PointSlot& ps = h->pts[dtype];
  if (!prog_idx || n_pairs <= 0 || !out_value || kstride < 0 || (!consts && kstride > 0) ||
      (!cov) != (!out_var) || ld_out < ps.n)
    return fail(h, VSR_EINVAL, "bad predict arguments");
  cudaStream_t st = (cudaStream_t)stream;
  VSR_CUDA(h, cudaSetDevice(h->device));
  // group pairs by tangent width; without a covariance, and for programs wider than VSR_MAX_DUAL,
  // the width-0 group (values only; its variance row is 0 for k == 0 and nan otherwise)
  std::vector<Group> groups(kNumWidths);
  std::vector<std::vector<int32_t>> outs(kNumWidths);
  for (int i = 0; i < kNumWidths; ++i) groups[i].K = kWidths[i];
  for (int p = 0; p < n_pairs; ++p) {
    const int c = prog_idx[p];
    if (c < 0 || c >= h->n_programs) return fail(h, VSR_EINVAL, "pair %d: program %d out of range", p, c);
    const int k = h->h_k[c];
    if (k > kstride) return fail(h, VSR_EINVAL, "pair %d: %d constants > kstride %d", p, k, kstride);
    if ((rc = check_vars(h, c, dtype))) return rc;
    const int w = out_var ? pick_width(k) : 0;
    const int gi = w < 0 ? 0 : (int)(std::find(kWidths, kWidths + kNumWidths, w) - kWidths);
    Group& g = groups[gi];
    g.prog.push_back(c);
    g.slot.push_back(const_row ? const_row[p] : p);
    g.kmax = std::max(g.kmax, k);
    g.max_insn = std::max(g.max_insn, h->h_ninsn[c]);
    g.max_imm = std::max(g.max_imm, h->h_nimm[c]);
    outs[gi].push_back(p);
  }
  std::vector<int32_t> all;
  std::vector<size_t> off(kNumWidths, 0);
  for (int gi = 0; gi < kNumWidths; ++gi) {
    off[gi] = all.size();
    all.insert(all.end(), groups[gi].prog.begin(), groups[gi].prog.end());
    all.insert(all.end(), groups[gi].slot.begin(), groups[gi].slot.end());
    all.insert(all.end(), outs[gi].begin(), outs[gi].end());
  }
  rc = stage_lists(h, all, st);
  if (rc) return rc;
  const int32_t* dl = (const int32_t*)h->d_lists.p;
  for (int gi = 0; gi < kNumWidths; ++gi) {
    const Group& g = groups[gi];
    const int n = (int)g.prog.size();
    if (!n) continue;
    const int K = g.K;
    const int64_t tile = (int64_t)vsr::kPredictThreads * points_per_thread(K);
    const int64_t tiles = (ps.n + tile - 1) / tile;
    // splits of the points: enough CTAs to fill the machine several times over (no result depends
    // on this choice)
    const int64_t want = ((int64_t)h->num_sms * 32 + n - 1) / n;
    vsr::PredictArgs a;
    a.pt = table_of(h);
    a.pts = points_of(ps);
    a.pair_prog = dl + off[gi];
    a.pair_row = dl + off[gi] + n;
    a.pair_out = dl + off[gi] + 2 * n;
    a.n_pairs = n;
    a.kstride = kstride;
    a.consts = consts;
    a.cov = cov;
    a.out_value = out_value;
    a.out_var = out_var;
    a.ld_out = ld_out;
    a.nsplit = (int)std::max<int64_t>(1, std::min<int64_t>({want, tiles, 65535}));
    const size_t smem = sizeof(double) * ((size_t)K * K + g.kmax + 1 + g.max_imm) +
                        sizeof(vsr_insn_t) * (g.max_insn + 1);
    cudaError_t e = dtype == VSR_F64 ? launch_predict<double>(K, a, smem, st) : launch_predict<float>(K, a, smem, st);
    if (e != cudaSuccess) return fail(h, VSR_ECUDA, "predict kernel launch failed: %s", cudaGetErrorString(e));
    h->launches += 1;
  }
  return VSR_OK;
}

int vsr_score(vsr_handle* h, const int32_t* prog_idx, const int32_t* const_row, int32_t n_pairs,
              const double* consts, int32_t kstride, int32_t dtype, double* out_mse, void* stream) {
  int rc = check_ready(h, dtype);
  if (rc) return rc;
  if (!prog_idx || n_pairs <= 0 || !out_mse || kstride < 0 || (!consts && kstride > 0))
    return fail(h, VSR_EINVAL, "bad score arguments");
  cudaStream_t st = (cudaStream_t)stream;
  VSR_CUDA(h, cudaSetDevice(h->device));
  int kmax = 0, max_insn = 0, max_imm = 0;
  unsigned var_mask = 0;
  std::vector<int32_t> all;
  for (int p = 0; p < n_pairs; ++p) {
    const int c = prog_idx[p];
    if (c < 0 || c >= h->n_programs) return fail(h, VSR_EINVAL, "pair %d: program %d out of range", p, c);
    if (h->h_k[c] > kstride) return fail(h, VSR_EINVAL, "pair %d: %d constants > kstride %d", p, h->h_k[c], kstride);
    if ((rc = check_vars(h, c, dtype))) return rc;
    var_mask |= h->h_varmask[c];
    kmax = std::max(kmax, h->h_k[c]);
    max_insn = std::max(max_insn, h->h_ninsn[c]);
    max_imm = std::max(max_imm, h->h_nimm[c]);
    all.push_back(c);
  }
  for (int p = 0; p < n_pairs; ++p) all.push_back(const_row ? const_row[p] : p);
  for (int p = 0; p < n_pairs; ++p) all.push_back(p);
  rc = stage_lists(h, all, st);
  if (rc) return rc;
  const int32_t* dl = (const int32_t*)h->d_lists.p;
  return run_eval_group(h, 0, dtype, dl, dl + n_pairs, dl + 2 * n_pairs, n_pairs, kmax, max_insn, max_imm,
                        consts, kstride, out_mse, nullptr, st, /*nan_to_num=*/1, var_mask);
}

int vsr_fit(vsr_handle* h, const int32_t* run_prog, const int32_t* run_slot, int32_t n_runs,
            const double* x0, int32_t kstride, const vsr_fit_opts* opts, double* out_consts,
            double* out_lastx, double* out_loss, double* out_final_mse, int32_t* out_info,
            void* stream) {
  if (!h || !opts) return VSR_EINVAL;
  int rc = check_ready(h, opts->eval_dtype);
  if (rc) return rc;
  rc = check_ready(h, opts->score_dtype);
  if (rc) return rc;
  if (!run_prog || !run_slot || n_runs <= 0 || !x0 || kstride < 1 || !out_consts || !out_lastx ||
      !out_loss || !out_final_mse || !out_info)
    return fail(h, VSR_EINVAL, "bad fit arguments");
  if (opts->grad_mode != VSR_GRAD_DUAL && opts->grad_mode != VSR_GRAD_FD)
    return fail(h, VSR_EINVAL, "bad grad_mode %d", opts->grad_mode);
  cudaStream_t st = (cudaStream_t)stream;
  VSR_CUDA(h, cudaSetDevice(h->device));

  // group runs: (tangent width, gradient mode).  k == 0 and FD runs use the width-0 kernel.
  std::vector<Group> groups;
  auto group_of = [&](int K, int mode) -> Group& {
    for (auto& g : groups)
      if (g.K == K && g.grad_mode == mode) return g;
    groups.emplace_back();
    groups.back().K = K;
    groups.back().grad_mode = mode;
    return groups.back();
  };
  for (int r = 0; r < n_runs; ++r) {
    const int c = run_prog[r];
    if (c < 0 || c >= h->n_programs) return fail(h, VSR_EINVAL, "run %d: program %d out of range", r, c);
    const int k = h->h_k[c];
    if (k > kstride) return fail(h, VSR_EINVAL, "run %d: %d constants > kstride %d", r, k, kstride);
    if (run_slot[r] < 0) return fail(h, VSR_EINVAL, "run %d: slot %d", r, run_slot[r]);
    if ((rc = check_vars(h, c, opts->eval_dtype)) || (rc = check_vars(h, c, opts->score_dtype))) return rc;
    int mode = opts->grad_mode, K = 0;
    if (k > 0 && mode == VSR_GRAD_DUAL) {
      K = pick_width(k);
      if (K < 0) {  // more constants than the widest dual kernel: forward differences
        K = 0;
        mode = VSR_GRAD_FD;
      }
    }
    if (k == 0) mode = VSR_GRAD_DUAL;
    Group& g = group_of(K, mode);
    g.prog.push_back(c);
    g.slot.push_back(run_slot[r]);
    g.kmax = std::max(g.kmax, k);
    g.max_insn = std::max(g.max_insn, h->h_ninsn[c]);
    g.max_imm = std::max(g.max_imm, h->h_nimm[c]);
    g.var_mask |= h->h_varmask[c];
  }
  // widest groups first: their runs have the highest iteration caps (200 k)
  std::stable_sort(groups.begin(), groups.end(), [](const Group& x, const Group& y) { return x.kmax > y.kmax; });
  // Queue order of a group.  Runs with more constants first (iteration cap 200 k); among those,
  // the runs of ONE program (the restarts of a candidate) are spread out: r-th restart of every
  // program before the (r+1)-th of any.  A hard candidate tends to drive most of its restarts to the
  // iteration cap, and the seats of a cluster take consecutive queue entries when the launch starts:
  // candidate-major order put four capped runs into one cluster (each then advances at a quarter of
  // the cluster's sweep rate) while other clusters ran dry.
  const bool by_candidate = h->queue_by_candidate;  // measurement hook (VSR_QUEUE_BY_CANDIDATE, read once in vsr_create): the old order
  for (auto& g : groups) {
    std::vector<int> order(g.prog.size()), rep(g.prog.size());
    {
      std::vector<int> seen(h->n_programs, 0);
      for (size_t i = 0; i < order.size(); ++i) rep[i] = seen[g.prog[i]]++;
    }
    for (size_t i = 0; i < order.size(); ++i) order[i] = (int)i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
      const int ka = h->h_k[g.prog[a]], kb = h->h_k[g.prog[b]];
      if (ka != kb) return ka > kb;
      if (!by_candidate && rep[a] != rep[b]) return rep[a] < rep[b];
      return h->h_ninsn[g.prog[a]] > h->h_ninsn[g.prog[b]];
    });
    std::vector<int32_t> p2(order.size()), s2(order.size());
    for (size_t i = 0; i < order.size(); ++i) {
      p2[i] = g.prog[order[i]];
      s2[i] = g.slot[order[i]];
    }
    g.prog.swap(p2);
    g.slot.swap(s2);
  }
  // lists: programs of all groups (launch order) | their slots ; then for the final score: prog | slot
  std::vector<int32_t> all;
  std::vector<int32_t> g_begin;  // first run of each group in the global lists
  for (auto& g : groups) {
    g_begin.push_back((int32_t)all.size());
    all.insert(all.end(), g.prog.begin(), g.prog.end());
  }
  g_begin.push_back((int32_t)all.size());
  const size_t n_listed = all.size();
  for (auto& g : groups) all.insert(all.end(), g.slot.begin(), g.slot.end());
  // what any launch may meet when it takes runs of a narrower group: the longest program, and the
  // union of the variables (a resident slice stages the columns of that union)
  int all_insn = 0;
  unsigned all_vars = 0;
  for (auto& g : groups) {
    all_insn = std::max(all_insn, g.max_insn);
    all_vars |= g.var_mask;
  }
  const size_t score_off = all.size();
  int s_kmax = 0, s_insn = 0, s_imm = 0;
  for (int r = 0; r < n_runs; ++r) all.push_back(run_prog[r]);
  for (int r = 0; r < n_runs; ++r) all.push_back(run_slot[r]);
  for (int r = 0; r < n_runs; ++r) {
    const int c = run_prog[r];
    s_kmax = std::max(s_kmax, h->h_k[c]);
    s_insn = std::max(s_insn, h->h_ninsn[c]);
    s_imm = std::max(s_imm, h->h_nimm[c]);
  }
  rc = stage_lists(h, all, st);
  if (rc) return rc;
  const int32_t* dl = (const int32_t*)h->d_lists.p;

  const PointSlot& ps = h->pts[opts->eval_dtype];
  const int elem = opts->eval_dtype == VSR_F64 ? 8 : 4;
  const bool tma_ok = ((uintptr_t)ps.X % 16 == 0) && ((uintptr_t)ps.y % 16 == 0) && ((ps.ldx * elem) % 16 == 0) &&
                      ((uintptr_t)ps.w % 16 == 0);
  cudaEvent_t ev_a = nullptr, ev_b = nullptr, ev_c = nullptr;
  if (h->profiling) {
    ev_a = take_event(h);
    ev_b = take_event(h);
    ev_c = take_event(h);
    VSR_CUDA(h, cudaEventRecord(ev_a, st));
  }
  // one run counter per group: the persistent clusters of a launch pull their runs from it
  VSR_CUDA(h, h->d_queue.reserve(groups.size() * sizeof(int32_t)));
  VSR_CUDA(h, cudaMemsetAsync(h->d_queue.p, 0, groups.size() * sizeof(int32_t), st));
  // hand-over boards: one per group, sized for the group's widest run
  std::vector<size_t> ho_off(groups.size() + 1, 0);
  std::vector<int> ho_slot_d(groups.size(), 0);
  if (h->handover) {
    for (size_t gi = 0; gi < groups.size(); ++gi) {
      ho_slot_d[gi] = (vsr::kHandoverHead + vsr::kFitStateDoubles + vsr::fit_workspace_doubles(std::max(1, groups[gi].kmax)) + 1) & ~1;
      ho_off[gi + 1] = ho_off[gi] + 16 + (size_t)vsr::kHandoverSlots * ho_slot_d[gi] * sizeof(double);
    }
    VSR_CUDA(h, h->d_handover.reserve(ho_off.back()));
    VSR_CUDA(h, cudaMemsetAsync(h->d_handover.p, 0, ho_off.back(), st));
  }
  // measurement hook: VSR_GEOMETRY="cluster:threads:seats[:optimiser warps]" overrides the launch geometry
  const int hook_cluster = h->hook[0], hook_threads = h->hook[1], hook_seats = h->hook[2], hook_reserved = h->hook[3];

  // groups run concurrently: group 0 on the caller's stream, the others on side streams
  // forked from / joined to it with events
  const size_t n_side = groups.size() > 1 ? groups.size() - 1 : 0;
  if (n_side > h->ev_join.size()) return fail(h, VSR_EINVAL, "%zu launch groups: too many", n_side + 1);
  if (n_side && !h->ev_fork) VSR_CUDA(h, cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
  if (n_side) VSR_CUDA(h, cudaEventRecord(h->ev_fork, st));
  for (size_t gi = 0; gi < groups.size(); ++gi) {
    Group& g = groups[gi];
    const int n = (int)g.prog.size();
    cudaStream_t gs = gi == 0 ? st : h->side_streams[(gi - 1) % h->side_streams.size()];
    if (gi > 0) VSR_CUDA(h, cudaStreamWaitEvent(gs, h->ev_fork, 0));
    vsr::FitArgs a;
    a.pt = table_of(h);
    a.pts = points_of(ps);
    a.run_prog = dl;
    a.run_slot = dl + n_listed;
    // queues: the group's own, then the next narrower groups of the same gradient mode, as long as
    // their kernels are at most `steal_span` widths apart (a k-run costs a K-wide kernel's sweep)
    a.n_queues = 0;
    for (size_t gj = gi; gj < groups.size() && a.n_queues < vsr::kMaxQueues; ++gj) {
      if (gj > gi && (groups[gj].grad_mode != g.grad_mode || groups[gj].K == 0 || g.K - groups[gj].K > h->steal_span ||
                      gj != gi + (size_t)a.n_queues))
        break;
      a.q_begin[a.n_queues] = g_begin[gj];
      a.q_end[a.n_queues] = g_begin[gj + 1];
      ++a.n_queues;
    }
    for (int q = a.n_queues; q < vsr::kMaxQueues; ++q) a.q_begin[q] = a.q_end[q] = 0;
    a.kstride = kstride;
    a.x0 = x0;
    a.out_consts = out_consts;
    a.out_lastx = out_lastx;
    a.out_loss = out_loss;
    a.out_info = out_info;
    a.O.gtol = opts->gtol;
    a.O.c1 = opts->c1;
    a.O.c2 = opts->c2;
    a.O.xrtol = opts->xrtol;
    a.O.fd_eps = opts->fd_eps;
    a.O.penalty = opts->penalty;
    a.O.loss_scale = opts->loss_scale;
    a.O.stop_time = opts->stop_time;
    a.O.maxiter_per_k = opts->maxiter_per_k;
    a.O.grad_mode = g.grad_mode;
    const int P = points_per_thread(g.K);
    int cap = opts->eval_dtype == VSR_F64 ? fit_threads_cap<double>(g.K) : fit_threads_cap<float>(g.K);
    if (hook_threads > 0) cap = std::min(cap, std::max(32, hook_threads & ~31));
    // experiment hook: VSR_LATENCY_K=k -- groups of width >= k use 16 half-width CTAs per cluster
    if (h->latency_k > 0 && g.K >= h->latency_k && hook_threads <= 0) cap = std::min(cap, 320);
    const int max_cluster = hook_cluster > 0 ? std::min(hook_cluster, kMaxCluster) : kMaxCluster;
    int n_cols = 0;
    for (int j = 0; j < VSR_MAX_VARS; ++j) a.col_of_var[j] = ((all_vars >> j) & 1u) ? n_cols++ : -1;
    g.max_insn = all_insn;
    // a weighted launch stages one column more (the weights) into a resident slice
    Geometry geo = choose_geometry(g.kmax == 0 ? 1 : ps.n, P, cap, opts->warps_per_run, g.kmax, g.K, g.max_insn,
                                   n_cols + (ps.w ? 1 : 0), elem, max_cluster,
                                   hook_seats > 0 ? hook_seats : kDefaultSeats, hook_reserved);
    if (g.kmax == 0) {  // runs without constants are only marked "not run": no points needed
      geo.resident = 0;
      geo.smem = vsr::fit_smem_bytes(geo.seats, g.kmax, g.K, geo.threads / 32, geo.cs, g.max_insn, -1, 0, elem);
    }
    a.phase_cycles = h->phase_cycles;
    a.hold_passes = h->hold_passes;
    a.handover = (h->handover && g.kmax > 0) ? (vsr::Handover*)((char*)h->d_handover.p + ho_off[gi]) : nullptr;
    a.handover_slot_d = ho_slot_d[gi];
    a.resident = geo.resident;
    a.tma_ok = tma_ok ? 1 : 0;
    a.slice_stride = geo.stride;
    a.seats = geo.seats;
    a.reserved = geo.reserved;
    {
      const vsr::SeatLayout L = vsr::fit_seat_layout(g.kmax, g.K, geo.cs, g.max_insn);
      a.seat_d = L.seat_d;
      a.off_cred = L.off_cred;
      a.off_ctrl = L.off_ctrl;
      a.off_insn = L.off_insn;
    }
    a.kmax = g.kmax;
    a.max_insn = g.max_insn;
    a.max_imm = g.max_imm;
    a.n_cols = n_cols;
    a.queue = (int32_t*)h->d_queue.p + gi;
    const int want_clusters = (n + geo.seats - 1) / geo.seats;
    cudaError_t e = opts->eval_dtype == VSR_F64
                        ? launch_fit<double>(g.K, a, geo.threads, geo.cs, geo.smem, want_clusters, gs, ps.w)
                        : launch_fit<float>(g.K, a, geo.threads, geo.cs, geo.smem, want_clusters, gs, ps.w);
    if (e != cudaSuccess)
      return fail(h, VSR_ECUDA, "fit kernel launch failed (K=%d threads=%d cluster=%d seats=%d smem=%zu): %s", g.K,
                  geo.threads, geo.cs, geo.seats, geo.smem, cudaGetErrorString(e));
    h->launches += 1;
    if (gi > 0) {
      VSR_CUDA(h, cudaEventRecord(h->ev_join[gi - 1], gs));
      VSR_CUDA(h, cudaStreamWaitEvent(st, h->ev_join[gi - 1], 0));
    }
  }
  if (h->profiling) VSR_CUDA(h, cudaEventRecord(ev_b, st));
  // per-restart score: plain MSE at the last evaluated point, in score_dtype (bfgs.py:120-132); with
  // weights on the score slot the weighted mean of w r^2
  rc = run_eval_group(h, 0, opts->score_dtype, dl + score_off, dl + score_off + n_runs,
                      dl + score_off + n_runs, n_runs, s_kmax, s_insn, s_imm, out_lastx, kstride,
                      out_final_mse, nullptr, st, 0, 0, h->pts[opts->score_dtype].w);
  if (h->profiling) {
    VSR_CUDA(h, cudaEventRecord(ev_c, st));
    h->spans.push_back({ev_a, ev_b, 0, (int)groups.size()});
    h->spans.push_back({ev_b, ev_c, 1, 2});
  }
  return rc;
}

int vsr_fit_host(vsr_handle* h, const int32_t* run_prog, const int32_t* run_slot, int32_t n_runs,
                 int32_t n_slots, const double* x0, int32_t kstride, const vsr_fit_opts* opts,
                 double* out_consts, double* out_lastx, double* out_loss, double* out_final_mse,
                 int32_t* out_info, void* stream) {
  if (!h) return VSR_EINVAL;
  if (n_slots <= 0 || kstride < 1 || !x0 || !out_consts || !out_lastx || !out_loss ||
      !out_final_mse || !out_info)
    return fail(h, VSR_EINVAL, "bad fit_host arguments");
  if (!run_slot || n_runs <= 0) return fail(h, VSR_EINVAL, "bad fit_host arguments");
  for (int r = 0; r < n_runs; ++r)  // the kernels write rows run_slot[r] of buffers sized n_slots
    if (run_slot[r] < 0 || run_slot[r] >= n_slots)
      return fail(h, VSR_EINVAL, "run %d: slot %d outside [0, %d)", r, run_slot[r], n_slots);
  cudaStream_t st = (cudaStream_t)stream;
  VSR_CUDA(h, cudaSetDevice(h->device));
  const size_t row = (size_t)kstride * sizeof(double);
  const size_t b_x = (size_t)n_slots * row;
  const size_t b_s = (size_t)n_slots * sizeof(double);
  const size_t b_i = (size_t)n_slots * 4 * sizeof(int32_t);
  VSR_CUDA(h, h->d_stage.reserve(3 * b_x + 2 * b_s + b_i));
  char* base = (char*)h->d_stage.p;
  double* d_x0 = (double*)base;
  double* d_c = (double*)(base + b_x);
  double* d_l = (double*)(base + 2 * b_x);
  double* d_loss = (double*)(base + 3 * b_x);
  double* d_mse = (double*)(base + 3 * b_x + b_s);
  int32_t* d_info = (int32_t*)(base + 3 * b_x + 2 * b_s);
  VSR_CUDA(h, cudaMemcpyAsync(d_x0, x0, b_x, cudaMemcpyHostToDevice, st));
  // slots no run touches come back as nan / NOT_RUN
  VSR_CUDA(h, cudaMemsetAsync(d_c, 0xff, 2 * b_x + 2 * b_s, st));
  VSR_CUDA(h, cudaMemsetAsync(d_info, 0xff, b_i, st));
  int rc = vsr_fit(h, run_prog, run_slot, n_runs, d_x0, kstride, opts, d_c, d_l, d_loss, d_mse,
                   d_info, stream);
  if (rc) return rc;
  VSR_CUDA(h, cudaMemcpyAsync(out_consts, d_c, b_x, cudaMemcpyDeviceToHost, st));
  VSR_CUDA(h, cudaMemcpyAsync(out_lastx, d_l, b_x, cudaMemcpyDeviceToHost, st));
  VSR_CUDA(h, cudaMemcpyAsync(out_loss, d_loss, b_s, cudaMemcpyDeviceToHost, st));
  VSR_CUDA(h, cudaMemcpyAsync(out_final_mse, d_mse, b_s, cudaMemcpyDeviceToHost, st));
  VSR_CUDA(h, cudaMemcpyAsync(out_info, d_info, b_i, cudaMemcpyDeviceToHost, st));
  VSR_CUDA(h, cudaStreamSynchronize(st));
  return VSR_OK;
}

}  // extern "C"
