// Batched box-constrained regulator QP on B200: Douglas-Rachford / ADMM over the shared
// condensed operator, one FP64 tensor-core GEMM per iteration with the whole update fused
// into its epilogue.
//
// Replaces, for a whole batch of samples at once, DenseQPRegulator.solve
// (/root/reference/lib/linearMPC.py:495-512: one cvxopt interior-point solve per sample) for the
// box path G = tE (:481):      min_u 1/2 u'Pu + q'u,  lb <= u <= ub,  q = tq x0.
//
// Iteration (state v, one vector per sample; z = clip(v) is the feasible iterate and
// y = rho (v - z) the multiplier estimate):
//     w  = 2 clip(v) - v
//     x  = (P + diag(rho))^-1 (rho . w - q) = Top w - c ,   c = Mtq x0           <- GEMM
//     v+ = v + alpha (x - clip(v))                                                <- epilogue
// Fixed points satisfy the KKT conditions exactly.  Every `check` iterations the feasible iterate
// is verified with the true Hessian, g = P z + q (one more GEMM, epilogue reduces
// ||z - clip(z - g)||_inf and the cost per sample); samples that pass leave the active row list.
#include "qp.cuh"
#include <cmath>
#include <mutex>
#include <vector>

namespace nnmpc {

thread_local char g_last_error[512] = "";
std::atomic<long long> g_launches{0};
std::atomic<long long> g_iterations{0};

// ---- live timing of the iteration GEMM (bench.py roofline) ------------------------------------
static std::mutex g_prof_mu;
static bool g_prof_on = false;
static std::vector<ProfSpan> g_prof_spans;   // recorded since the last reset
static std::vector<ProfSpan> g_prof_pool;    // events to reuse
constexpr int NNMPC_PROF_CHANNELS = 4;
static double g_prof_extra_flops[NNMPC_PROF_CHANNELS] = {};

void prof_add_flops(double flops, int chan) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (g_prof_on) g_prof_extra_flops[chan & (NNMPC_PROF_CHANNELS - 1)] += flops;
}

bool prof_begin(ProfSpan* sp, cudaStream_t st) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (!g_prof_on) return false;
  if (!g_prof_pool.empty()) {
    *sp = g_prof_pool.back();
    g_prof_pool.pop_back();
  } else if (cudaEventCreate(&sp->a) != cudaSuccess || cudaEventCreate(&sp->b) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  cudaEventRecord(sp->a, st);
  return true;
}
void prof_end(ProfSpan sp, cudaStream_t st, double flops, long long launches, int chan) {
  cudaEventRecord(sp.b, st);
  sp.flops = flops;
  sp.launches = launches;
  sp.chan = chan & (NNMPC_PROF_CHANNELS - 1);
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_spans.push_back(sp);
}

// ------------------------------------------------------------------------------------ small kernels
__global__ void k_init_lists(int* rows, int* counts, unsigned long long* iter_sum, int B) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) rows[i] = i;
  if (i == 0) {
    counts[0] = B;
    counts[1] = 0;
    counts[2] = 0;
    *iter_sum = 0ull;
  }
}

// w = 2 clip(v) - v for all B x n entries
__global__ void k_init_w(const double* __restrict__ V, double* __restrict__ W, const double* __restrict__ lb,
                         const double* __restrict__ ub, long long total, int n, int nu) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    long long r = i / n;
    int k = (int)(i - r * n) % nu;
    double v = V[i];
    W[i] = 2.0 * clipd(v, lb[r * nu + k], ub[r * nu + k]) - v;
  }
}

// one warp per active row: fold the per-slot partials in a fixed order, retire converged rows,
// append the rest to the next row list
__global__ void k_status(const int* __restrict__ rows_cur, const int* __restrict__ count_cur,
                         int* __restrict__ rows_next, int* __restrict__ count_next, int* __restrict__ flag_maxiter,
                         unsigned long long* __restrict__ iter_sum, const double* __restrict__ part_max,
                         const double* __restrict__ part_sum, int nslots, double tol, int it_total, int last,
                         QpOutputs out) {
  const int warps_per_block = blockDim.x >> 5;
  const int lane = threadIdx.x & 31;
  const int cnt = *count_cur;
  for (int lr = blockIdx.x * warps_per_block + (threadIdx.x >> 5); lr < cnt; lr += gridDim.x * warps_per_block) {
    double m = 0.0, s = 0.0;
    for (int k = lane; k < nslots; k += 32) {
      m = fmax(m, part_max[(long long)lr * nslots + k]);
      s += part_sum[(long long)lr * nslots + k];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
      s += __shfl_xor_sync(0xffffffffu, s, o);
    }
    if (lane == 0) {
      const int pr = rows_cur[lr];
      const bool conv = m <= tol;
      if (conv || last) {
        if (out.kkt) out.kkt[(long long)pr * out.stride] = m;
        if (out.cost) out.cost[(long long)pr * out.stride] = s;
        if (out.iters) out.iters[(long long)pr * out.stride] = it_total;
        atomicAdd(iter_sum, (unsigned long long)it_total);
        if (!conv) atomicExch(flag_maxiter, 1);
      } else {
        int idx = atomicAdd(count_next, 1);
        rows_next[idx] = pr;
      }
    }
  }
}

int qp_ensure_scratch(nnmpc_qp* h, long long B) {
  const long long n = h->n;
  const int nslots = row_slots_auto(B, h->n);
  if (B <= h->cap && nslots <= h->nslots_cap) return 0;
  long long cap = B > h->cap ? B : h->cap;
  int ns = nslots > h->nslots_cap ? nslots : h->nslots_cap;
  NNMPC_TRY(h->V.ensure(cap * n));
  NNMPC_TRY(h->W0.ensure(cap * n));
  NNMPC_TRY(h->W1.ensure(cap * n));
  NNMPC_TRY(h->C.ensure(cap * n));
  NNMPC_TRY(h->Ql.ensure(cap * n));
  NNMPC_TRY(h->part_max.ensure(cap * ns));
  NNMPC_TRY(h->part_sum.ensure(cap * ns));
  NNMPC_TRY(h->rows0.ensure(cap));
  NNMPC_TRY(h->rows1.ensure(cap));
  h->cap = cap;
  h->nslots_cap = ns;
  return 0;
}

int qp_solve_device(nnmpc_qp* h, int B, const double* x0, const double* lb, const double* ub, double* u,
                    double* v_state, int warm, QpOutputs out, double tol, int max_iter, cudaStream_t st,
                    long long* iter_sum_out) {
  if (B <= 0) return 0;
  if (h->ipm) return ipm_solve_device(h, B, x0, lb, ub, u, out, tol, max_iter, st, iter_sum_out);
  if (max_iter < 1) max_iter = 1;
  NNMPC_TRY(qp_ensure_scratch(h, B));
  const int n = h->n, nu = h->nu, nxa = h->nxa;
  double* V = v_state ? v_state : h->V.p;
  double* Wc = h->W0.p;
  double* Wn = h->W1.p;
  int* rows_c = h->rows0.p;
  int* rows_n = h->rows1.p;
  int* cnt_c = h->counts + 0;
  int* cnt_n = h->counts + 1;
  const int nslots = row_slots_auto(B, n);

  k_init_lists<<<(B + 255) / 256, 256, 0, st>>>(rows_c, h->counts, h->iter_sum, B);
  count_launch();

  // q-build: c = x0 Mtq', q = x0 tq' (and the unconstrained law v0 = x0 Kunc' on a cold start)
  GemmOperands g{};
  g.A = x0; g.lda = nxa; g.ldb = nxa; g.M = B; g.N = n; g.K = nxa; g.rows = nullptr; g.m_count = nullptr;
  g.Bt = h->Mtq;
  NNMPC_TRY(gemm_auto<EpiStore>(g, EpiStore::Params{h->C.p, n, nullptr, 0}, st));
  g.Bt = h->tq;
  NNMPC_TRY(gemm_auto<EpiStore>(g, EpiStore::Params{h->Ql.p, n, nullptr, 0}, st));
  if (!(warm && v_state)) {
    g.Bt = h->Kunc;
    NNMPC_TRY(gemm_auto<EpiStore>(g, EpiStore::Params{V, n, nullptr, 0}, st));
  }
  {
    long long total = (long long)B * n;
    int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
    k_init_w<<<blocks, 256, 0, st>>>(V, Wc, lb, ub, total, n, nu);
    count_launch();
  }

  int it = 0, active = B, chunk_idx = 0;
  while (active > 0) {
    int chunk = chunk_idx == 0 ? 1 : (chunk_idx == 1 ? 4 : (chunk_idx == 2 ? 5 : 10));
    if (it + chunk > max_iter) chunk = max_iter - it;
    ++chunk_idx;
    GemmOperands gi{};
    gi.lda = n; gi.Bt = h->Top; gi.ldb = n; gi.M = B; gi.N = n; gi.K = n; gi.rows = rows_c; gi.m_count = cnt_c;
    ProfSpan span;
    const bool prof = prof_begin(&span, st);
    for (int k = 0; k < chunk; ++k) {
      gi.A = Wc;
      EpiAdmm::Params ep{V, h->C.p, Wn, u, lb, ub, n, nu, h->alpha, k == chunk - 1 ? 1 : 0, nullptr, nullptr, 0};
      NNMPC_TRY(gemm_auto<EpiAdmm>(gi, ep, st));
      double* t = Wc; Wc = Wn; Wn = t;
    }
    if (prof) prof_end(span, st, 2.0 * n * (double)n * active * chunk, chunk);
    it += chunk;
    // verify with the true Hessian: g = P z + q
    GemmOperands gv = gi;
    gv.A = u; gv.Bt = h->P;
    EpiVerify::Params ev{u, h->Ql.p, lb, ub, h->part_max.p, h->part_sum.p, n, nu, nslots};
    NNMPC_TRY(gemm_auto<EpiVerify>(gv, ev, st));
    const int last = it >= max_iter ? 1 : 0;
    int sblocks = (active + 7) / 8 < 148 * 8 ? (active + 7) / 8 : 148 * 8;
    k_status<<<sblocks, 256, 0, st>>>(rows_c, cnt_c, rows_n, cnt_n, h->counts + 2, h->iter_sum, h->part_max.p,
                                      h->part_sum.p, nslots, tol, it, last, out);
    count_launch();
    // swap lists, clear the new "next" counter, fetch the active count
    { int* t = rows_c; rows_c = rows_n; rows_n = t; }
    { int* t = cnt_c; cnt_c = cnt_n; cnt_n = t; }
    NNMPC_CUDA(cudaMemsetAsync(cnt_n, 0, sizeof(int), st));
    NNMPC_CUDA(cudaMemcpyAsync(h->h_pinned, h->counts, 3 * sizeof(int), cudaMemcpyDeviceToHost, st));
    NNMPC_CUDA(cudaStreamSynchronize(st));
    active = h->h_pinned[cnt_c - h->counts];
    if (last) break;
  }
  NNMPC_CUDA(cudaMemcpyAsync(h->h_pinned + 4, h->iter_sum, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaStreamSynchronize(st));
  unsigned long long isum;
  memcpy(&isum, h->h_pinned + 4, sizeof(isum));
  g_iterations.fetch_add((long long)isum, std::memory_order_relaxed);
  if (iter_sum_out) *iter_sum_out = (long long)isum;
  return h->h_pinned[2] ? NNMPC_WARN_MAXITER : 0;
}

}  // namespace nnmpc

using namespace nnmpc;

extern "C" {

int nnmpc_version(void) { return 100; }
const char* nnmpc_last_error(void) { return g_last_error; }
long long nnmpc_launch_count(void) { return g_launches.load(); }
long long nnmpc_iteration_count(void) { return g_iterations.load(); }

int nnmpc_prof_enable(int on) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_on = on != 0;
  return 0;
}

// ms/flops/launches: arrays of nchan <= 4.  channel 0 = iteration passes, 1 = exact anchors and KKT checks of the
// mixed mode, 2 = FP64 tail iterations of the mixed mode (few live rows), 3 = the rest of a full engine loop
// (plant step, target selector, q-build, list kernels)
int nnmpc_prof_readn(int nchan, double* ms, double* flops, long long* launches, int reset) {
  if (nchan < 1 || nchan > NNMPC_PROF_CHANNELS) return set_error(NNMPC_ERR_BADARG, "nnmpc_prof_readn: 1..4 channels");
  std::lock_guard<std::mutex> lk(g_prof_mu);
  double t[NNMPC_PROF_CHANNELS] = {}, f[NNMPC_PROF_CHANNELS] = {};
  long long l[NNMPC_PROF_CHANNELS] = {};
  for (int c = 0; c < NNMPC_PROF_CHANNELS; ++c) f[c] = g_prof_extra_flops[c];
  for (const ProfSpan& sp : g_prof_spans) {
    float e = 0.f;
    if (cudaEventSynchronize(sp.b) != cudaSuccess || cudaEventElapsedTime(&e, sp.a, sp.b) != cudaSuccess)
      return set_error(NNMPC_ERR_CUDA, "nnmpc_prof_read: %s", cudaGetErrorString(cudaGetLastError()));
    const int c = sp.chan & (NNMPC_PROF_CHANNELS - 1);
    t[c] += e;
    f[c] += sp.flops;
    l[c] += sp.launches;
  }
  for (int c = 0; c < nchan; ++c) {
    if (ms) ms[c] = t[c];
    if (flops) flops[c] = f[c];
    if (launches) launches[c] = l[c];
  }
  if (reset) {
    for (const ProfSpan& sp : g_prof_spans) g_prof_pool.push_back(sp);
    g_prof_spans.clear();
    for (int c = 0; c < NNMPC_PROF_CHANNELS; ++c) g_prof_extra_flops[c] = 0.0;
  }
  return 0;
}

int nnmpc_prof_read2(double* ms, double* flops, long long* launches, int reset) {
  return nnmpc_prof_readn(2, ms, flops, launches, reset);
}

int nnmpc_prof_read(double* ms, double* flops, long long* launches, int reset) {
  double t[2], f[2];
  long long l[2];
  int rc = nnmpc_prof_read2(t, f, l, reset);
  if (rc < 0) return rc;
  if (ms) *ms = t[0];
  if (flops) *flops = f[0];
  if (launches) *launches = l[0];
  return 0;
}

int nnmpc_qp_create(nnmpc_qp_t** out, int n, int nxa, int nu, int N, const double* P_host, const double* tq_host,
                    const double* Top_host, const double* Mtq_host, const double* Kunc_host, double alpha,
                    int device) {
  if (!out || !P_host || !tq_host || !Top_host || !Mtq_host || !Kunc_host)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_qp_create: null argument");
  if (n <= 0 || nu <= 0 || N <= 0 || n != N * nu) return set_error(NNMPC_ERR_BADARG, "nnmpc_qp_create: n must equal N*nu");
  if ((n & 1) || (nxa & 1)) return set_error(NNMPC_ERR_BADARG, "nnmpc_qp_create: n and nxa must be even (pad with zeros)");
  if (!(alpha > 0.0 && alpha < 2.0)) return set_error(NNMPC_ERR_BADARG, "nnmpc_qp_create: alpha must be in (0,2)");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return set_error(NNMPC_ERR_CUDA, "nnmpc_qp_create: no CUDA device (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return set_error(NNMPC_ERR_BADARG, "nnmpc_qp_create: bad device %d", device);
  DeviceGuard dg(device);
  nnmpc_qp* h = new (std::nothrow) nnmpc_qp();
  if (!h) return set_error(NNMPC_ERR_NOMEM, "out of host memory");
  h->n = n; h->nxa = nxa; h->nu = nu; h->N = N; h->device = device; h->alpha = alpha;
  h->cap = 0; h->nslots_cap = 0;
  h->p_norm_inf = 0.0;
  h->top_max = 0.0;
  for (int r = 0; r < n; ++r) {
    double a = 0.0;
    for (int c = 0; c < n; ++c) {
      a += fabs(P_host[(size_t)r * n + c]);
      const double t = fabs(Top_host[(size_t)r * n + c]);
      if (t > h->top_max) h->top_max = t;
    }
    if (a > h->p_norm_inf) h->p_norm_inf = a;
  }
  h->P = h->Top = h->tq = h->Mtq = h->Kunc = nullptr;
  h->counts = nullptr; h->iter_sum = nullptr; h->h_pinned = nullptr;
  int rc = upload(&h->P, P_host, (size_t)n * n);
  if (rc == 0) rc = upload(&h->Top, Top_host, (size_t)n * n);
  if (rc == 0) rc = upload(&h->tq, tq_host, (size_t)n * nxa);
  if (rc == 0) rc = upload(&h->Mtq, Mtq_host, (size_t)n * nxa);
  if (rc == 0) rc = upload(&h->Kunc, Kunc_host, (size_t)n * nxa);
  if (rc == 0 && (cudaMalloc((void**)&h->counts, 4 * sizeof(int)) != cudaSuccess ||
                  cudaMalloc((void**)&h->iter_sum, sizeof(unsigned long long)) != cudaSuccess ||
                  cudaMallocHost((void**)&h->h_pinned, 8 * sizeof(int)) != cudaSuccess))
    rc = set_error(NNMPC_ERR_NOMEM, "nnmpc_qp_create: allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
  if (rc < 0) {          // a half-built handle is released, not leaked
    nnmpc_qp_destroy(h);
    return rc;
  }
  *out = h;
  return 0;
}

int nnmpc_qp_set_penalty(nnmpc_qp_t* h, const double* rho_host) {
  if (!h || !rho_host) return set_error(NNMPC_ERR_BADARG, "nnmpc_qp_set_penalty: null argument");
  if (h->ipm)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_qp_set_penalty: this handle solves by interior point (nnmpc_qp_create_ipm) "
                     "and has no ADMM penalty");
  DeviceGuard dg(h->device);
  double* tmp = new (std::nothrow) double[(size_t)h->n];
  if (!tmp) return set_error(NNMPC_ERR_NOMEM, "out of host memory");
  for (int i = 0; i < h->n; ++i) {
    if (!(rho_host[i] > 0.0) || !(rho_host[i] <= 1.7e308)) {
      delete[] tmp;
      return set_error(NNMPC_ERR_BADARG, "nnmpc_qp_set_penalty: rho[%d] must be positive and finite", i);
    }
    tmp[i] = 1.0 / rho_host[i];
  }
  int rc = 0;
  if (!h->rinv && cudaMalloc((void**)&h->rinv, (size_t)h->n * sizeof(double)) != cudaSuccess) {
    cudaGetLastError();
    h->rinv = nullptr;
    rc = set_error(NNMPC_ERR_NOMEM, "cudaMalloc failed for the penalty vector");
  }
  if (rc == 0 && cudaMemcpy(h->rinv, tmp, (size_t)h->n * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess)
    rc = set_error(NNMPC_ERR_CUDA, "nnmpc_qp_set_penalty: upload failed: %s", cudaGetErrorString(cudaGetLastError()));
  delete[] tmp;
  return rc;
}

int nnmpc_qp_destroy(nnmpc_qp_t* h) {
  if (!h) return 0;
  DeviceGuard dg(h->device);
  if (h->rinv) cudaFree(h->rinv);
  for (double* p : {h->P, h->Top, h->tq, h->Mtq, h->Kunc, h->iA, h->iB, h->iQ, h->iR, h->iM, h->iPf, h->iK, h->iAo, h->iQo, h->iMo})
    if (p) cudaFree(p);
  if (h->counts) cudaFree(h->counts);
  if (h->iter_sum) cudaFree(h->iter_sum);
  if (h->h_pinned) cudaFreeHost(h->h_pinned);
  h->V.release(); h->W0.release(); h->W1.release(); h->C.release(); h->Ql.release();
  h->part_max.release(); h->part_sum.release(); h->rows0.release(); h->rows1.release();
  h->hx0.release(); h->hlb.release(); h->hub.release(); h->hu.release(); h->hcost.release(); h->hkkt.release();
  h->hiters.release();
  h->lpop.release();
  h->ozP.release();
  h->ozTop.release();
  h->ipm_scr.release();
  delete h;
  return 0;
}

int nnmpc_qp_solve(nnmpc_qp_t* h, int B, const double* x0, const double* lb, const double* ub, double* u,
                   double* v_state, int warm, double* cost, double* kkt, int* iters, double tol, int max_iter,
                   void* stream) {
  if (B == 0 && h) return 0;
  if (!h || !x0 || !lb || !ub || !u) return set_error(NNMPC_ERR_BADARG, "nnmpc_qp_solve: null argument");
  if (B < 0) return set_error(NNMPC_ERR_BADARG, "nnmpc_qp_solve: negative batch");
  DeviceGuard dg(h->device);
  return qp_solve_device(h, B, x0, lb, ub, u, v_state, warm, QpOutputs{cost, kkt, iters, 1}, tol, max_iter,
                         (cudaStream_t)stream, nullptr);
}

int nnmpc_qp_solve_host(nnmpc_qp_t* h, int B, const double* x0, const double* lb, const double* ub, double* u,
                        double* cost, double* kkt, int* iters, double tol, int max_iter) {
  if (B == 0 && h) return 0;
  if (!h || !x0 || !lb || !ub || !u) return set_error(NNMPC_ERR_BADARG, "nnmpc_qp_solve_host: null argument");
  if (B <= 0) return B == 0 ? 0 : set_error(NNMPC_ERR_BADARG, "nnmpc_qp_solve_host: negative batch");
  DeviceGuard dg(h->device);
  const size_t b = (size_t)B;
  NNMPC_TRY(h->hx0.ensure(b * h->nxa));
  NNMPC_TRY(h->hlb.ensure(b * h->nu));
  NNMPC_TRY(h->hub.ensure(b * h->nu));
  NNMPC_TRY(h->hu.ensure(b * h->n));
  NNMPC_TRY(h->hcost.ensure(b));
  NNMPC_TRY(h->hkkt.ensure(b));
  NNMPC_TRY(h->hiters.ensure(b));
  cudaStream_t st = 0;
  NNMPC_CUDA(cudaMemcpyAsync(h->hx0.p, x0, b * h->nxa * 8, cudaMemcpyHostToDevice, st));
  NNMPC_CUDA(cudaMemcpyAsync(h->hlb.p, lb, b * h->nu * 8, cudaMemcpyHostToDevice, st));
  NNMPC_CUDA(cudaMemcpyAsync(h->hub.p, ub, b * h->nu * 8, cudaMemcpyHostToDevice, st));
  int rc = qp_solve_device(h, B, h->hx0.p, h->hlb.p, h->hub.p, h->hu.p, nullptr, 0,
                           QpOutputs{h->hcost.p, h->hkkt.p, h->hiters.p, 1}, tol, max_iter, st, nullptr);
  if (rc < 0) return rc;
  NNMPC_CUDA(cudaMemcpyAsync(u, h->hu.p, b * h->n * 8, cudaMemcpyDeviceToHost, st));
  if (cost) NNMPC_CUDA(cudaMemcpyAsync(cost, h->hcost.p, b * 8, cudaMemcpyDeviceToHost, st));
  if (kkt) NNMPC_CUDA(cudaMemcpyAsync(kkt, h->hkkt.p, b * 8, cudaMemcpyDeviceToHost, st));
  if (iters) NNMPC_CUDA(cudaMemcpyAsync(iters, h->hiters.p, b * 4, cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaStreamSynchronize(st));
  return rc;
}

int nnmpc_gemm_tn(int M, int N, int K, const double* A, long long lda, const double* Bt, long long ldb, double* C,
                  long long ldc, const int* rows, void* stream) {
  if (!A || !Bt || !C) return set_error(NNMPC_ERR_BADARG, "nnmpc_gemm_tn: null argument");
  if ((lda & 1) || (ldb & 1)) return set_error(NNMPC_ERR_BADARG, "nnmpc_gemm_tn: lda/ldb must be even");
  GemmOperands g{A, lda, Bt, ldb, M, N, K, rows, nullptr};
  return gemm_auto<EpiStore>(g, EpiStore::Params{C, ldc, nullptr, 0}, (cudaStream_t)stream);
}

}  // extern "C"
