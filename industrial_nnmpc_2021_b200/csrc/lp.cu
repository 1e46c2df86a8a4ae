// Host-side glue of the tcgen05 split-operator GEMM: fp16 operator split of a regulator handle,
// tensor maps, and the self-test entry point.
#include "lp_iter.cuh"
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace nnmpc {

// Which tcgen05 kernel serves the TWO-term passes (small QPs, NNMPC_T2_EVERY=0): the one-CTA kernel with 128 x 128 tiles
// unless NNMPC_LP_KERNEL=pair selects the CTA-pair kernel (cta_group::2, 256 x 256 tiles) or NNMPC_LP_TILE=m256 the
// 256 x 128 tiles.  Measured on B200: both halve the operator bytes pulled from L2 per flop and both are SLOWER (pair:
// 332 vs 372 TFLOP/s algorithmic, round 1ab/1ae; 256-row tiles: 343 vs 367, round 2c) - the two-term pass is bound by
// board power and its FP64 epilogue, not by L2->SM operand traffic (profiles/r02n_pass_energy_diagnosis.md).
static int lp_tile_m256() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("NNMPC_LP_TILE");
    v = (e && strcmp(e, "m256") == 0) ? 1 : 0;
  }
  return v;
}

static bool lp_use_pair() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("NNMPC_LP_KERNEL");
    v = (e && strcmp(e, "pair") == 0) ? 1 : 0;
  }
  return v == 1;
}

int device_sm_count(int device) {
  static int cache[64] = {};
  if (cache[device & 63] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || v <= 0) v = 148;
    cache[device & 63] = v;
  }
  return cache[device & 63];
}

// 0 = 128 x 128 tiles, 1 = 256 x 128 tiles for the ONE-term passes of the deferred-second-term form (NNMPC_LP1_TILE=m256):
// with one product per staged operand pair the L2->SM bytes per flop double, which the 256-row tile halves again.
static int lp1_tile_m256() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("NNMPC_LP1_TILE");
    v = (e && strcmp(e, "m256") == 0) ? 1 : 0;
  }
  return v;
}

int lp_state_ensure(LpState* s, long long B, int n, cudaStream_t st) {
  if (B <= s->cap && n == s->n && (!s->defer2 || s->S[0].p)) return 0;
  const long long cap = B > s->cap ? B : s->cap;
  s->n = n;
  s->ldd = ((long long)n + 63) / 64 * 64;
  NNMPC_TRY(s->X.ensure((size_t)cap * n));
  NNMPC_TRY(s->E.ensure((size_t)cap * n));
  NNMPC_TRY(s->Wl.ensure((size_t)cap * n));
  NNMPC_TRY(s->sc_in.ensure((size_t)cap));
  NNMPC_TRY(s->sc_out.ensure((size_t)cap));
  // rows and columns padded to whole TMA boxes (zeros), so no tile ever reaches outside the tensor
  const long long cap_pad = (cap + 2 * lp::BM - 1) / (2 * lp::BM) * (2 * lp::BM);
  for (int b = 0; b < 2; ++b) {
    NNMPC_TRY(s->D[b].ensure((size_t)cap_pad * s->ldd));
    NNMPC_CUDA(cudaMemsetAsync(s->D[b].p, 0, (size_t)cap_pad * s->ldd * sizeof(__half), st));   // ordered before the first writer on st
    if (!lp::make_tmap_f16(&s->tmD[b], s->D[b].p, cap_pad, s->ldd, s->ldd, lp::BM) ||
        !lp::make_tmap_f16(&s->tmD256[b], s->D[b].p, cap_pad, s->ldd, s->ldd, 2 * lp::BM))
      return set_error(NNMPC_ERR_CUDA, "cuTensorMapEncodeTiled failed for the increment buffers");
    if (s->defer2) {
      NNMPC_TRY(s->S[b].ensure((size_t)cap_pad * s->ldd));
      NNMPC_CUDA(cudaMemsetAsync(s->S[b].p, 0, (size_t)cap_pad * s->ldd * sizeof(__half), st));
      if (!lp::make_tmap_f16(&s->tmS[b], s->S[b].p, cap_pad, s->ldd, s->ldd, lp::BM) ||
          !lp::make_tmap_f16(&s->tmS256[b], s->S[b].p, cap_pad, s->ldd, s->ldd, 2 * lp::BM))
        return set_error(NNMPC_ERR_CUDA, "cuTensorMapEncodeTiled failed for the pending-sum buffers");
    }
  }
  if (s->defer2) {
    NNMPC_TRY(s->sS.ensure((size_t)cap));
    NNMPC_CUDA(cudaMemsetAsync(s->sS.p, 0, (size_t)cap * sizeof(double), st));
  }
  s->cap = cap;
  s->cur = 0;
  return 0;
}

int lp_anchor_prep(const int* rows, const int* count, int max_rows, const double* V, double* W, LpState* s,
                   const double* lb, const double* ub, int nu, cudaStream_t st) {
  if (max_rows <= 0) return 0;
  k_anchor_prep<<<row_grid(max_rows), 256, 0, st>>>(rows, count, V, W, s->E.p, lb, ub, s->n, nu);
  count_launch();
  NNMPC_CUDA(cudaGetLastError());
  return 0;
}

int lp_anchor_gemm(const int* rows, const int* count, int max_rows, const double* W, const double* Top, const double* C,
                   double* X, int n, cudaStream_t st) {
  if (max_rows <= 0) return 0;
  GemmOperands g{};
  g.A = W; g.lda = n; g.Bt = Top; g.ldb = n; g.M = max_rows; g.N = n; g.K = n; g.rows = rows; g.m_count = count;
  return gemm_by_count<EpiAnchor>(g, EpiAnchor::Params{X, C, n}, st);
}

int lp_dr_first(const int* rows, const int* count, int max_rows, LpState* s, double* V, double* W, const double* lb,
                const double* ub, int* state, int* it, int iter_state, int nu, double alpha, const int* pos_r,
                cudaStream_t st, unsigned char* need2) {
  if (max_rows <= 0) return 0;
  k_dr_first<<<row_grid(max_rows), 256, 0, st>>>(rows, count, s->X.p, V, W, s->E.p, s->D[s->cur].p, s->ldd, lb, ub, s->sc_in.p,
                                       s->sc_out.p, state, it, iter_state, s->n, nu, alpha, pos_r, need2,
                                       s->defer2 ? s->S[s->cur].p : nullptr, s->defer2 ? s->sS.p : nullptr);
  count_launch();
  NNMPC_CUDA(cudaGetLastError());
  return 0;
}

int lp_reanchor(const int* rows, const int* count, int max_rows, const int* state, int emit_state, const double* Z,
                const double* rinv, LpState* s, cudaStream_t st) {
  if (max_rows <= 0) return 0;
  k_reanchor<<<row_grid(max_rows), 256, 0, st>>>(rows, count, state, emit_state, Z, s->Wl.p, rinv, s->X.p, s->n);
  count_launch();
  NNMPC_CUDA(cudaGetLastError());
  return 0;
}

int lp_emit(const int* rows, const int* count, int max_rows, int* state, int emit_state, int iter_state, LpState* s,
            const double* V, const double* lb, const double* ub, const double* dtrig, int nu, double alpha,
            const int* pos_r, cudaStream_t st, unsigned char* need2) {
  if (max_rows <= 0) return 0;
  k_lp_emit<<<row_grid(max_rows), 256, 0, st>>>(rows, count, state, emit_state, iter_state, V, s->Wl.p, s->E.p, s->D[s->cur].p,
                                      s->ldd, lb, ub, s->sc_in.p, s->sc_out.p, dtrig, s->n, nu, alpha, pos_r, need2,
                                      s->defer2 ? s->S[s->cur].p : nullptr, s->defer2 ? s->sS.p : nullptr);
  count_launch();
  NNMPC_CUDA(cudaGetLastError());
  return 0;
}

int lp_iterate(const LpOperator* op, LpState* s, int B, const int* list_r, const int* len_r, const int* pos_w, double* V,
               const double* lb, const double* ub, const int* state, int iter_state, unsigned long long* dres, int nu,
               double alpha, int device, cudaStream_t st, const unsigned char* need2, unsigned long long* tile_stat,
               int s_mode, int kernel) {
  if (B <= 0) return 0;
  if (s_mode && !s->defer2) return set_error(NNMPC_ERR_BADARG, "lp_iterate: pending-sum buffers were not allocated");
  if (kernel < -1 || kernel > (s_mode ? 1 : 2)) return set_error(NNMPC_ERR_BADARG, "lp_iterate: no kernel %d for s_mode %d", kernel, s_mode);
  const int k2 = kernel >= 0 ? kernel : (lp_use_pair() ? 2 : lp_tile_m256());
  const int k1 = kernel >= 0 ? kernel : lp1_tile_m256();
  EpiDelta::Params ep{};
  ep.s_mode = s_mode;
  if (s_mode) { ep.Sc = s->S[s->cur].p; ep.Sn = s->S[s->cur ^ 1].p; ep.sS = s->sS.p; }
  ep.X = s->X.p; ep.V = V; ep.E = s->E.p; ep.Dn = s->D[s->cur ^ 1].p; ep.ldd = s->ldd; ep.lb = lb; ep.ub = ub;
  ep.state = state; ep.iter_state = iter_state; ep.list_r = list_r; ep.pos_w = pos_w; ep.sc_in = s->sc_in.p; ep.sc_out = s->sc_out.p; ep.dres = dres;
  ep.n = s->n; ep.nu = nu; ep.alpha = alpha; ep.inv_sT = 1.0 / op->scale;
  // column-tile groups of at most ~24 MB of operator (both fp16 terms) per group
  const int bn_tile = k2 == 2 ? lp::BN2 : LpTileN128::BN;
  const double tile_mb = 2.0 * bn_tile * (double)op->ldh * 2.0 / 1048576.0;
  int group_cols = (int)(24.0 / tile_mb);
  if (group_cols < 1) group_cols = 1;
  lp::LpShape g{B, s->n, s->n, len_r, group_cols, need2, tile_stat, 0, 0};
  if (s_mode) {      // one-term pass (the kernel never touches the second operator map)
    g.need2 = nullptr;
    g.group_cols = 2 * group_cols;        // one term: the same bytes of operator cover twice the column tiles
    cudaError_t e1 = k1 == 1
                         ? lp::launch_lp_gemm<LpTile1M256, EpiDelta>(s->tmD256[s->cur], op->tm1, op->tm1, g, ep, device_sm_count(device), st)
                         : lp::launch_lp_gemm<LpTile1N128, EpiDelta>(s->tmD[s->cur], op->tm1, op->tm1, g, ep, device_sm_count(device), st);
    count_launch();
    if (e1 != cudaSuccess) return set_error(NNMPC_ERR_CUDA, "lp_gemm launch failed: %s", cudaGetErrorString(e1));
    s->cur ^= 1;
    return 0;
  }
  cudaError_t e = k2 == 2
                      ? lp::launch_lp_gemm_pair<EpiDelta>(s->tmD[s->cur], op->tm1, op->tm2, g, ep, device_sm_count(device), st)
                  : k2 == 1
                      ? lp::launch_lp_gemm<LpTileM256, EpiDelta>(s->tmD256[s->cur], op->tm1, op->tm2, g, ep, device_sm_count(device), st)
                      : lp::launch_lp_gemm<LpTileN128, EpiDelta>(s->tmD[s->cur], op->tm1, op->tm2, g, ep, device_sm_count(device), st);
  count_launch();
  if (e != cudaSuccess) return set_error(NNMPC_ERR_CUDA, "lp_gemm launch failed: %s", cudaGetErrorString(e));
  s->cur ^= 1;
  return 0;
}

int lp_correct(const LpOperator* op, LpState* s, int B, const int* list_r, const int* len_r, const int* state,
               int iter_state, int device, cudaStream_t st, unsigned long long* tile_stat, int kernel) {
  if (B <= 0) return 0;
  if (!s->defer2) return set_error(NNMPC_ERR_BADARG, "lp_correct: pending-sum buffers were not allocated");
  if (kernel < -1 || kernel > 1) return set_error(NNMPC_ERR_BADARG, "lp_correct: no kernel %d", kernel);
  EpiAddX::Params ep{s->X.p, state, iter_state, list_r, s->sS.p, s->n, 1.0 / op->scale};
  const double tile_mb = LpTile1N128::BN * (double)op->ldh * 2.0 / 1048576.0;
  int group_cols = (int)(24.0 / tile_mb);
  if (group_cols < 1) group_cols = 1;
  lp::LpShape g{B, s->n, s->n, len_r, group_cols, nullptr, tile_stat, 0, 0};
  cudaError_t e = (kernel >= 0 ? kernel : lp1_tile_m256()) == 1
                      ? lp::launch_lp_gemm<LpTile1M256, EpiAddX>(s->tmS256[s->cur], op->tm2, op->tm2, g, ep, device_sm_count(device), st)
                      : lp::launch_lp_gemm<LpTile1N128, EpiAddX>(s->tmS[s->cur], op->tm2, op->tm2, g, ep, device_sm_count(device), st);
  count_launch();
  if (e != cudaSuccess) return set_error(NNMPC_ERR_CUDA, "lp_gemm (second-term delivery) launch failed: %s", cudaGetErrorString(e));
  return 0;
}

// T (n x n FP64 on the device, max |T| = tmax) -> two fp16 matrices with leading dimension ldh and their
// tensor maps (boxes of BN rows).  The scale is the power of two that puts max |s T| in [512, 1024).
int lp_split_operator(const double* T_dev, int n, double tmax, LpOperator* op, cudaStream_t st) {
  op->n = n;
  op->ldh = ((long long)n + 63) / 64 * 64;
  int ex = 0;
  frexp(tmax > 0.0 ? tmax : 1.0, &ex);
  op->scale = ldexp(1.0, 10 - ex);
  const long long rows_pad = ((long long)n + lp::BN2 - 1) / lp::BN2 * lp::BN2;
  NNMPC_TRY(op->T1.ensure((size_t)rows_pad * op->ldh));
  NNMPC_TRY(op->T2.ensure((size_t)rows_pad * op->ldh));
  NNMPC_CUDA(cudaMemsetAsync(op->T1.p, 0, (size_t)rows_pad * op->ldh * sizeof(__half), st));
  NNMPC_CUDA(cudaMemsetAsync(op->T2.p, 0, (size_t)rows_pad * op->ldh * sizeof(__half), st));
  k_split_f16<<<148 * 8, 256, 0, st>>>(T_dev, n, op->ldh, op->scale, op->T1.p, op->T2.p);
  count_launch();
  NNMPC_CUDA(cudaGetLastError());
  if (!lp::make_tmap_f16(&op->tm1, op->T1.p, rows_pad, op->ldh, op->ldh, LpTileN128::BN) ||
      !lp::make_tmap_f16(&op->tm2, op->T2.p, rows_pad, op->ldh, op->ldh, LpTileN128::BN))
    return set_error(NNMPC_ERR_CUDA, "cuTensorMapEncodeTiled failed for the fp16 operator split");
  op->ready = true;
  return 0;
}

__global__ void k_to_half(const double* __restrict__ A, long long rows, int cols, long long ld, __half* __restrict__ H) {
  const long long total = rows * ld;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const long long r = i / ld;
    const int c = (int)(i - r * ld);
    H[i] = __double2half(c < cols ? A[r * cols + c] : 0.0);
  }
}

enum { LP_SPLIT, LP_ANCHOR_PREP, LP_DR_FIRST, LP_REANCHOR, LP_EMIT, LP_ITERATE, LP_CORRECT };

static int copy_rows_f16(void* dst, size_t dpitch, const void* src, size_t spitch, int n, int B, cudaStream_t st) {
  if (!dst || !src) return 0;
  NNMPC_CUDA(cudaMemcpy2DAsync(dst, dpitch, src, spitch, (size_t)n * sizeof(__half), (size_t)B, cudaMemcpyDeviceToDevice, st));
  return 0;
}
template <class T>
static int copy_n(T* dst, const T* src, size_t count, cudaStream_t st) {
  if (!dst || !src) return 0;
  NNMPC_CUDA(cudaMemcpyAsync(dst, src, count * sizeof(T), cudaMemcpyDeviceToDevice, st));
  return 0;
}

static int lp_step_run(int op, int kernel, int s_mode, double alpha, int n, int nu, int B, const double* Top,
                       double top_max, const int* rows, const int* count, const int* list_r, const int* len_r,
                       const int* pos_w, const int* pos_r, int* state, int iter_state, int emit_state,
                       unsigned char* need2, double* X, double* V, double* W, float* E, double* sc_in, double* sc_out,
                       double* sS, unsigned long long* dres, int* it, const double* dtrig, const double* rinv,
                       const double* Z, const double* lb, const double* ub, const __half* D_in, const __half* S_in,
                       __half* D_out, __half* S_out, unsigned long long* tile_stat, LpState& ls, LpOperator& lo,
                       cudaStream_t st) {
  int dev = 0;
  NNMPC_CUDA(cudaGetDevice(&dev));
  if (op == LP_SPLIT || op == LP_ITERATE || op == LP_CORRECT) NNMPC_TRY(lp_split_operator(Top, n, top_max, &lo, st));
  if (op == LP_SPLIT) {
    NNMPC_TRY(copy_rows_f16(D_out, lo.ldh * sizeof(__half), lo.T1.p, lo.ldh * sizeof(__half), (int)lo.ldh, n, st));
    NNMPC_TRY(copy_rows_f16(S_out, lo.ldh * sizeof(__half), lo.T2.p, lo.ldh * sizeof(__half), (int)lo.ldh, n, st));
    NNMPC_CUDA(cudaMemcpyAsync(sc_out, &lo.scale, sizeof(double), cudaMemcpyHostToDevice, st));
    return 0;
  }
  ls.defer2 = s_mode != 0 || op == LP_CORRECT;
  NNMPC_TRY(lp_state_ensure(&ls, B, n, st));
  const size_t bn = (size_t)B * n, dp = (size_t)ls.ldd * sizeof(__half), sp = (size_t)n * sizeof(__half);
  const bool wl = op == LP_REANCHOR || op == LP_EMIT;     // W is the state's Wl (else the caller's own buffer)
  NNMPC_TRY(copy_n(ls.X.p, X, bn, st));
  NNMPC_TRY(copy_n(ls.E.p, E, bn, st));
  if (wl) NNMPC_TRY(copy_n(ls.Wl.p, W, bn, st));
  NNMPC_TRY(copy_n(ls.sc_in.p, sc_in, (size_t)B, st));
  NNMPC_TRY(copy_n(ls.sc_out.p, sc_out, (size_t)B, st));
  if (ls.defer2) NNMPC_TRY(copy_n(ls.sS.p, sS, (size_t)B, st));
  const int wr = op == LP_ITERATE ? 1 : 0;                 // buffer the op writes (it reads buffer 0)
  if (op == LP_ITERATE || op == LP_CORRECT) {
    NNMPC_TRY(copy_rows_f16(ls.D[0].p, dp, D_in, sp, n, B, st));
    if (ls.defer2) NNMPC_TRY(copy_rows_f16(ls.S[0].p, dp, S_in, sp, n, B, st));
  }
  NNMPC_TRY(copy_rows_f16(ls.D[wr].p, dp, D_out, sp, n, B, st));
  if (ls.defer2) NNMPC_TRY(copy_rows_f16(ls.S[wr].p, dp, S_out, sp, n, B, st));
  ls.cur = 0;
  switch (op) {
    case LP_ANCHOR_PREP: NNMPC_TRY(lp_anchor_prep(rows, count, B, V, W, &ls, lb, ub, nu, st)); break;
    case LP_DR_FIRST:
      NNMPC_TRY(lp_dr_first(rows, count, B, &ls, V, W, lb, ub, state, it, iter_state, nu, alpha, pos_r, st, need2));
      break;
    case LP_REANCHOR: NNMPC_TRY(lp_reanchor(rows, count, B, state, emit_state, Z, rinv, &ls, st)); break;
    case LP_EMIT:
      NNMPC_TRY(lp_emit(rows, count, B, state, emit_state, iter_state, &ls, V, lb, ub, dtrig, nu, alpha, pos_r, st, need2));
      break;
    case LP_ITERATE:
      NNMPC_TRY(lp_iterate(&lo, &ls, B, list_r, len_r, pos_w, V, lb, ub, state, iter_state, dres, nu, alpha, dev, st,
                           need2, tile_stat, s_mode, kernel));
      break;
    default: NNMPC_TRY(lp_correct(&lo, &ls, B, list_r, len_r, state, iter_state, dev, st, tile_stat, kernel)); break;
  }
  NNMPC_TRY(copy_n(X, (const double*)ls.X.p, bn, st));
  NNMPC_TRY(copy_n(E, (const float*)ls.E.p, bn, st));
  if (wl) NNMPC_TRY(copy_n(W, (const double*)ls.Wl.p, bn, st));
  NNMPC_TRY(copy_n(sc_in, (const double*)ls.sc_in.p, (size_t)B, st));
  NNMPC_TRY(copy_n(sc_out, (const double*)ls.sc_out.p, (size_t)B, st));
  if (ls.defer2) NNMPC_TRY(copy_n(sS, (const double*)ls.sS.p, (size_t)B, st));
  NNMPC_TRY(copy_rows_f16(D_out, sp, ls.D[wr].p, dp, n, B, st));
  if (ls.defer2) NNMPC_TRY(copy_rows_f16(S_out, sp, ls.S[wr].p, dp, n, B, st));
  return 0;
}

}  // namespace nnmpc

using namespace nnmpc;

extern "C" {

// Self test of the tcgen05 path:  C[M x N] = fp16(A)[M x K] * (T1 + T2)[N x K]^T / s  with (T1, T2, s) the
// two-term fp16 split of Bt.  A, Bt, C are FP64 device matrices (row-major, dense).
int nnmpc_lp_gemm_test(int M, int N, int K, const double* A, const double* Bt, double bt_max, double* C, int pair,
                       void* stream) {
  if (!A || !Bt || !C || M <= 0 || N <= 0 || K <= 0) return set_error(NNMPC_ERR_BADARG, "nnmpc_lp_gemm_test: bad argument");
  if (N != K) return set_error(NNMPC_ERR_BADARG, "nnmpc_lp_gemm_test: the operator must be square (N == K)");
  cudaStream_t st = (cudaStream_t)stream;
  int dev = 0;
  NNMPC_CUDA(cudaGetDevice(&dev));
  LpOperator op;
  int rc = lp_split_operator(Bt, N, bt_max, &op, st);
  DevBuf<__half> Ah;
  const long long m_pad = ((long long)M + 2 * lp::BM - 1) / (2 * lp::BM) * (2 * lp::BM);
  if (rc == 0) rc = Ah.ensure((size_t)m_pad * op.ldh);
  if (rc == 0) {
    cudaMemsetAsync(Ah.p, 0, (size_t)m_pad * op.ldh * sizeof(__half), st);
    k_to_half<<<148 * 4, 256, 0, st>>>(A, M, K, op.ldh, Ah.p);
    count_launch();
    CUtensorMap tmA;
    if (!lp::make_tmap_f16(&tmA, Ah.p, m_pad, op.ldh, op.ldh, pair == 2 ? 2 * lp::BM : lp::BM)) {
      rc = set_error(NNMPC_ERR_CUDA, "cuTensorMapEncodeTiled failed");
    } else {
      lp::LpShape g{M, N, K, nullptr, 2, nullptr, nullptr, 0, 0};
      const EpiLpStore::Params ep{C, N, 1.0 / op.scale};
      cudaError_t e = pair == 1 ? lp::launch_lp_gemm_pair<EpiLpStore>(tmA, op.tm1, op.tm2, g, ep, device_sm_count(dev), st)
                    : pair == 2 ? lp::launch_lp_gemm<LpTileM256, EpiLpStore>(tmA, op.tm1, op.tm2, g, ep, device_sm_count(dev), st)
                                : lp::launch_lp_gemm<LpTileN128, EpiLpStore>(tmA, op.tm1, op.tm2, g, ep, device_sm_count(dev), st);
      count_launch();
      if (e == cudaSuccess) e = cudaStreamSynchronize(st);
      if (e != cudaSuccess) rc = set_error(NNMPC_ERR_CUDA, "lp_gemm launch failed: %s", cudaGetErrorString(e));
    }
  }
  cudaStreamSynchronize(st);
  Ah.release();
  op.T1.release();
  op.T2.release();
  return rc;
}

// Self test of the mixed-precision iteration as the engine calls it (include/nnmpc.h).  The caller's state is copied
// into an LpState / LpOperator sized for B rows (padded, TMA-mapped, padding zero); the operand buffer an op writes is
// pre-loaded from D_out / S_out, so positions it must not write come back as the caller left them.
int nnmpc_lp_step_test(int op, int kernel, int s_mode, double alpha, int n, int nu, int B, const double* Top,
                       double top_max, const int* rows, const int* count, const int* list_r, const int* len_r,
                       const int* pos_w, const int* pos_r, int* state, int iter_state, int emit_state,
                       unsigned char* need2, double* X, double* V, double* W, float* E, double* sc_in, double* sc_out,
                       double* sS, unsigned long long* dres, int* it, const double* dtrig, const double* rinv,
                       const double* Z, const double* lb, const double* ub, const unsigned short* D_in,
                       const unsigned short* S_in, unsigned short* D_out, unsigned short* S_out,
                       unsigned long long* tile_stat, void* stream) {
  if (op < LP_SPLIT || op > LP_CORRECT || n <= 0 || (n & 1) || nu <= 0 || B <= 0 || s_mode < 0 || s_mode > 2 ||
      kernel < -1 || kernel > 2)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_lp_step_test: bad op, kernel, s_mode or shape (n must be even and > 0, nu > 0)");
  if ((s_mode != 0 || op == LP_CORRECT) && kernel == 2)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_lp_step_test: the CTA-pair kernel has no one-term form");
  const bool listed = op != LP_SPLIT && op != LP_ITERATE && op != LP_CORRECT;
  const bool defer = s_mode != 0 && (op == LP_DR_FIRST || op == LP_EMIT || op == LP_ITERATE);
  bool ok = true;
  switch (op) {
    case LP_SPLIT: ok = Top && D_out && S_out && sc_out; break;
    case LP_ANCHOR_PREP: ok = V && W && E && lb && ub; break;
    case LP_DR_FIRST: ok = X && V && W && E && lb && ub && sc_in && sc_out && state && it && D_out; break;
    case LP_REANCHOR: ok = state && Z && W && rinv && X; break;
    case LP_EMIT: ok = state && V && W && E && D_out && lb && ub && sc_in && sc_out && dtrig; break;
    case LP_ITERATE: ok = Top && len_r && X && V && E && lb && ub && state && dres && sc_in && sc_out && D_in && D_out &&
                          (s_mode != 1 || S_in); break;
    default: ok = Top && len_r && state && X && S_in && sS; break;
  }
  if (!ok || (listed && (!rows || !count)) || (defer && (!S_out || !sS)))
    return set_error(NNMPC_ERR_BADARG, "nnmpc_lp_step_test: a buffer the op needs is missing");
  cudaStream_t st = (cudaStream_t)stream;
  LpState ls;
  LpOperator lo;
  int rc = lp_step_run(op, kernel, s_mode, alpha, n, nu, B, Top, top_max, rows, count, list_r, len_r, pos_w, pos_r,
                       state, iter_state, emit_state, need2, X, V, W, E, sc_in, sc_out, sS, dres, it, dtrig, rinv, Z,
                       lb, ub, reinterpret_cast<const __half*>(D_in), reinterpret_cast<const __half*>(S_in),
                       reinterpret_cast<__half*>(D_out), reinterpret_cast<__half*>(S_out), tile_stat, ls, lo, st);
  if (rc == 0 && cudaStreamSynchronize(st) != cudaSuccess)
    rc = set_error(NNMPC_ERR_CUDA, "nnmpc_lp_step_test: %s", cudaGetErrorString(cudaGetLastError()));
  cudaStreamSynchronize(st);
  ls.release();
  lo.release();
  return rc;
}

// Probe (tools/probes/lp_pass_split.py, not on the product path): what the tensor-core pass costs with and without its
// FP64 epilogue.  B rows x n columns of synthetic state, `reps` passes each of
//   ms[0]  the production kernel (EpiDelta: the whole Douglas-Rachford update on the accumulators)
//   ms[1]  the same TMA + tcgen05 main loop with an epilogue that only drains TMEM (no state traffic, no FP64)
// so ms[1] is what the operand supply and the MMA issue can sustain and ms[0] - ms[1] what the epilogue exposes.
struct EpiLpDrain {
  struct Params { float* sink; };
  Params p;
  float acc;
  __device__ EpiLpDrain(const Params& p_, lp::EpiWarpSmem*, int) : p(p_), acc(0.f) {}
  __device__ void begin_tile(int, int) {}
  __device__ void chunk(int, const uint32_t (&a)[lp::CW], int) {
#pragma unroll
    for (int j = 0; j < lp::CW; ++j) acc += __uint_as_float(a[j]);
  }
  __device__ void end_tile() {
    if (acc == 123456.789f) *p.sink = acc;     // keeps the TMEM loads alive
  }
};

__global__ void k_probe_fill(double* V, double* X, float* E, __half* D, long long ldd, double* sc, int* state, long long B, int n) {
  const long long total = B * n;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / n;
    const int c = (int)(i - r * n);
    const double t = (double)((i * 2654435761ull) % 2001) / 1000.0 - 1.0;
    V[i] = 0.7 * t; X[i] = 0.6 * t; E[i] = 0.f;
    D[r * ldd + c] = __double2half(8.0 * t);
    if (c == 0) { sc[r] = 1024.0; state[r] = 1; }
  }
}

int nnmpc_lp_pass_probe(int B, int n, int reps, float* ms) {
  if (B <= 0 || n <= 0 || (n & 1) || n > B || reps <= 0 || !ms)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_lp_pass_probe: need even n <= B, reps > 0");
  cudaStream_t st = 0;
  int dev = 0;
  NNMPC_CUDA(cudaGetDevice(&dev));
  DevBuf<double> Top, V, lb, ub, sc;
  DevBuf<int> state;
  DevBuf<unsigned long long> dres;
  DevBuf<float> sink;
  LpState lps;
  LpOperator op;
  int rc = Top.ensure((size_t)n * n);
  if (rc == 0) rc = V.ensure((size_t)B * n);
  if (rc == 0) rc = lb.ensure((size_t)B * 32);
  if (rc == 0) rc = ub.ensure((size_t)B * 32);
  if (rc == 0) rc = sc.ensure((size_t)B);
  if (rc == 0) rc = state.ensure((size_t)B);
  if (rc == 0) rc = dres.ensure((size_t)B);
  if (rc == 0) rc = sink.ensure(1);
  lps.defer2 = true;
  if (rc == 0) rc = lp_state_ensure(&lps, B, n, st);
  if (rc == 0) {
    k_probe_fill<<<148 * 8, 256, 0, st>>>(Top.p, Top.p, lps.E.p, lps.D[0].p, lps.ldd, sc.p, state.p, n, n);   // any bounded operator
    k_probe_fill<<<148 * 8, 256, 0, st>>>(V.p, lps.X.p, lps.E.p, lps.D[0].p, lps.ldd, sc.p, state.p, B, n);
    cudaMemsetAsync(lb.p, 0xc0, (size_t)B * 32 * 8, st);     // -2.0...
    cudaMemsetAsync(ub.p, 0x40, (size_t)B * 32 * 8, st);     // +2.0...
    cudaMemsetAsync(dres.p, 0, (size_t)B * 8, st);
    cudaMemcpyAsync(lps.sc_in.p, sc.p, (size_t)B * 8, cudaMemcpyDeviceToDevice, st);
    cudaMemcpyAsync(lps.sc_out.p, sc.p, (size_t)B * 8, cudaMemcpyDeviceToDevice, st);
    rc = lp_split_operator(Top.p, n, 1.0, &op, st);
  }
  cudaEvent_t e0, e1, e2, e3, e4, e5, e6;
  cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventCreate(&e2); cudaEventCreate(&e3); cudaEventCreate(&e4); cudaEventCreate(&e5); cudaEventCreate(&e6);
  if (rc == 0) {
    const double tile_mb = 2.0 * LpTileN128::BN * (double)op.ldh * 2.0 / 1048576.0;
    int group_cols = (int)(24.0 / tile_mb);
    if (group_cols < 1) group_cols = 1;
    lp::LpShape g{B, n, n, nullptr, group_cols, nullptr, nullptr, 0, 0, 0};
    lp::LpShape g_epi = g;
    g_epi.skip_mma = 1;
    EpiDelta::Params ep{};
    ep.X = lps.X.p; ep.V = V.p; ep.E = lps.E.p; ep.Dn = lps.D[1].p; ep.ldd = lps.ldd; ep.lb = lb.p; ep.ub = ub.p;
    ep.state = state.p; ep.iter_state = 1; ep.list_r = nullptr; ep.pos_w = nullptr; ep.sc_in = lps.sc_in.p; ep.sc_out = lps.sc_out.p;
    ep.dres = dres.p; ep.n = n; ep.nu = 32; ep.alpha = 1.8; ep.inv_sT = 1.0 / op.scale;
    const int sms = device_sm_count(dev);
    for (int w = 0; w < 2; ++w) {
      lp::launch_lp_gemm<LpTileN128, EpiDelta>(lps.tmD[0], op.tm1, op.tm2, g, ep, sms, st);
      lp::launch_lp_gemm<LpTileN128, EpiLpDrain>(lps.tmD[0], op.tm1, op.tm2, g, EpiLpDrain::Params{sink.p}, sms, st);
    }
    // NNMPC_PROBE_ONLY = 0 / 1 / 2 runs one of the three phases alone (clock and power sampling from outside)
    const char* only_s = getenv("NNMPC_PROBE_ONLY");
    const int only = only_s ? atoi(only_s) : -1;
    cudaEventRecord(e0, st);
    for (int i = 0; i < reps && (only < 0 || only == 0); ++i)
      lp::launch_lp_gemm<LpTileN128, EpiDelta>(lps.tmD[0], op.tm1, op.tm2, g, ep, sms, st);
    cudaEventRecord(e1, st);
    for (int i = 0; i < reps && (only < 0 || only == 1); ++i)
      lp::launch_lp_gemm<LpTileN128, EpiLpDrain>(lps.tmD[0], op.tm1, op.tm2, g, EpiLpDrain::Params{sink.p}, sms, st);
    cudaEventRecord(e2, st);
    for (int i = 0; i < reps && (only < 0 || only == 2); ++i)
      lp::launch_lp_gemm<LpTileN128, EpiDelta>(lps.tmD[0], op.tm1, op.tm2, g_epi, ep, sms, st);
    cudaEventRecord(e3, st);
    // deferred second term: the one-term pass (increment added to the pending sum) and the delivery GEMM
    cudaMemcpyAsync(lps.sS.p, sc.p, (size_t)B * 8, cudaMemcpyDeviceToDevice, st);
    cudaMemcpyAsync(lps.S[0].p, lps.D[0].p, (size_t)B * lps.ldd * sizeof(__half), cudaMemcpyDeviceToDevice, st);
    EpiDelta::Params ep1 = ep;
    ep1.s_mode = 1; ep1.Sc = lps.S[0].p; ep1.Sn = lps.S[1].p; ep1.sS = lps.sS.p;
    lp::LpShape g1 = g;
    g1.group_cols = 2 * group_cols;
    EpiAddX::Params epx{lps.X.p, state.p, 1, nullptr, lps.sS.p, n, 1.0 / op.scale};
    const bool m256 = getenv("NNMPC_LP1_TILE") && strcmp(getenv("NNMPC_LP1_TILE"), "m256") == 0;
    auto pass1 = [&]() {
      if (m256) lp::launch_lp_gemm<LpTile1M256, EpiDelta>(lps.tmD256[0], op.tm1, op.tm1, g1, ep1, sms, st);
      else lp::launch_lp_gemm<LpTile1N128, EpiDelta>(lps.tmD[0], op.tm1, op.tm1, g1, ep1, sms, st);
    };
    auto corr = [&]() {
      if (m256) lp::launch_lp_gemm<LpTile1M256, EpiAddX>(lps.tmS256[0], op.tm2, op.tm2, g1, epx, sms, st);
      else lp::launch_lp_gemm<LpTile1N128, EpiAddX>(lps.tmS[0], op.tm2, op.tm2, g1, epx, sms, st);
    };
    pass1(); corr();
    cudaEventRecord(e6, st);
    for (int i = 0; i < reps && (only < 0 || only == 3); ++i) pass1();
    cudaEventRecord(e4, st);
    for (int i = 0; i < reps && (only < 0 || only == 4); ++i) corr();
    cudaEventRecord(e5, st);
    if (cudaEventSynchronize(e5) != cudaSuccess)
      rc = set_error(NNMPC_ERR_CUDA, "lp pass probe failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (rc == 0) {
      cudaEventElapsedTime(&ms[0], e0, e1);
      cudaEventElapsedTime(&ms[1], e1, e2);
      cudaEventElapsedTime(&ms[2], e2, e3);
      cudaEventElapsedTime(&ms[3], e6, e4);
      cudaEventElapsedTime(&ms[4], e4, e5);
      ms[0] /= reps; ms[1] /= reps; ms[2] /= reps; ms[3] /= reps; ms[4] /= reps;
    }
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(e2); cudaEventDestroy(e3); cudaEventDestroy(e4); cudaEventDestroy(e5); cudaEventDestroy(e6);
  cudaStreamSynchronize(st);
  for (DevBuf<double>* b : {&Top, &V, &lb, &ub, &sc}) b->release();
  state.release(); dres.release(); sink.release(); lps.release(); op.release();
  return rc;
}

}  // extern "C"
