// Host-visible interface of the mixed-precision (tcgen05 fp16 increments + FP64 anchors) iteration
// of the regulator QP; device code lives in lp_gemm.cuh / lp_iter.cuh and is compiled in lp.cu.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include "qp.cuh"

namespace nnmpc {

// per-sample state of the mixed-precision iteration for up to `cap` rows (see lp_iter.cuh)
struct LpState {
  long long cap = 0;
  int n = 0;
  long long ldd = 0;                 // leading dimension of the fp16 increment buffers
  DevBuf<double> X, sc_in, sc_out;
  DevBuf<double> Wl;                 // exact gradient of the last check, then w_lp, then the staged first increment
  DevBuf<float> E;
  DevBuf<__half> D[2];               // double buffered: the TMA reads D[cur], the epilogue writes D[cur ^ 1]
  CUtensorMap tmD[2];
  CUtensorMap tmD256[2];             // the same buffers with 256-row boxes (LpTile<.,.,2>)
  // deferred second operator term (lp_iter.cuh): pending sums of the increments, laid out and flipped like D, and the
  // per-row scale of each sum.  Allocated when defer2 is set before lp_state_ensure.
  bool defer2 = false;
  DevBuf<__half> S[2];
  DevBuf<double> sS;
  CUtensorMap tmS[2];
  CUtensorMap tmS256[2];
  int cur = 0;
  void release() {
    Wl.release(); X.release(); sc_in.release(); sc_out.release(); E.release(); D[0].release(); D[1].release();
    S[0].release(); S[1].release(); sS.release(); cap = 0;
  }
};

#ifdef __CUDACC__
// largest power of two s with s * est in [8, 16], clamped to 2^+-60 (est = 0, NaN or Inf -> 2^60 / 2^-60)
__device__ __forceinline__ double pow2_scale(double est) {
  if (!(est > 0.0)) return 1152921504606846976.0;                 // 2^60
  if (!(est <= 1.7e308)) return 8.673617379884035e-19;            // 2^-60
  int ex;
  frexp(est, &ex);                                                // est = m 2^ex, m in [0.5, 1)
  int sh = 4 - ex;
  sh = sh > 60 ? 60 : (sh < -60 ? -60 : sh);
  return ldexp(1.0, sh);
}
#endif

int device_sm_count(int device);
int lp_split_operator(const double* T_dev, int n, double tmax, LpOperator* op, cudaStream_t st);
int lp_state_ensure(LpState* s, long long B, int n, cudaStream_t st);

// rows listed in rows[0..*count): w = 2 clip(v) - v into W (the FP64 anchor GEMM operand), E = 0
int lp_anchor_prep(const int* rows, const int* count, int max_rows, const double* V, double* W, LpState* s,
                   const double* lb, const double* ub, int nu, cudaStream_t st);
// FP64 anchor GEMM x = Top w - c over the listed rows (DMMA kernel, tile shape picked by the device-side count)
int lp_anchor_gemm(const int* rows, const int* count, int max_rows, const double* W, const double* Top, const double* C,
                   double* X, int n, cudaStream_t st);
// listed rows: one FP64 Douglas-Rachford step from the exact x, first fp16 increment, state := iter_state
// pos_r: sample row -> row of the operand buffer the next pass reads (null = identity); a negative position writes no
// operand row (no D, S or need2 flag; E, the scales, state and it are updated)
int lp_dr_first(const int* rows, const int* count, int max_rows, LpState* s, double* V, double* W, const double* lb,
                const double* ub, int* state, int* it, int iter_state, int nu, double alpha, const int* pos_r,
                cudaStream_t st, unsigned char* need2 = nullptr);   // need2: operand tiles of these rows get both operator terms
// candidates that failed their exact check (state == emit_state; Wl holds g = P z + q): x := z, Wl := w_lp = z + g / rho
int lp_reanchor(const int* rows, const int* count, int max_rows, const int* state, int emit_state, const double* Z,
                const double* rinv, LpState* s, cudaStream_t st);
// listed rows in emit_state: first fp16 increment from the exactly anchored (x, w_lp); state := iter_state
// (pos_r as for lp_dr_first, a negative position included)
int lp_emit(const int* rows, const int* count, int max_rows, int* state, int emit_state, int iter_state, LpState* s,
            const double* V, const double* lb, const double* ub, const double* dtrig, int nu, double alpha,
            const int* pos_r, cudaStream_t st, unsigned char* need2 = nullptr);
// One tensor-core pass over the operand rows [0, *len_r) (at most B); flips s->cur.  Operand row p belongs to
// sample list_r[p]; it takes part iff state[sample] == iter_state, and its next increment is written to
// operand row pos_w[sample] of the other buffer (so the layout is re-compacted one pass behind the live list).
// Precondition: 0 <= pos_w[sample] < B for every sample that takes part (the epilogue does not check it).  The engine
// (sim.cu) meets it, and passes non-negative positions to lp_dr_first / lp_emit as well: k_step gives every live row
// (ITER, RENEW, ANCHOR, EMIT) a position and -1 only to IDLE rows, a row is IDLE only when no chunk is left for its slot,
// and an IDLE row never becomes live again; the rows of one layout that iterate, start a QP (anchor) or are re-emitted
// before the next k_step were live when it was built.
// kernel: -1 = the process default (NNMPC_LP_KERNEL, NNMPC_LP_TILE; NNMPC_LP1_TILE for s_mode != 0), else s_mode 0:
// 0 = 128 x 128 tiles, 1 = 256 x 128 tiles, 2 = CTA pair; s_mode 1 / 2: 0 = 128 x 128, 1 = 256 x 128.
int lp_iterate(const LpOperator* op, LpState* s, int B, const int* list_r, const int* len_r, const int* pos_w, double* V,
               const double* lb, const double* ub, const int* state, int iter_state, unsigned long long* dres, int nu,
               double alpha, int device, cudaStream_t st, const unsigned char* need2 = nullptr,
               unsigned long long* tile_stat = nullptr, int s_mode = 0, int kernel = -1);
// Deferred second operator term: x += T2 S / (s_T sS) over the operand rows the NEXT lp_iterate will read (same
// list / state predicate); that pass must then run with s_mode = 2 (a new pending sum starts).  s_mode of
// lp_iterate: 0 = two-term pass (no pending sums), 1 = one-term pass, increment added to the pending sum, 2 = one-term
// pass, pending sum restarted.
int lp_correct(const LpOperator* op, LpState* s, int B, const int* list_r, const int* len_r, const int* state,
               int iter_state, int device, cudaStream_t st, unsigned long long* tile_stat = nullptr,   // tile_stat[0] += tiles
               int kernel = -1);     // -1 = NNMPC_LP1_TILE, 0 = 128 x 128 tiles, 1 = 256 x 128 tiles


}  // namespace nnmpc
