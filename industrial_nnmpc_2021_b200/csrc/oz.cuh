// Host-visible interface of the INT8-sliced FP64-accurate GEMM (oz_gemm.cuh); compiled in oz.cu.
#pragma once
#include <cuda.h>
#include <stdint.h>
#include "nnmpc_common.cuh"

namespace nnmpc {

// a shared FP64 operator (rows = output columns of the GEMM) cut into signed base-128 digit planes
struct OzOperator {
  int nrows = 0, ncols = 0;
  long long ldb = 0;        // bytes per row of a plane (multiple of 128, zero padded)
  long long rows_pad = 0;   // rows per plane (multiple of 128, zero padded)
  DevBuf<int8_t> S;         // NS planes stacked: [(s * rows_pad + row) * ldb + k]
  DevBuf<double> escale;    // per row: 2^e, max |row| <= 2^(e-1)
  CUtensorMap tm;           // boxes of 64 operator rows
  CUtensorMap tm128;        // boxes of 128 operator rows
  bool ready = false;
  void release() { S.release(); escale.release(); ready = false; }
};

// digit planes of up to cap sample rows (rewritten before every GEMM)
struct OzRows {
  long long cap_pad = 0;    // rows per plane (multiple of 128)
  long long ldb = 0;
  int ncols = 0;
  int ns = 0;               // digit planes kept (8 for the FP64-exact applies, 4 for the structured-network layers)
  DevBuf<int8_t> S;
  DevBuf<double> fscale;    // per position: 2^f
  DevBuf<double> partial;   // cap_pad x ncols: partial level sums between the two launches of the 128-column kernel
  CUtensorMap tm;
  void release() { S.release(); fscale.release(); partial.release(); cap_pad = 0; }
};

int oz_slice_operator(const double* T_dev, int nrows, int ncols, OzOperator* op, cudaStream_t st, long long ld = 0);
int oz_rows_ensure(OzRows* r, long long cap, int ncols, cudaStream_t st, int ns = 0);
// One Dense layer of the structured network on the INT8 tensor cores: out[M x N] = act(A[M x K] W^T + bias), with A
// (FP64, leading dimension lda) cut into 4 signed base-128 digit planes per row (28 bits below the row maximum) and
// the 10 digit-plane products of levels 0..3 accumulated exactly in INT32 - no accumulation error, truncation
// <= 4 K 2^-30 relative to (row max) x (weight-row max).  W: operator planes from oz_slice_operator (N x K).
int oz_dense_layer(const OzOperator* W, OzRows* r, int M, const double* A, long long lda, const double* bias, int relu,
                   double* out, long long ldo, int device, cudaStream_t st);
// The same layer between DIGIT-PLANE operands: reads the planes already in `rin` (scales in rin->fscale); the epilogue
// writes relu(. + bias) as fp32 into hbuf (row pitch ldh floats, a multiple of 4 and >= the width rounded up to 64) and
// the exact row maxima into amax_out (atomicMax, zeroed by the caller), then one slicing pass cuts the planes of `rout`
// with exact scales - no FP64 activations in memory.  out != NULL (last layer, no bias / ReLU): plain FP64 result.
int oz_dense_planes(const OzOperator* W, OzRows* rin, int M, const double* bias, OzRows* rout, float* hbuf, long long ldh,
                    float* amax_out, double* out, long long ldo, int device, cudaStream_t st);
// first-layer operand of the structured network straight into digit planes: rows 2b / 2b+1 = [x/s, (uprev), xs/s, us] /
// [xs/s, (us), xs/s, us] (controller_evaluation.py:863-866), one warp per sample
int oz_pack_network_input(OzRows* r, long long B, const double* x, const double* uprev, const double* xs, const double* us,
                          const double* xscale, int nx, int nu, int with_uprev, float* amax, cudaStream_t st);
// x = Top w - c for the listed rows (W, C, X are B x n with the sample row as physical row)
int oz_anchor(const OzOperator* top, OzRows* r, const int* rows, const int* count, int max_rows, const double* W,
              const double* C, double* X, int n, int device, cudaStream_t st, int variant = -1);
// g = P z + q for the listed rows; per row ||z - clip(z - g)||_inf folded into kres (atomicMax of the bit pattern),
// g itself into G when non-null
// variant (both): kernel variant of the apply, -1 = the process default (NNMPC_OZ_VARIANT, read once)
int oz_verify(const OzOperator* P, OzRows* r, const int* rows, const int* count, int max_rows, const double* Z,
              const double* Ql, const double* lb, const double* ub, unsigned long long* kres, double* G, int n, int nu,
              int device, cudaStream_t st, int variant = -1);

}  // namespace nnmpc
