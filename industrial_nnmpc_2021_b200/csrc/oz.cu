// Host-side glue and fused epilogues of the INT8-sliced FP64-accurate GEMM (oz_gemm.cuh): the exact anchors
// x = Top w - c and the exact KKT checks g = P z + q of the mixed-precision closed-loop engine, and the
// self-test entry point.
#include "oz_gemm.cuh"
#include "oz.cuh"
#include "lp.cuh"     // device_sm_count
#include <cstdlib>
#include <cstring>

namespace nnmpc {

constexpr int OZ_LMAX = 7;     // levels 0..7: 36 INT8 products, truncation (LMAX+1) K 2^(-7 (LMAX+1) - 2) ~ 1.2e-13 at K = 4480
constexpr int OZ_NS = OZ_LMAX + 1;
#ifndef NNMPC_OZ_LMAX_ANCHOR
#define NNMPC_OZ_LMAX_ANCHOR 5
#endif
constexpr int OZ_LMAX_ANCHOR = NNMPC_OZ_LMAX_ANCHOR;   // anchors: 6 levels = 21 products (|Top| <= 1; the result only steers the iteration, the 8-level check certifies; measured: same checks per QP as with 7 levels)

// kernel variant: 2 (default) = 128-column tiles, two level windows; 3 = the high window on 128-column tiles, the low
// window (levels 0..3, whose epilogue - partial sums in, functor out - is as long as its 10 products) on 64-column
// tiles with DOUBLE-BUFFERED accumulators, so that epilogue overlaps the next tile's products; 1 = 64-column tiles, one
// launch, just-in-time operator slices; 0 = first-generation kernel (64 columns, double-buffered slice sets)
static int oz_variant() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("NNMPC_OZ_VARIANT");
    v = e ? atoi(e) : 2;
    if (v < 0 || v > 3) v = 2;
  }
  return v;
}

// ---- epilogues (one lane = one output row, CH consecutive columns per call) ---------------------
struct OzEpiStore {
  struct Params {
    double* C;
    long long ldc;
  };
  Params p;
  long long pos;
  __device__ explicit OzEpiStore(const Params& p_) : p(p_), pos(0) {}
  __device__ void begin_row(int pos_, bool) { pos = pos_; }
  __device__ void chunk(int col0, const double (&v)[oz::CH], int N) {
#pragma unroll
    for (int k = 0; k < oz::CH; ++k)
      if (col0 + k < N) p.C[pos * p.ldc + col0 + k] = v[k];
  }
  __device__ void end_row() {}
};

struct OzEpiAnchor {
  struct Params {
    double* X;
    const double* C;
    const int* rows;
    int n;
  };
  Params p;
  long long base;
  __device__ explicit OzEpiAnchor(const Params& p_) : p(p_), base(0) {}
  __device__ void begin_row(int pos, bool ok) { base = ok ? (long long)(p.rows ? p.rows[pos] : pos) * p.n : 0; }
  __device__ void chunk(int col0, const double (&v)[oz::CH], int N) {
    // all loads of C first: a load cannot be moved above the store of X of an earlier column pair (they may alias)
    double2 c[oz::CH / 2];
#pragma unroll
    for (int k = 0; k < oz::CH; k += 2) {
      const int col = col0 + k;
      c[k / 2] = make_double2(0.0, 0.0);
      if (col + 1 < N) c[k / 2] = *reinterpret_cast<const double2*>(p.C + base + col);
      else if (col < N) c[k / 2].x = p.C[base + col];
    }
#pragma unroll
    for (int k = 0; k < oz::CH; k += 2) {
      const int col = col0 + k;
      if (col + 1 < N) *reinterpret_cast<double2*>(p.X + base + col) = make_double2(v[k] - c[k / 2].x, v[k + 1] - c[k / 2].y);
      else if (col < N) p.X[base + col] = v[k] - c[k / 2].x;
    }
  }
  __device__ void end_row() {}
};

struct OzEpiVerify {
  struct Params {
    const double* Z;
    const double* Ql;
    const double* lb;
    const double* ub;
    unsigned long long* kres;
    double* G;        // nullable
    const int* rows;
    int n, nu;
  };
  Params p;
  long long pr;
  bool ok;
  double rmax;
  __device__ explicit OzEpiVerify(const Params& p_) : p(p_), pr(0), ok(false), rmax(0.0) {}
  __device__ void begin_row(int pos, bool ok_) {
    ok = ok_;
    pr = ok ? (long long)(p.rows ? p.rows[pos] : pos) : 0;
    rmax = 0.0;
  }
  __device__ void chunk(int col0, const double (&v)[oz::CH], int N) {
    const long long base = pr * p.n;
    const double* lbr = p.lb + pr * p.nu;
    const double* ubr = p.ub + pr * p.nu;
    // two halves, each: all loads, then the arithmetic and the stores - a load cannot be moved above the store of G of
    // an earlier column (they may alias), so a column-by-column loop pays one exposed round trip per column
#pragma unroll
    for (int h = 0; h < oz::CH; h += oz::CH / 2) {
      double z[oz::CH / 2], ql[oz::CH / 2], l[oz::CH / 2], u[oz::CH / 2];
#pragma unroll
      for (int k = 0; k < oz::CH / 2; ++k) {
        const int col = col0 + h + k;
        const bool in = col < N;
        const int s = (in ? col : 0) % p.nu;
        z[k] = in ? p.Z[base + col] : 0.0;
        ql[k] = in ? p.Ql[base + col] : 0.0;
        l[k] = lbr[s];
        u[k] = ubr[s];
      }
#pragma unroll
      for (int k = 0; k < oz::CH / 2; ++k) {
        const int col = col0 + h + k;
        if (col < N) {
          const double g = v[h + k] + ql[k];
          if (p.G) p.G[base + col] = g;
          double r = fabs(z[k] - fmin(fmax(z[k] - g, l[k]), u[k]));
          // NaN/Inf must not look converged (an infinite g clips to a bound and leaves r finite)
          if (!(r <= 1.7e308 && fabs(g) <= 1.7e308)) r = __longlong_as_double(0x7ff0000000000000ll);
          rmax = fmax(rmax, r);
        }
      }
    }
  }
  __device__ void end_row() {
    if (ok) atomicMax(p.kres + pr, (unsigned long long)__double_as_longlong(rmax));
  }
};

// ---- host side ---------------------------------------------------------------------------------
int oz_slice_operator(const double* T_dev, int nrows, int ncols, OzOperator* op, cudaStream_t st, long long ld) {
  if (ncols > 32768) return set_error(NNMPC_ERR_BADARG, "oz_slice_operator: contraction length %d above 32768 (int32 accumulators)", ncols);
  op->nrows = nrows; op->ncols = ncols;
  op->ldb = ((long long)ncols + oz::BKB - 1) / oz::BKB * oz::BKB;
  op->rows_pad = ((long long)nrows + 127) / 128 * 128;
  const size_t bytes = (size_t)OZ_NS * op->rows_pad * op->ldb;
  NNMPC_TRY(op->S.ensure(bytes));
  NNMPC_TRY(op->escale.ensure((size_t)op->rows_pad));
  NNMPC_CUDA(cudaMemsetAsync(op->S.p, 0, bytes, st));
  NNMPC_CUDA(cudaMemsetAsync(op->escale.p, 0, (size_t)op->rows_pad * sizeof(double), st));
  oz::k_oz_slice<OZ_NS><<<nrows, 256, 0, st>>>(nullptr, nullptr, T_dev, ld > 0 ? ld : ncols, ncols, op->S.p, op->rows_pad,
                                               op->ldb, op->escale.p, nrows);
  count_launch();
  NNMPC_CUDA(cudaGetLastError());
  if (!oz::make_tmap_u8(&op->tm, op->S.p, OZ_NS * op->rows_pad, op->ldb, op->ldb, oz::BN))
    return set_error(NNMPC_ERR_CUDA, "cuTensorMapEncodeTiled failed for the operator digit planes");
  if (!oz::make_tmap_u8(&op->tm128, op->S.p, OZ_NS * op->rows_pad, op->ldb, op->ldb, 128))
    return set_error(NNMPC_ERR_CUDA, "cuTensorMapEncodeTiled failed for the operator digit planes");
  op->ready = true;
  return 0;
}

int oz_rows_ensure(OzRows* r, long long cap, int ncols, cudaStream_t st, int ns) {
  if (ns <= 0) ns = OZ_NS;
  const long long ldb = ((long long)ncols + oz::BKB - 1) / oz::BKB * oz::BKB;
  const long long cap_pad = (cap + oz::BM - 1) / oz::BM * oz::BM;
  if (cap_pad <= r->cap_pad && ldb == r->ldb && ncols == r->ncols && ns == r->ns) return 0;
  const long long cp = cap_pad > r->cap_pad ? cap_pad : r->cap_pad;
  const size_t bytes = (size_t)ns * cp * ldb;
  NNMPC_TRY(r->S.ensure(bytes));
  NNMPC_TRY(r->fscale.ensure((size_t)cp));
  NNMPC_CUDA(cudaMemsetAsync(r->S.p, 0, bytes, st));      // the k-padding stays zero: the slicing kernel writes ncols bytes per row
  NNMPC_CUDA(cudaMemsetAsync(r->fscale.p, 0, (size_t)cp * sizeof(double), st));
  if (!oz::make_tmap_u8(&r->tm, r->S.p, ns * cp, ldb, ldb, oz::BM))
    return set_error(NNMPC_ERR_CUDA, "cuTensorMapEncodeTiled failed for the sample digit planes");
  r->cap_pad = cp; r->ldb = ldb; r->ncols = ncols; r->ns = ns;
  return 0;
}

static int oz_slice_rows(OzRows* r, const int* rows, const int* count, int max_rows, const double* src, long long ld_src,
                         cudaStream_t st) {
  if (r->ns == 4 && !rows && !count && r->ncols <= 4096)      // dense list of short rows: one warp per row
    oz::k_oz_slice_warp<4><<<row_grid((max_rows + 7) / 8), 256, 0, st>>>(src, ld_src, r->ncols, r->S.p, r->cap_pad, r->ldb,
                                                                         r->fscale.p, max_rows);
  else if (r->ns == 4)
    oz::k_oz_slice<4><<<row_grid(max_rows), 256, 0, st>>>(rows, count, src, ld_src, r->ncols, r->S.p, r->cap_pad, r->ldb,
                                                          r->fscale.p, max_rows);
  else
    oz::k_oz_slice<OZ_NS><<<row_grid(max_rows), 256, 0, st>>>(rows, count, src, ld_src, r->ncols, r->S.p, r->cap_pad, r->ldb,
                                                              r->fscale.p, max_rows);
  count_launch();
  NNMPC_CUDA(cudaGetLastError());
  return 0;
}

static oz::OzShape oz_shape(const OzOperator* op, const OzRows* r, int max_rows, const int* count) {
  oz::OzShape g{};
  g.M = max_rows; g.N = op->nrows; g.KB = (int)(op->ldb / oz::BKB); g.m_dev = count;
  g.a_rows_pad = r->cap_pad; g.b_rows_pad = op->rows_pad; g.fscale = r->fscale.p; g.escale = op->escale.p;
  g.group_rows = 8;
  return g;
}

// one FP64-accurate apply over the sliced rows: levels 0..LMAX through kernel variant `variant` (-1: oz_variant())
template <int LMAX, class Epi>
static int oz_apply(const OzOperator* op, OzRows* r, int max_rows, const int* count, const typename Epi::Params& ep,
                    int device, cudaStream_t st, int variant = -1) {
  const int sms = device_sm_count(device);
  const oz::OzShape g = oz_shape(op, r, max_rows, count);
  cudaError_t e;
  const int var = variant >= 0 ? variant : oz_variant();
  if (var == 0) {
    e = oz::launch_oz_gemm<LMAX, Epi>(r->tm, op->tm, g, ep, sms, st);
    count_launch();
  } else if (var == 1) {
    e = oz::launch_oz_gemm2<0, LMAX, 64, Epi>(r->tm, op->tm, oz::OzShape2{g, nullptr, 0, 0}, ep, sms, st);
    count_launch();
  } else {
    NNMPC_TRY(r->partial.ensure((size_t)r->cap_pad * op->nrows));
    e = oz::launch_oz_gemm2<4, LMAX, 128, OzEpiStore>(r->tm, op->tm128, oz::OzShape2{g, nullptr, 0, 1},
                                                      OzEpiStore::Params{r->partial.p, op->nrows}, sms, st);
    if (e == cudaSuccess)
      e = var == 3 ? oz::launch_oz_gemm2<0, 3, 64, Epi>(r->tm, op->tm, oz::OzShape2{g, r->partial.p, op->nrows, 0}, ep, sms, st)
                   : oz::launch_oz_gemm2<0, 3, 128, Epi>(r->tm, op->tm128, oz::OzShape2{g, r->partial.p, op->nrows, 0}, ep, sms, st);
    count_launch(2);
  }
  if (e != cudaSuccess) return set_error(NNMPC_ERR_CUDA, "oz_gemm launch failed: %s", cudaGetErrorString(e));
  return 0;
}

int oz_anchor(const OzOperator* top, OzRows* r, const int* rows, const int* count, int max_rows, const double* W,
              const double* C, double* X, int n, int device, cudaStream_t st, int variant) {
  if (max_rows <= 0) return 0;
  if (!top->ready || top->ncols != n || r->ncols != n || max_rows > r->cap_pad)
    return set_error(NNMPC_ERR_BADARG, "oz_anchor: operator / row planes not prepared for n = %d, %d rows", n, max_rows);
  NNMPC_TRY(oz_slice_rows(r, rows, count, max_rows, W, n, st));
  return oz_apply<OZ_LMAX_ANCHOR, OzEpiAnchor>(top, r, max_rows, count, OzEpiAnchor::Params{X, C, rows, n}, device, st,
                                               variant);
}

int oz_verify(const OzOperator* P, OzRows* r, const int* rows, const int* count, int max_rows, const double* Z,
              const double* Ql, const double* lb, const double* ub, unsigned long long* kres, double* G, int n, int nu,
              int device, cudaStream_t st, int variant) {
  if (max_rows <= 0) return 0;
  if (!P->ready || P->ncols != n || r->ncols != n || max_rows > r->cap_pad)
    return set_error(NNMPC_ERR_BADARG, "oz_verify: operator / row planes not prepared for n = %d, %d rows", n, max_rows);
  NNMPC_TRY(oz_slice_rows(r, rows, count, max_rows, Z, n, st));
  return oz_apply<OZ_LMAX, OzEpiVerify>(P, r, max_rows, count, OzEpiVerify::Params{Z, Ql, lb, ub, kres, G, rows, n, nu},
                                        device, st, variant);
}

// ---- structured-network Dense layer (mlp.cu) ---------------------------------------------------------------------
struct OzEpiDense {
  struct Params {
    double* out;
    long long ldo;
    const double* bias;   // nullable
    int relu;
  };
  Params p;
  long long pos;
  __device__ explicit OzEpiDense(const Params& p_) : p(p_), pos(0) {}
  __device__ void begin_row(int pos_, bool) { pos = pos_; }
  __device__ void chunk(int col0, const double (&v)[oz::CH], int N) {
#pragma unroll
    for (int k = 0; k < oz::CH; ++k) {
      const int col = col0 + k;
      if (col < N) {
        double h = v[k] + (p.bias ? __ldg(p.bias + col) : 0.0);
        if (p.relu) h = relu_keep_nan(h);
        p.out[pos * p.ldo + col] = h;
      }
    }
  }
  __device__ void end_row() {}
};

int oz_dense_layer(const OzOperator* W, OzRows* r, int M, const double* A, long long lda, const double* bias, int relu,
                   double* out, long long ldo, int device, cudaStream_t st) {
  if (M <= 0) return 0;
  if (!W->ready) return set_error(NNMPC_ERR_BADARG, "oz_dense_layer: weights not sliced");
  NNMPC_TRY(oz_rows_ensure(r, M, W->ncols, st, 4));
  NNMPC_TRY(oz_slice_rows(r, nullptr, nullptr, M, A, lda, st));
  const oz::OzShape g = oz_shape(W, r, M, nullptr);
  // 64-column tiles: the 4-level window then fits TMEM twice and the accumulators are double buffered
  cudaError_t e = oz::launch_oz_gemm2<0, 3, 64, OzEpiDense>(r->tm, W->tm, oz::OzShape2{g, nullptr, 0, 0},
                                                            OzEpiDense::Params{out, ldo, bias, relu},
                                                            device_sm_count(device), st);
  count_launch();
  if (e != cudaSuccess) return set_error(NNMPC_ERR_CUDA, "oz_gemm launch failed: %s", cudaGetErrorString(e));
  return 0;
}

// hidden layer: relu(. + bias) as fp32 plus the exact row maximum; k_oz_slice_f32 then cuts the digit planes of the next
// layer's operand with the EXACT power-of-two scale of each row.  (Cutting the planes right in this epilogue needs the
// scale before the row is complete, i.e. an a-priori bound max|a| ||W||_1 + max|b|; measured on B200: that bound is
// ~25x loose on the CDU network, the level-truncation error of the next GEMM scales with it, and the outputs drift to
// 4.6e-6 of the float64 layer instead of 1.3e-7 - too close to the 1e-5 tolerance.)
struct OzEpiDenseF32 {
  struct Params {
    float* H;
    long long ldh;
    const double* bias;
    float* amax_out;       // per row: max entry written (atomicMax on the bit pattern; entries are >= 0 or +NaN)
  };
  Params p;
  long long pos;
  float hmax;
  __device__ explicit OzEpiDenseF32(const Params& p_) : p(p_), pos(0), hmax(0.f) {}
  __device__ void begin_row(int pos_, bool) {
    pos = pos_;
    hmax = 0.f;
  }
  __device__ void chunk(int col0, const double (&v)[oz::CH], int N) {
    __align__(16) float h[oz::CH];
#pragma unroll
    for (int k = 0; k < oz::CH; ++k) {
      double t = 0.0;
      if (col0 + k < N) {
        t = relu_keep_nan(v[k] + __ldg(p.bias + col0 + k));
      }
      h[k] = (float)t;
      hmax = row_max_keep_nan(hmax, h[k]);    // a NaN row must reach k_oz_slice_f32 with a NaN maximum
    }
    float4* dst = reinterpret_cast<float4*>(p.H + pos * p.ldh + col0);
#pragma unroll
    for (int q = 0; q < oz::CH / 4; ++q) dst[q] = reinterpret_cast<const float4*>(h)[q];
  }
  __device__ void end_row() {
    atomicMax(reinterpret_cast<unsigned int*>(p.amax_out + pos), __float_as_uint(hmax));
  }
};

// fp32 rows with KNOWN maxima -> 4 digit planes (one warp per row, one pass)
__global__ void __launch_bounds__(256)
k_oz_slice_f32(const float* __restrict__ H, long long ldh, int ncols, const float* __restrict__ amax, int8_t* __restrict__ dst,
               long long rows_pad, long long ldb, double* __restrict__ fscale, long long nrows) {
  const int lane = threadIdx.x & 31;
  const long long wpg = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long p = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); p < nrows; p += wpg) {
    const float* a = H + p * ldh;
    const double m = (double)amax[p];
    const bool bad = !(m <= 1.7e308);
    int ex = 0;
    if (!bad && m > 0.0) frexp(m, &ex);
    const double inv = bad ? 0.0 : ldexp(1.0, -(ex + 1));
    for (int k = 4 * lane; k < ncols; k += 128) {          // ldh and the plane pitch are multiples of 4: whole float4 / char4
      const float4 f = *reinterpret_cast<const float4*>(a + k);
      double t[4] = {bad ? 0.0 : f.x * inv, bad ? 0.0 : f.y * inv, bad ? 0.0 : f.z * inv, bad ? 0.0 : f.w * inv};
#pragma unroll
      for (int s = 0; s < 4; ++s) {
        char4 d;
        int8_t* dd = reinterpret_cast<int8_t*>(&d);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          t[e] *= 128.0;
          const double r = rint(t[e]);
          t[e] -= r;
          dd[e] = (k + e < ncols) ? (int8_t)(int)r : (int8_t)0;
        }
        *reinterpret_cast<char4*>(dst + ((long long)s * rows_pad + p) * ldb + k) = d;
      }
    }
    if (lane == 0) fscale[p] = bad ? __longlong_as_double(0x7ff8000000000000ll) : ldexp(1.0, ex + 1);
  }
}

int oz_dense_planes(const OzOperator* W, OzRows* rin, int M, const double* bias, OzRows* rout, float* hbuf, long long ldh,
                    float* amax_out, double* out, long long ldo, int device, cudaStream_t st) {
  if (M <= 0) return 0;
  if (!W->ready || rin->ns != 4 || rin->ncols != W->ncols || M > rin->cap_pad)
    return set_error(NNMPC_ERR_BADARG, "oz_dense_planes: operands not prepared");
  const oz::OzShape g = oz_shape(W, rin, M, nullptr);
  cudaError_t e;
  if (out) {
    e = oz::launch_oz_gemm2<0, 3, 64, OzEpiDense>(rin->tm, W->tm, oz::OzShape2{g, nullptr, 0, 0},
                                                  OzEpiDense::Params{out, ldo, bias, 0}, device_sm_count(device), st);
    count_launch();
  } else {
    if (rout->ns != 4 || rout->ncols != W->nrows || M > rout->cap_pad || (ldh & 3) || ldh < ((W->nrows + 63) / 64) * 64)
      return set_error(NNMPC_ERR_BADARG, "oz_dense_planes: output planes / fp32 scratch not prepared");
    e = oz::launch_oz_gemm2<0, 3, 64, OzEpiDenseF32>(rin->tm, W->tm, oz::OzShape2{g, nullptr, 0, 0},
                                                     OzEpiDenseF32::Params{hbuf, ldh, bias, amax_out}, device_sm_count(device), st);
    if (e == cudaSuccess) {
      k_oz_slice_f32<<<row_grid((M + 7) / 8), 256, 0, st>>>(hbuf, ldh, W->nrows, amax_out, rout->S.p, rout->cap_pad, rout->ldb,
                                                            rout->fscale.p, M);
      e = cudaGetLastError();
    }
    count_launch(2);
  }
  if (e != cudaSuccess) return set_error(NNMPC_ERR_CUDA, "oz_gemm launch failed: %s", cudaGetErrorString(e));
  return 0;
}

__global__ void __launch_bounds__(256)
k_oz_pack_network_input(const double* __restrict__ x, const double* __restrict__ uprev, const double* __restrict__ xs,
                        const double* __restrict__ us, const double* __restrict__ xscale, int8_t* __restrict__ dst,
                        long long rows_pad, long long ldb, double* __restrict__ fscale, float* __restrict__ amax, long long B,
                        int nx, int nu, int with_uprev) {
  const int lane = threadIdx.x & 31;
  const long long wpg = (long long)gridDim.x * (blockDim.x >> 5);
  const int o1 = nx, o2 = nx + (with_uprev ? nu : 0), o3 = o2 + nx, o4 = o3 + nu;
  for (long long b = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); b < B; b += wpg) {
    auto value = [&](int c, double& v1, double& v2) {
      if (c < o1) {
        v1 = x[b * nx + c];
        v2 = xs[b * nx + c];
        if (xscale) { v1 /= xscale[c]; v2 /= xscale[c]; }
      } else if (c < o2) {
        v1 = uprev[b * nu + (c - o1)];
        v2 = us[b * nu + (c - o1)];
      } else if (c < o3) {
        v1 = xs[b * nx + (c - o2)];
        if (xscale) v1 /= xscale[c - o2];
        v2 = v1;
      } else {
        v1 = v2 = us[b * nu + (c - o3)];
      }
    };
    double m1 = 0.0, m2 = 0.0;
    for (int c = lane; c < o4; c += 32) {
      double v1, v2;
      value(c, v1, v2);
      const double a1 = fabs(v1), a2 = fabs(v2);
      m1 = nan_max(m1, a1);
      m2 = nan_max(m2, a2);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double a1 = __shfl_xor_sync(0xffffffffu, m1, o), a2 = __shfl_xor_sync(0xffffffffu, m2, o);
      m1 = nan_max(m1, a1);
      m2 = nan_max(m2, a2);
    }
    double inv[2], fs[2];
    const double mm[2] = {m1, m2};
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const bool bad = !(mm[r] <= 1.7e308);
      int ex = 0;
      if (!bad && mm[r] > 0.0) frexp(mm[r], &ex);
      inv[r] = bad ? 0.0 : ldexp(1.0, -(ex + 1));
      fs[r] = bad ? __longlong_as_double(0x7ff8000000000000ll) : ldexp(1.0, ex + 1);
    }
    for (int c = lane; c < o4; c += 32) {
      double v1, v2;
      value(c, v1, v2);
      double t1 = v1 * inv[0], t2 = v2 * inv[1];
#pragma unroll
      for (int s = 0; s < 4; ++s) {
        t1 *= 128.0; t2 *= 128.0;
        const double r1 = rint(t1), r2 = rint(t2);
        t1 -= r1; t2 -= r2;
        dst[((long long)s * rows_pad + 2 * b) * ldb + c] = (int8_t)(int)r1;
        dst[((long long)s * rows_pad + 2 * b + 1) * ldb + c] = (int8_t)(int)r2;
      }
    }
    if (lane == 0) {
      fscale[2 * b] = fs[0]; fscale[2 * b + 1] = fs[1];
      amax[2 * b] = (float)m1 * 1.0000002f; amax[2 * b + 1] = (float)m2 * 1.0000002f;
    }
  }
}

int oz_pack_network_input(OzRows* r, long long B, const double* x, const double* uprev, const double* xs, const double* us,
                          const double* xscale, int nx, int nu, int with_uprev, float* amax, cudaStream_t st) {
  if (B <= 0) return 0;
  if (r->ns != 4 || 2 * B > r->cap_pad) return set_error(NNMPC_ERR_BADARG, "oz_pack_network_input: planes not prepared");
  k_oz_pack_network_input<<<row_grid((B + 7) / 8), 256, 0, st>>>(x, uprev, xs, us, xscale, r->S.p, r->cap_pad, r->ldb, r->fscale.p,
                                                                 amax, B, nx, nu, with_uprev);
  count_launch();
  NNMPC_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace nnmpc

using namespace nnmpc;

extern "C" {

// Self test of the INT8-sliced path:  C[M x N] = A[M x K] * Bt[N x K]^T, all FP64 device matrices (row-major, dense).
int nnmpc_oz_gemm_test(int M, int N, int K, const double* A, const double* Bt, double* C, void* stream) {
  if (!A || !Bt || !C || M <= 0 || N <= 0 || K <= 0) return set_error(NNMPC_ERR_BADARG, "nnmpc_oz_gemm_test: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  int dev = 0;
  NNMPC_CUDA(cudaGetDevice(&dev));
  OzOperator op;
  OzRows rows;
  int rc = oz_slice_operator(Bt, N, K, &op, st);
  if (rc == 0) rc = oz_rows_ensure(&rows, M, K, st);
  if (rc == 0) rc = oz_slice_rows(&rows, nullptr, nullptr, M, A, K, st);
  if (rc == 0) rc = oz_apply<OZ_LMAX, OzEpiStore>(&op, &rows, M, nullptr, OzEpiStore::Params{C, N}, dev, st);
  if (rc == 0 && cudaStreamSynchronize(st) != cudaSuccess)
    rc = set_error(NNMPC_ERR_CUDA, "oz_gemm failed: %s", cudaGetErrorString(cudaGetLastError()));
  cudaStreamSynchronize(st);
  op.release();
  rows.release();
  return rc;
}

// Self test of the exact anchors and KKT checks as the closed-loop engine calls them (include/nnmpc.h).  Like the
// engine, it slices the operator and sizes the sample planes for max_rows rows; the row list and its device-side
// length go to the kernels unchanged.
int nnmpc_exact_apply_test(int kind, int pipe, int variant, int B, int n, int nu, const double* Op, const int* rows,
                           const int* count, int max_rows, const double* A, const double* C, const double* lb,
                           const double* ub, double* X, unsigned long long* kres, void* stream) {
  if (kind < 0 || kind > 2 || pipe < 0 || pipe > 1 || variant < -1 || variant > 3 || B <= 0 || n <= 0 || (n & 1) ||
      max_rows <= 0 || (!rows && max_rows > B) || !Op || !A || !count || (kind != 2 && !C) || (kind != 1 && !X) ||
      (kind == 1 && (nu <= 0 || !lb || !ub || !kres)))
    return set_error(NNMPC_ERR_BADARG, "nnmpc_exact_apply_test: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  int dev = 0;
  NNMPC_CUDA(cudaGetDevice(&dev));
  int rc = 0;
  OzOperator op;
  OzRows r;
  DevBuf<double> zero;
  if (pipe == 0) {
    GemmOperands g{};
    g.A = A; g.lda = n; g.Bt = Op; g.ldb = n; g.M = max_rows; g.N = n; g.K = n; g.rows = rows; g.m_count = count;
    if (kind == 0) rc = lp_anchor_gemm(rows, count, max_rows, A, Op, C, X, n, st);
    else if (kind == 1) rc = gemm_by_count<EpiVerifyMax>(g, EpiVerifyMax::Params{A, C, lb, ub, kres, n, nu, X}, st);
    else rc = gemm_by_count<EpiStore>(g, EpiStore::Params{X, n, nullptr, 0}, st);
  } else {
    rc = oz_slice_operator(Op, n, n, &op, st);
    if (rc == 0) rc = oz_rows_ensure(&r, max_rows, n, st);
    if (rc == 0 && kind == 0) rc = oz_anchor(&op, &r, rows, count, max_rows, A, C, X, n, dev, st, variant);
    if (rc == 0 && kind == 1) rc = oz_verify(&op, &r, rows, count, max_rows, A, C, lb, ub, kres, X, n, nu, dev, st, variant);
    if (rc == 0 && kind == 2) {
      // all 8 levels through the anchor functor with c = 0: it scatters to the listed rows as the check does
      rc = zero.ensure((size_t)B * n);
      if (rc == 0 && cudaMemsetAsync(zero.p, 0, (size_t)B * n * sizeof(double), st) != cudaSuccess)
        rc = set_error(NNMPC_ERR_CUDA, "nnmpc_exact_apply_test: memset failed");
      if (rc == 0) rc = oz_slice_rows(&r, rows, count, max_rows, A, n, st);
      if (rc == 0)
        rc = oz_apply<OZ_LMAX, OzEpiAnchor>(&op, &r, max_rows, count, OzEpiAnchor::Params{X, zero.p, rows, n}, dev, st,
                                            variant);
    }
  }
  if (rc == 0 && cudaStreamSynchronize(st) != cudaSuccess)
    rc = set_error(NNMPC_ERR_CUDA, "exact apply failed: %s", cudaGetErrorString(cudaGetLastError()));
  cudaStreamSynchronize(st);
  op.release();
  r.release();
  zero.release();
  return rc;
}

// Probe (tools/probes/oz_rates.py, not on the product path): time `reps` applies over already sliced operands.
// ms[0] = sample slicing kernel, ms[1] = GEMM launches (the variant NNMPC_OZ_VARIANT selects), both per apply.
int nnmpc_oz_gemm_bench(int M, int N, int K, const double* A, const double* Bt, double* C, int reps, float* ms) {
  if (!A || !Bt || !C || !ms || M <= 0 || N <= 0 || K <= 0 || reps <= 0)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_oz_gemm_bench: bad argument");
  cudaStream_t st = 0;
  int dev = 0;
  NNMPC_CUDA(cudaGetDevice(&dev));
  OzOperator op;
  OzRows rows;
  int rc = oz_slice_operator(Bt, N, K, &op, st);
  if (rc == 0) rc = oz_rows_ensure(&rows, M, K, st);
  cudaEvent_t e0, e1, e2;
  cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventCreate(&e2);
  for (int w = 0; w < 2 && rc == 0; ++w) {
    rc = oz_slice_rows(&rows, nullptr, nullptr, M, A, K, st);
    if (rc == 0) rc = oz_apply<OZ_LMAX, OzEpiStore>(&op, &rows, M, nullptr, OzEpiStore::Params{C, N}, dev, st);
  }
  if (rc == 0) {
    cudaEventRecord(e0, st);
    for (int i = 0; i < reps && rc == 0; ++i) rc = oz_slice_rows(&rows, nullptr, nullptr, M, A, K, st);
    cudaEventRecord(e1, st);
    for (int i = 0; i < reps && rc == 0; ++i)
      rc = oz_apply<OZ_LMAX, OzEpiStore>(&op, &rows, M, nullptr, OzEpiStore::Params{C, N}, dev, st);
    cudaEventRecord(e2, st);
    if (cudaEventSynchronize(e2) != cudaSuccess) rc = set_error(NNMPC_ERR_CUDA, "oz bench failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (rc == 0) {
      cudaEventElapsedTime(&ms[0], e0, e1);
      cudaEventElapsedTime(&ms[1], e1, e2);
      ms[0] /= reps; ms[1] /= reps;
    }
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(e2);
  cudaStreamSynchronize(st);
  op.release();
  rows.release();
  return rc;
}

}  // extern "C"
