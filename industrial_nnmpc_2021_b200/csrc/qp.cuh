// Internal interface of the batched regulator-QP solver (shared by qp.cu, sim.cu and mlp.cu).
#pragma once
#include <cuda.h>        // CUtensorMap (type only)
#include <cuda_fp16.h>
#include "nnmpc_common.cuh"
#include "gemm_f64.cuh"
#include "oz.cuh"

namespace nnmpc {

// CTA tiles of the FP64 tensor-core GEMM.  Every shape accumulates each output element over k in
// the same order (sequential DMMA.8x8x4 steps, no split-K), so results are bitwise independent of
// the tile shape a sample happens to be computed with.
// Shapes and row-count windows were ranked on a B200 with tools/probes/gemm_tiles.py (n = 4480):
//   rows <= 48: 16x32 (280 CTAs stream the operator once; 83 us at 40 rows)   <= 512: 32x64 (23 TF/s)
//   <= 896: 64x64 (24.6 TF/s at 600 rows, 128x128 would run 17.9)              above: 128x128 (30-32 TF/s)
using TileBig = GemmTile<128, 128, 2, 4, 4>;
using TileMid = GemmTile<64, 64, 2, 2, 4>;
using TileSmall = GemmTile<32, 64, 2, 2, 6>;
using TileSkinny = GemmTile<16, 32, 1, 4, 8>;
constexpr int SKINNY_MAX_ROWS = 48;
constexpr int SMALL_MAX_ROWS = 512;
constexpr int MID_MAX_ROWS = 896;
inline bool use_big_tile(long long M, int N) { return M > 64 && N > 64; }

__device__ __forceinline__ double clipd(double v, double lo, double hi) { return fmin(fmax(v, lo), hi); }

// plain store epilogue: C = acc (+bias) (ReLU)
struct EpiStore {
  struct Params {
    double* C;
    long long ldc;
    const double* bias;  // nullable, per column
    int relu;
  };
  Params p;
  __device__ EpiStore(const Params& p_, int, int) : p(p_) {}
  __device__ void begin_row() {}
  __device__ void apply(int pr, int, int col, double v0, double v1, bool ok0, bool ok1) {
    if (p.bias) {
      if (ok0) v0 += p.bias[col];
      if (ok1) v1 += p.bias[col + 1];
    }
    if (p.relu) {
      v0 = relu_keep_nan(v0);
      v1 = relu_keep_nan(v1);
    }
    double* c = p.C + (long long)pr * p.ldc + col;
    if (ok1 && ((reinterpret_cast<uintptr_t>(c) & 15) == 0)) {
      *reinterpret_cast<double2*>(c) = make_double2(v0, v1);
    } else {
      if (ok0) c[0] = v0;
      if (ok1) c[1] = v1;
    }
  }
  __device__ void finish_row(int, int, int, bool) {}
};

// Douglas-Rachford update fused on the accumulators of  acc = Top w :
//   x = acc - c ;  d = x - clip(v) ;  v+ = v + alpha d ;  w+ = 2 clip(v+) - v+
// writes v (in place), the next GEMM operand w+, optionally z+ = clip(v+), and (dres != null)
// folds ||d||_inf of the row into dres[row] (bit pattern of a non-negative double, atomicMax):
// KKT(clip(v)) <= ||P + D||_inf ||d||_inf, the cheap convergence trigger of the closed-loop engine.
struct EpiAdmm {
  struct Params {
    double* V;
    const double* C;
    double* Wn;
    double* Z;  // written when write_z
    const double* lb;
    const double* ub;  // B x nu
    int n, nu;
    double alpha;
    int write_z;
    unsigned long long* dres;  // nullable, one per physical row
    const int* state;          // nullable: a row takes part iff state[row] == iter_state (closed-loop engine tail)
    int iter_state;
  };
  Params p;
  double dmax;
  __device__ EpiAdmm(const Params& p_, int, int) : p(p_), dmax(0.0) {}
  __device__ void begin_row() { dmax = 0.0; }
  __device__ void apply(int pr, int, int col, double a0, double a1, bool ok0, bool ok1) {
    if (!ok0) return;
    if (p.state && p.state[pr] != p.iter_state) return;
    const long long off = (long long)pr * p.n + col;
    const double* lbr = p.lb + (long long)pr * p.nu;
    const double* ubr = p.ub + (long long)pr * p.nu;
    const int k0 = col % p.nu;
    const int k1 = (k0 + 1 == p.nu) ? 0 : k0 + 1;
    if (ok1) {
      double2 v = *reinterpret_cast<const double2*>(p.V + off);
      double2 c = *reinterpret_cast<const double2*>(p.C + off);
      double l0 = lbr[k0], u0 = ubr[k0], l1 = lbr[k1], u1 = ubr[k1];
      double d0 = (a0 - c.x) - clipd(v.x, l0, u0);
      double d1 = (a1 - c.y) - clipd(v.y, l1, u1);
      double vn0 = v.x + p.alpha * d0;
      double vn1 = v.y + p.alpha * d1;
      double z0 = clipd(vn0, l0, u0), z1 = clipd(vn1, l1, u1);
      *reinterpret_cast<double2*>(p.V + off) = make_double2(vn0, vn1);
      *reinterpret_cast<double2*>(p.Wn + off) = make_double2(2.0 * z0 - vn0, 2.0 * z1 - vn1);
      if (p.write_z) *reinterpret_cast<double2*>(p.Z + off) = make_double2(z0, z1);
      dmax = fmax(dmax, fmax(fabs(d0), fabs(d1)));
    } else {
      double v = p.V[off], c = p.C[off], l0 = lbr[k0], u0 = ubr[k0];
      double d0 = (a0 - c) - clipd(v, l0, u0);
      double vn = v + p.alpha * d0;
      double z = clipd(vn, l0, u0);
      p.V[off] = vn;
      p.Wn[off] = 2.0 * z - vn;
      if (p.write_z) p.Z[off] = z;
      dmax = fmax(dmax, fabs(d0));
    }
  }
  __device__ void finish_row(int pr, int, int, bool rok) {
    if (!p.dres) return;
    if (p.state && rok && p.state[pr] != p.iter_state) rok = false;
    double m = dmax;
    m = fmax(m, __shfl_xor_sync(0xffffffffu, m, 1));
    m = fmax(m, __shfl_xor_sync(0xffffffffu, m, 2));
    // NaN/Inf (diverged or corrupted sample) must not look converged: map to +Inf
    if (!(m <= 1.7e308)) m = __longlong_as_double(0x7ff0000000000000ll);
    if (rok && (threadIdx.x & 3) == 0) atomicMax(p.dres + pr, (unsigned long long)__double_as_longlong(m));
  }
};

// acc = (P z) ; g = acc + q ; per-row partial KKT residual (max) and cost (sum)
struct EpiVerify {
  struct Params {
    const double* Z;
    const double* Ql;
    const double* lb;
    const double* ub;
    double* part_max;
    double* part_sum;
    int n, nu, nslots;
  };
  Params p;
  double rmax, rsum;
  __device__ EpiVerify(const Params& p_, int, int) : p(p_), rmax(0.0), rsum(0.0) {}
  __device__ void begin_row() { rmax = 0.0; rsum = 0.0; }
  __device__ void one(int pr, int col, double a) {
    const long long off = (long long)pr * p.n + col;
    const int k = col % p.nu;
    double z = p.Z[off], q = p.Ql[off];
    double l = p.lb[(long long)pr * p.nu + k], u = p.ub[(long long)pr * p.nu + k];
    double g = a + q;
    double r = fabs(z - clipd(z - g, l, u));
    if (!(r <= 1.7e308)) r = __longlong_as_double(0x7ff0000000000000ll);
    rmax = fmax(rmax, r);
    rsum += z * (0.5 * a + q);
  }
  __device__ void apply(int pr, int, int col, double a0, double a1, bool ok0, bool ok1) {
    if (ok0) one(pr, col, a0);
    if (ok1) one(pr, col + 1, a1);
  }
  __device__ void finish_row(int, int lr, int slot, bool rok) {
    // the 4 lanes of a fragment row hold disjoint column pairs: fixed-order butterfly
    double m = rmax, s = rsum;
    m = fmax(m, __shfl_xor_sync(0xffffffffu, m, 1));
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    m = fmax(m, __shfl_xor_sync(0xffffffffu, m, 2));
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    if (rok && (threadIdx.x & 3) == 0) {
      p.part_max[(long long)lr * p.nslots + slot] = m;
      p.part_sum[(long long)lr * p.nslots + slot] = s;
    }
  }
};

// acc = P z ; g = acc + q ; exact KKT residual ||z - clip(z - g)||_inf folded per row with atomicMax
struct EpiVerifyMax {
  struct Params {
    const double* Z;
    const double* Ql;
    const double* lb;
    const double* ub;
    unsigned long long* kres;
    int n, nu;
    double* G;   // nullable: the exact gradient g = P z + q per element (mixed mode re-anchors x from it)
  };
  Params p;
  double rmax;
  __device__ EpiVerifyMax(const Params& p_, int, int) : p(p_), rmax(0.0) {}
  __device__ void begin_row() { rmax = 0.0; }
  __device__ void one(int pr, int col, double a) {
    const long long off = (long long)pr * p.n + col;
    const int k = col % p.nu;
    const double z = p.Z[off], g = a + p.Ql[off];
    if (p.G) p.G[off] = g;
    double r = fabs(z - clipd(z - g, p.lb[(long long)pr * p.nu + k], p.ub[(long long)pr * p.nu + k]));
    // NaN/Inf must not look converged (an infinite g clips to a bound and leaves r finite)
    if (!(r <= 1.7e308 && fabs(g) <= 1.7e308)) r = __longlong_as_double(0x7ff0000000000000ll);
    rmax = fmax(rmax, r);
  }
  __device__ void apply(int pr, int, int col, double a0, double a1, bool ok0, bool ok1) {
    if (ok0) one(pr, col, a0);
    if (ok1) one(pr, col + 1, a1);
  }
  __device__ void finish_row(int pr, int, int, bool rok) {
    double m = rmax;
    m = fmax(m, __shfl_xor_sync(0xffffffffu, m, 1));
    m = fmax(m, __shfl_xor_sync(0xffffffffu, m, 2));
    if (rok && (threadIdx.x & 3) == 0) atomicMax(p.kres + pr, (unsigned long long)__double_as_longlong(m));
  }
};

template <class Epi>
inline int gemm_auto(const GemmOperands& g, const typename Epi::Params& ep, cudaStream_t st) {
  cudaError_t e = use_big_tile(g.M, g.N) ? launch_gemm<TileBig, Epi>(g, ep, st)
                                         : launch_gemm<TileMid, Epi>(g, ep, st);
  count_launch();
  if (e != cudaSuccess) return set_error(NNMPC_ERR_CUDA, "gemm launch failed: %s", cudaGetErrorString(e));
  return 0;
}
inline int row_slots_auto(long long M, int N) {
  return use_big_tile(M, N) ? gemm_row_slots<TileBig>(N) : gemm_row_slots<TileMid>(N);
}

// Row list whose length lives on the device (g.m_count, at most g.M rows): enqueue one launch per
// tile shape, each guarded by its row-count window; exactly one of them does the work.
template <class Epi>
inline int gemm_by_count(GemmOperands g, const typename Epi::Params& ep, cudaStream_t st) {
  const int Mmax = g.M;
  cudaError_t e = cudaSuccess;
  g.m_lo = 0; g.m_hi = SKINNY_MAX_ROWS; g.M = Mmax < SKINNY_MAX_ROWS ? Mmax : SKINNY_MAX_ROWS;
  e = launch_gemm<TileSkinny, Epi>(g, ep, st);
  count_launch();
  if (e == cudaSuccess && Mmax > SKINNY_MAX_ROWS) {
    g.m_lo = SKINNY_MAX_ROWS; g.m_hi = SMALL_MAX_ROWS; g.M = Mmax < SMALL_MAX_ROWS ? Mmax : SMALL_MAX_ROWS;
    e = launch_gemm<TileSmall, Epi>(g, ep, st);
    count_launch();
  }
  if (e == cudaSuccess && Mmax > SMALL_MAX_ROWS) {
    g.m_lo = SMALL_MAX_ROWS; g.m_hi = MID_MAX_ROWS; g.M = Mmax < MID_MAX_ROWS ? Mmax : MID_MAX_ROWS;
    e = launch_gemm<TileMid, Epi>(g, ep, st);
    count_launch();
  }
  if (e == cudaSuccess && Mmax > MID_MAX_ROWS) {
    g.m_lo = MID_MAX_ROWS; g.m_hi = 0x7fffffff; g.M = Mmax;
    e = launch_gemm<TileBig, Epi>(g, ep, st);
    count_launch();
  }
  if (e != cudaSuccess) return set_error(NNMPC_ERR_CUDA, "gemm launch failed: %s", cudaGetErrorString(e));
  return 0;
}

struct QpOutputs {
  double* cost;      // nullable
  double* kkt;       // nullable
  int* iters;        // nullable
  long long stride;  // element stride between samples in the three arrays
};

int qp_solve_device(nnmpc_qp* h, int B, const double* x0, const double* lb, const double* ub, double* u,
                    double* v_state, int warm, QpOutputs out, double tol, int max_iter, cudaStream_t st,
                    long long* iter_sum_out);
// the interior-point solver of a handle made by nnmpc_qp_create_ipm (ipm.cu); qp_solve_device dispatches to it
int ipm_solve_device(nnmpc_qp* h, int B, const double* x0, const double* lb, const double* ub, double* u,
                     QpOutputs out, double tol, int max_iter, cudaStream_t st, long long* iter_sum_out);

// live timing of the iteration GEMM (bench.py roofline); spans are recorded only while enabled
// channel 0: the iteration passes (FP64 DMMA GEMM, or the tcgen05 pass in mixed mode);
// channel 1: the FP64 anchor / exact-check GEMMs of the mixed mode
struct ProfSpan { cudaEvent_t a, b; double flops; long long launches; int chan; };
bool prof_begin(ProfSpan* sp, cudaStream_t st);
void prof_end(ProfSpan sp, cudaStream_t st, double flops, long long launches, int chan = 0);
// flops of spans whose row counts only the device knew at launch time (added once they are read back)
void prof_add_flops(double flops, int chan = 0);

// two-term fp16 split of a shared n x n operator, with the tensor maps the TMA producer reads it through
struct LpOperator {
  int n = 0;
  long long ldh = 0;       // leading dimension of T1/T2 (elements, multiple of 64)
  double scale = 1.0;      // T1 + T2 ~ scale * T
  DevBuf<__half> T1, T2;
  CUtensorMap tm1, tm2;
  bool ready = false;
  void release() { T1.release(); T2.release(); ready = false; }
};

}  // namespace nnmpc

struct nnmpc_qp {
  int n, nxa, nu, N, device;
  double alpha;
  double p_norm_inf;                  // ||P||_inf (max absolute row sum), scale of the convergence trigger
  double *P, *Top, *tq, *Mtq, *Kunc;  // device operators
  double top_max;                     // max |Top|
  double* rinv = nullptr;             // device n: 1 / rho (nnmpc_qp_set_penalty), null until set
  nnmpc::LpOperator lpop;             // fp16 split of Top, built on first use by the mixed-precision iteration
  nnmpc::OzOperator ozP, ozTop;       // INT8 digit planes of P and Top (FP64-accurate tensor-core applies), built on first use
  // scratch, sized for `cap` samples
  long long cap;
  int nslots_cap;
  nnmpc::DevBuf<double> V, W0, W1, C, Ql, part_max, part_sum;
  nnmpc::DevBuf<int> rows0, rows1;
  int* counts;                    // device: [0]=count A, [1]=count B, [2]=hit-maxiter flag
  unsigned long long* iter_sum;   // device accumulator of per-sample iterations
  int* h_pinned;                  // pinned host mirror (4 ints + 1 u64)
  // host-buffer staging for *_host entry points
  nnmpc::DevBuf<double> hx0, hlb, hub, hu, hcost, hkkt;
  nnmpc::DevBuf<int> hiters;
  // nnmpc_qp_create_ipm: stagewise v-space operators of the interior-point solver (ipm.cu) instead of P, Top, ...
  int ipm = 0;
  double *iA = nullptr, *iB = nullptr, *iQ = nullptr, *iR = nullptr, *iM = nullptr, *iPf = nullptr, *iK = nullptr;
  double *iAo = nullptr, *iQo = nullptr, *iMo = nullptr;   // the stage in the original inputs (Newton-step factorisation)
  nnmpc::DevBuf<double> ipm_scr;      // per-CTA Riccati factors and iterates
};
