// Batched steady-state target selector, one warp per sample.
//
// Replaces TargetSelector.solve (/root/reference/lib/linearMPC.py:298-311), which calls cvxopt on
//     min_(xs,us) 1/2|us-usp|^2_Rs + 1/2|C xs + Cd d - ysp|^2_Qs
//     s.t. (I-A) xs - B us = Bd d ,  ulb <= us <= uub                 (:182-187, H empty)
// With I - A invertible the equality eliminates xs = Gx us + Gd d and leaves an nu-dimensional
// strictly convex box QP,  min 1/2 us'Ht us + f'us,  f = Fy ysp + Fd d + f0  (operators built on
// the host, see linearMPC.TargetSelector).  nu <= 32, so lane i of a warp owns variable i and the
// QP is solved EXACTLY by a primal active-set method: equality-constrained solves through a
// Cholesky factorisation of the masked Hessian held in shared memory, ratio test with warp
// reductions, multiplier sign check.  (The CDU tuning makes Ht ill-conditioned - Rs = 1e-6 I,
// cdu_parameters.py:94 - so a first-order method is not an option here.)
#include "ts.cuh"

namespace nnmpc {

constexpr int TS_WARPS = 4;
constexpr int TS_LD = 33;
#define FULLMASK 0xffffffffu

struct TsParams {
  int B, nx, nu, ny, nd;
  const double *Ht, *Fy, *Fd, *f0, *Gx, *Gd, *ulb, *uub;
  const double* ysp; long long ysp_stride;
  const double* d;   long long d_stride;
  double* xs; long long xs_stride;
  double* us; long long us_stride;
  int* iters; long long iters_stride;
  int fused;
  TsFused f;
  int indexed;
  TsIndex ix;
  int* fail;   // nullable device flag, set when a solve stalls at the iteration cap or produces non-finite targets
  // 1: us (and iters) were written by k_ts_general; this kernel only forms xs and the fused outputs
  // 2: xs was written too (reduced targets); this kernel only forms the fused outputs
  int given;
  // k_ts_general (see nnmpc_ts in ts.cuh)
  int nw, mb, nR, rld, rny, reduced;
  const double *Hinv, *Abar, *AH, *Mbar, *R, *lo0, *hi0, *Kx, *Ku, *Zx, *Zu;
};

__device__ __forceinline__ double warp_min_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(FULLMASK, v, o));
  return v;
}
__device__ __forceinline__ double warp_max_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(FULLMASK, v, o));
  return v;
}

__global__ void __launch_bounds__(TS_WARPS * 32) k_target_selector(TsParams p) {
  __shared__ double Hs[32 * TS_LD];
  __shared__ double Sw[TS_WARPS][32 * TS_LD];
  __shared__ double uw[TS_WARPS][32];
  const int nu = p.nu, nx = p.nx, ny = p.ny, nd = p.nd;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (!p.given)
    for (int i = threadIdx.x; i < nu * nu; i += blockDim.x) Hs[(i / nu) * TS_LD + (i % nu)] = p.Ht[i];
  __syncthreads();
  double* S = Sw[warp];
  double* uvec = uw[warp];
  const bool act = lane < nu;
  const double lo = act ? p.ulb[lane] : 0.0;
  const double hi = act ? p.uub[lane] : 0.0;
  const int maxit = 10 * nu + 20;

  const int Bn = p.indexed && p.ix.count ? min(*p.ix.count, p.B) : p.B;
  for (int lb_ = blockIdx.x * TS_WARPS + warp; lb_ < Bn; lb_ += gridDim.x * TS_WARPS) {
    // s: per-slot buffers; b: position in the strided sample arrays
    const long long s = p.indexed ? (long long)p.ix.rows[lb_] : (long long)lb_;
    const long long b = p.indexed ? (p.ix.chunk ? (long long)p.ix.chunk[s] : s) * p.ix.T + p.ix.tcur[s] : s;
    const double* ysp = p.ysp + b * p.ysp_stride;
    const double* dd = p.d + b * p.d_stride;
    // Set-points and disturbances are piecewise constant (sample_prbs_like holds each level for
    // hundreds of steps, controller_evaluation.py:31-47): when this step's (ysp, d) equal the previous
    // step's bit for bit, the target is the previous one - the solve is deterministic - so reuse it.
    bool same = false;
    if (!p.given && p.indexed && p.ix.tcur[s] > 0) {
      bool eq = true;
      const double* yprev = ysp - p.ysp_stride;
      const double* dprev = dd - p.d_stride;
      for (int y = lane; y < ny; y += 32) eq = eq && (ysp[y] == yprev[y]);
      for (int k = lane; k < nd; k += 32) eq = eq && (dd[k] == dprev[k]);
      same = __all_sync(FULLMASK, eq);
    }
    double f = 0.0;
    if (act && !same && !p.given) {      // (with given targets Fy / Fd / f0 may be k_ts_general's nw-row operators)
      f = p.f0[lane];
      const double* fy = p.Fy + (long long)lane * ny;
      for (int y = 0; y < ny; ++y) f += fy[y] * ysp[y];
      const double* fd = p.Fd + (long long)lane * nd;
      for (int k = 0; k < nd; ++k) f += fd[k] * dd[k];
    }
    // Start: the projection of the origin.  (Starting inside a trajectory from the previous step's target was measured
    // and dropped: with the CDU tuning the targets sit in corners of the input box, and leaving a corner one
    // multiplier at a time takes twice as long as reaching the next one from the interior.)
    double u = act ? fmin(fmax(0.0, lo), hi) : 0.0;
    int st = 2;  // 0 free, -1 at lower, +1 at upper, 2 padding lane / degenerate (never released)
    if (act) st = (hi <= lo) ? 2 : (u <= lo ? -1 : (u >= hi ? 1 : 0));
    int it = 0;
    bool done = same || p.given;
    if (same && act) u = p.us[(b - 1) * p.us_stride + lane];
    if (p.given && act) u = p.us[b * p.us_stride + lane];
    for (; it < maxit && !done; ++it) {
      uvec[lane] = u;
      __syncwarp();
      const unsigned fixedmask = __ballot_sync(FULLMASK, st != 0);
      double rhs;
      if (act) {
        if (st != 0) {
          rhs = u;
          for (int j = 0; j <= lane; ++j) S[lane * TS_LD + j] = (j == lane) ? 1.0 : 0.0;
        } else {
          rhs = -f;
          for (int j = 0; j < nu; ++j) {
            const double hij = Hs[lane * TS_LD + j];
            const bool jfixed = (fixedmask >> j) & 1u;
            if (jfixed) rhs -= hij * uvec[j];
            if (j <= lane) S[lane * TS_LD + j] = jfixed ? 0.0 : hij;
          }
        }
      } else {
        rhs = 0.0;
      }
      __syncwarp();
      // in-place lower Cholesky of the masked (block-diagonal SPD) matrix
      for (int k = 0; k < nu; ++k) {
        const double sd = sqrt(S[k * TS_LD + k]);
        const double inv = 1.0 / sd;
        double lik = 0.0;
        if (lane > k && act) {
          lik = S[lane * TS_LD + k] * inv;
          S[lane * TS_LD + k] = lik;
        }
        __syncwarp();
        if (lane == k) S[k * TS_LD + k] = sd;
        for (int j = k + 1; j < nu; ++j) {
          const double ljk = S[j * TS_LD + k];
          if (lane >= j && act) S[lane * TS_LD + j] -= lik * ljk;
        }
        __syncwarp();
      }
      double bb = rhs;
      for (int k = 0; k < nu; ++k) {  // L y = rhs
        const double yk = __shfl_sync(FULLMASK, bb, k) / S[k * TS_LD + k];
        if (lane == k) bb = yk;
        else if (lane > k && act) bb -= S[lane * TS_LD + k] * yk;
      }
      for (int k = nu - 1; k >= 0; --k) {  // L' x = y
        const double xk = __shfl_sync(FULLMASK, bb, k) / S[k * TS_LD + k];
        if (lane == k) bb = xk;
        else if (lane < k) bb -= S[k * TS_LD + lane] * xk;
      }
      const double uh = (st == 0) ? bb : u;
      double a = 2.0;
      if (st == 0) {
        if (uh > hi) a = (hi - u) / (uh - u);
        else if (uh < lo) a = (lo - u) / (uh - u);
      }
      double amin = warp_min_d(a);
      if (amin >= 1.0) {
        // full step: u is the minimiser on the current face; check multiplier signs
        u = uh;
        __syncwarp();
        uvec[lane] = u;
        __syncwarp();
        double g = f, scale = fabs(f);
        if (act) {
          for (int j = 0; j < nu; ++j) {
            const double t = Hs[lane * TS_LD + j] * uvec[j];
            g += t;
            scale += fabs(t);
          }
        }
        double viol = 0.0;
        if (st == 1) viol = g;         // upper bound active needs g <= 0
        else if (st == -1) viol = -g;  // lower bound active needs g >= 0
        if (!(viol > 1.5e-14 * scale)) viol = 0.0;
        const double vmax = warp_max_d(viol);
        if (vmax <= 0.0) {
          done = true;
        } else {
          const unsigned who = __ballot_sync(FULLMASK, viol == vmax);
          if (lane == __ffs(who) - 1) st = 0;
        }
      } else {
        if (amin < 0.0) amin = 0.0;
        const unsigned who = __ballot_sync(FULLMASK, a <= amin);
        const int blk = __ffs(who) - 1;
        if (st == 0) u += amin * (uh - u);
        if (lane == blk) {
          if (uh > hi) { u = hi; st = 1; }
          else { u = lo; st = -1; }
        }
      }
      __syncwarp();
    }
    uvec[lane] = u;
    __syncwarp();
    // The reference's cvxopt call would report a status (linearMPC.py:304-306 ignores it); here a solve that ran
    // out of active-set steps or went non-finite (NaN pivot of the masked Cholesky, NaN/Inf inputs) raises the
    // flag the callers turn into NNMPC_WARN_TARGET, and its iteration count is written negated.
    const bool bad = !done || __any_sync(FULLMASK, act && !(fabs(u) <= 1.7e308));
    if (bad && p.fail && lane == 0) atomicExch(p.fail, 1);
    if (act) p.us[(long long)b * p.us_stride + lane] = u;
    if (p.iters && lane == 0 && !p.given) p.iters[(long long)b * p.iters_stride] = bad ? -it - 1 : it;
    const TsFused& F = p.f;
    for (int r = lane; r < nx; r += 32) {
      double acc = 0.0;
      if (p.given == 2) {
        acc = p.xs[(long long)b * p.xs_stride + r];
      } else {
        const double* gx = p.Gx + (long long)r * nu;
        for (int j = 0; j < nu; ++j) acc += gx[j] * uvec[j];
        const double* gd = p.Gd + (long long)r * nd;
        for (int k = 0; k < nd; ++k) acc += gd[k] * dd[k];
        p.xs[(long long)b * p.xs_stride + r] = acc;
      }
      if (p.fused) {
        const double xv = F.x[s * nx + r];
        F.x0[s * F.nxa_ld + r] = xv - acc;
        F.row_x[(long long)b * F.row_stride_x + r] = xv;
      }
    }
    if (p.fused) {
      if (act) {
        const double up = F.uprev[s * nu + lane];
        F.x0[s * F.nxa_ld + nx + lane] = up - u;
        F.row_uprev[(long long)b * F.row_stride_u + lane] = up;
        F.lb[s * nu + lane] = lo - u;
        F.ub[s * nu + lane] = hi - u;
        F.dus[s * nu + lane] = F.us_prev[s * nu + lane] - u;
        F.us_prev[s * nu + lane] = u;
      }
      for (int c = nx + nu + lane; c < F.nxa_ld; c += 32) F.x0[s * F.nxa_ld + c] = 0.0;
    }
    __syncwarp();
  }
}


// ---- output-constrained targets: ylb <= C xs + Cd d <= yub next to the input box (linearMPC.py:242-248, :284-288) ----
// After the elimination of xs the problem is  min 1/2 u'Ht u + f'u  s.t.  lo_i <= abar_i'u <= hi_i  over the mb = ny + nu
// rows abar = [C Gx; I], with lo/hi = [ylb - Ryd d; ulb], [yub - Ryd d; uub] per sample.  Solved EXACTLY by the dual
// active-set method of Goldfarb and Idnani in its range-space form, one warp per sample: start at the unconstrained
// minimiser, add the most violated constraint p, moving along z = Hinv a_p - Hinv A_W' r with r = (A_W Hinv A_W')^-1
// A_W Hinv a_p until p holds (full step) or a multiplier of the working set W reaches zero (that constraint is
// dropped).  Hinv, AH = Abar Hinv and Mbar = Abar Hinv Abar' are shared by all samples (host set-up), so a step costs
// one |W| x |W| Cholesky in shared memory (|W| <= nu <= 32) and a few gathers.  The final point is re-solved from its
// working set, so rounding does not accumulate over the steps.  An infeasible sample (no step length exists) or one
// that runs out of steps raises the fail flag and carries a negative iteration count - cvxopt would report a status.
//
// ---- reduced targets: H non-empty (H C xs = H (ysp - Cd d), linearMPC.py:254-267) or I - A singular ----
// xs cannot be eliminated through (I - A)^-1 there.  The host takes an orthonormal basis Z of null(tA) instead and
// writes [xs; us] = K s + Z v, s = [ysp; d], K = tA^+ tb, so the equalities hold for every v of the nw = nu - nz
// remaining dimensions.  The same kernel then solves over v: lane i owns v_i (i < nw), the mb = nu (+ ny) rows are
// [C Zx; Zu] with the per-sample offsets R s, R = [C Kx + [0 Cd]; Ku], and the warp reconstructs xs and us from the
// final v.  The output-bounded mode above is the case Z = [Gx; I], v = us.  nw = 0 leaves no freedom: the target is
// K s, returned when it satisfies the rows and flagged infeasible otherwise.
constexpr int TS_MAXC = 160;      // mb

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULLMASK, v, o);
  return v;
}

// Cholesky of the leading m x m block of S (lower, in place, lane j owns row j) and the solve S x = rhs (lane j: rhs_j);
// returns x_j in lane j.  A non-positive pivot yields NaN, which the caller turns into the fail flag.
__device__ __forceinline__ double ws_chol_solve(double* S, int m, double rhs, int lane) {
  for (int k = 0; k < m; ++k) {
    const double sd = sqrt(S[k * TS_LD + k]);
    const double inv = 1.0 / sd;
    double lik = 0.0;
    if (lane > k && lane < m) {
      lik = S[lane * TS_LD + k] * inv;
      S[lane * TS_LD + k] = lik;
    }
    __syncwarp();
    if (lane == k) S[k * TS_LD + k] = sd;
    for (int j = k + 1; j < m; ++j) {
      const double ljk = S[j * TS_LD + k];
      if (lane >= j && lane < m) S[lane * TS_LD + j] -= lik * ljk;
    }
    __syncwarp();
  }
  double bb = lane < m ? rhs : 0.0;
  for (int k = 0; k < m; ++k) {  // L y = rhs
    const double yk = __shfl_sync(FULLMASK, bb, k) / S[k * TS_LD + k];
    if (lane == k) bb = yk;
    else if (lane > k && lane < m) bb -= S[lane * TS_LD + k] * yk;
  }
  for (int k = m - 1; k >= 0; --k) {  // L' x = y
    const double xk = __shfl_sync(FULLMASK, bb, k) / S[k * TS_LD + k];
    if (lane == k) bb = xk;
    else if (lane < k) bb -= S[k * TS_LD + lane] * xk;
  }
  return bb;
}

__global__ void __launch_bounds__(TS_WARPS * 32) k_ts_general(TsParams p) {
  __shared__ double Sw[TS_WARPS][32 * TS_LD];
  __shared__ double uw[TS_WARPS][32], fw[TS_WARPS][32], lamw[TS_WARPS][32], rw[TS_WARPS][32];
  __shared__ double blo[TS_WARPS][TS_MAXC], bhi[TS_WARPS][TS_MAXC];
  __shared__ int widx[TS_WARPS][32], wsgn[TS_WARPS][32];
  const int nu = p.nu, nx = p.nx, ny = p.ny, nd = p.nd, mb = p.mb, nw = p.nw;
  const int row_u = mb - nu;      // first input row
  const int ns = ny + nd;         // columns of Kx / Ku
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* S = Sw[warp];
  double* uvec = uw[warp];
  double* fvec = fw[warp];
  double* lam = lamw[warp];
  double* rvec = rw[warp];
  double* lo = blo[warp];
  double* hi = bhi[warp];
  int* wi = widx[warp];
  int* ws = wsgn[warp];
  const bool act = lane < nw;
  const int maxit = 8 * (nu + 8) + 2 * row_u;
  const double INF = __longlong_as_double(0x7ff0000000000000ll);

  const int Bn = p.indexed && p.ix.count ? min(*p.ix.count, p.B) : p.B;
  for (int lb_ = blockIdx.x * TS_WARPS + warp; lb_ < Bn; lb_ += gridDim.x * TS_WARPS) {
    const long long s = p.indexed ? (long long)p.ix.rows[lb_] : (long long)lb_;
    const long long b = p.indexed ? (p.ix.chunk ? (long long)p.ix.chunk[s] : s) * p.ix.T + p.ix.tcur[s] : s;
    const double* ysp = p.ysp + b * p.ysp_stride;
    const double* dd = p.d + b * p.d_stride;
    // linear term and per-sample bounds
    double f = 0.0;
    if (act) {
      f = p.f0[lane];
      const double* fy = p.Fy + (long long)lane * ny;
      for (int y = 0; y < ny; ++y) f += fy[y] * ysp[y];
      const double* fd = p.Fd + (long long)lane * nd;
      for (int k = 0; k < nd; ++k) f += fd[k] * dd[k];
    }
    fvec[lane] = f;
    for (int i = lane; i < mb; i += 32) {
      if (i < p.nR) {
        double r = 0.0;
        const double* Ri = p.R + (long long)i * p.rld;
        for (int y = 0; y < p.rny; ++y) r += Ri[y] * ysp[y];
        for (int k = 0; k < nd; ++k) r += Ri[p.rny + k] * dd[k];
        lo[i] = p.lo0[i] - r;
        hi[i] = p.hi0[i] - r;
      } else {
        lo[i] = p.lo0[i];
        hi[i] = p.hi0[i];
      }
    }
    __syncwarp();
    // unconstrained minimiser
    double u = 0.0;
    if (act)
      for (int j = 0; j < nw; ++j) u -= p.Hinv[(long long)lane * nw + j] * fvec[j];
    int nW = 0, it = 0;
    bool done = false, failed = false;
    for (; it < maxit && !done && !failed; ++it) {
      uvec[lane] = u;
      __syncwarp();
      // most violated constraint (scaled tolerance)
      double best = 0.0;
      int bi = -1, bs = 0;
      for (int i = lane; i < mb; i += 32) {
        double val = 0.0, mag = 0.0;
        const double* a = p.Abar + (long long)i * nw;
        for (int k = 0; k < nw; ++k) {
          const double t = a[k] * uvec[k];
          val += t;
          mag += fabs(t);
        }
        const double vu = val - hi[i], vl = lo[i] - val;
        const double v = vu >= vl ? vu : vl;
        const double tol = 1e-11 * (1.0 + mag + fabs(vu >= vl ? hi[i] : lo[i]));
        if (v > tol && v > best) { best = v; bi = i; bs = vu >= vl ? 1 : -1; }
        if (!(v <= 1.7e308)) { best = INF; bi = i; bs = 1; }      // NaN / Inf: make it visible
      }
      const double vmax = warp_max_d(best);
      if (!(vmax > 0.0)) { done = true; break; }
      if (!(vmax <= 1.7e308)) { failed = true; break; }
      const unsigned who = __ballot_sync(FULLMASK, best == vmax && bi >= 0);
      const int src = __ffs(who) - 1;
      const int ip = __shfl_sync(FULLMASK, bi, src);
      const int sp = __shfl_sync(FULLMASK, bs, src);
      double vp = vmax;
      double lam_p = 0.0;
      const double mpp = p.Mbar[(long long)ip * mb + ip];
      for (int inner = 0; inner <= 2 * nw + 2; ++inner) {
        // d = A_W Hinv a_p, S = A_W Hinv A_W'
        double dj = 0.0;
        if (lane < nW) {
          const long long ij = wi[lane];
          dj = (double)(ws[lane] * sp) * p.Mbar[ij * mb + ip];
          for (int k = 0; k <= lane; ++k) S[lane * TS_LD + k] = (double)(ws[lane] * ws[k]) * p.Mbar[ij * mb + wi[k]];
        }
        __syncwarp();
        const double rj = nW > 0 ? ws_chol_solve(S, nW, dj, lane) : 0.0;
        rvec[lane] = lane < nW ? rj : 0.0;
        __syncwarp();
        // z = Hinv a_p - Hinv A_W' r  (lane k holds z_k),  a_p'z = Mbar[p][p] - d'r
        double z = 0.0;
        if (act) {
          z = (double)sp * p.AH[(long long)ip * nw + lane];
          for (int j = 0; j < nW; ++j) z -= rvec[j] * (double)ws[j] * p.AH[(long long)wi[j] * nw + lane];
        }
        const double apz = mpp - warp_sum_d(lane < nW ? dj * rj : 0.0);
        // step lengths
        double t1l = INF;
        if (lane < nW && rj > 1e-13 * (1.0 + fabs(dj))) t1l = lam[lane] / rj;
        const double t1 = warp_min_d(t1l);
        const double t2 = apz > 1e-12 * mpp ? vp / apz : INF;
        if (!(t1 <= 1.7e308) && !(t2 <= 1.7e308)) { failed = true; break; }      // infeasible (or NaN)
        const double t = t1 < t2 ? t1 : t2;
        u -= t * z;
        if (lane < nW) lam[lane] -= t * rj;
        lam_p += t;
        vp -= t * apz;
        __syncwarp();
        if (t2 <= t1) {      // full step: p joins the working set
          if (nW >= 32) { failed = true; break; }
          if (lane == 0) { wi[nW] = ip; ws[nW] = sp; lam[nW] = lam_p; }
          ++nW;
          __syncwarp();
          break;
        }
        // partial step: drop the blocking constraint, keep p for another try
        const unsigned blk = __ballot_sync(FULLMASK, t1l == t1);
        const int jb = __ffs(blk) - 1;
        const int wi_n = (lane >= jb && lane + 1 < nW) ? wi[lane + 1] : 0;
        const int ws_n = (lane >= jb && lane + 1 < nW) ? ws[lane + 1] : 0;
        const double lam_n = (lane >= jb && lane + 1 < nW) ? lam[lane + 1] : 0.0;
        __syncwarp();
        if (lane >= jb && lane + 1 < nW) { wi[lane] = wi_n; ws[lane] = ws_n; lam[lane] = lam_n; }
        --nW;
        __syncwarp();
        if (inner == 2 * nw + 2) failed = true;
      }
    }
    if (!done && !failed) failed = true;      // out of steps
    // re-solve on the final working set: lambda = -(A_W Hinv A_W')^-1 (b_W + A_W Hinv f), u = -Hinv f - Hinv A_W' lambda
    if (done && nW > 0) {
      double rhs = 0.0;
      if (lane < nW) {
        const long long ij = wi[lane];
        double ahf = 0.0;
        for (int k = 0; k < nw; ++k) ahf += p.AH[ij * nw + k] * fvec[k];
        const double bw = ws[lane] > 0 ? hi[ij] : -lo[ij];
        rhs = -(bw + (double)ws[lane] * ahf);
        for (int k = 0; k <= lane; ++k) S[lane * TS_LD + k] = (double)(ws[lane] * ws[k]) * p.Mbar[ij * mb + wi[k]];
      }
      __syncwarp();
      const double lj = ws_chol_solve(S, nW, rhs, lane);
      rvec[lane] = lane < nW ? lj : 0.0;
      __syncwarp();
      if (act) {
        double un = 0.0;
        for (int j = 0; j < nw; ++j) un -= p.Hinv[(long long)lane * nw + j] * fvec[j];
        for (int j = 0; j < nW; ++j) un -= rvec[j] * (double)ws[j] * p.AH[(long long)wi[j] * nw + lane];
        u = un;
      }
    }
    uvec[lane] = u;
    __syncwarp();
    bool xs_bad = false;
    if (p.reduced) {      // xs = Kx s + Zx v, us = Ku s + Zu v
      for (int r = lane; r < nx; r += 32) {
        double acc = 0.0;
        const double* kx = p.Kx + (long long)r * ns;
        for (int y = 0; y < ny; ++y) acc += kx[y] * ysp[y];
        for (int k = 0; k < nd; ++k) acc += kx[ny + k] * dd[k];
        const double* zx = p.Zx + (long long)r * nw;
        for (int j = 0; j < nw; ++j) acc += zx[j] * uvec[j];
        p.xs[(long long)b * p.xs_stride + r] = acc;
        xs_bad = xs_bad || !(fabs(acc) <= 1.7e308);
      }
      double un = 0.0;
      if (lane < nu) {
        const double* ku = p.Ku + (long long)lane * ns;
        for (int y = 0; y < ny; ++y) un += ku[y] * ysp[y];
        for (int k = 0; k < nd; ++k) un += ku[ny + k] * dd[k];
        const double* zu = p.Zu + (long long)lane * nw;
        for (int j = 0; j < nw; ++j) un += zu[j] * uvec[j];
      }
      __syncwarp();
      uvec[lane] = u = un;
      __syncwarp();
    }
    // inputs whose own bound is in the working set sit on it exactly; the others are inside the box up to the
    // violation tolerance (1e-11 relative) and are clipped to it, so that the regulator's shifted bounds
    // ulb - us <= 0 <= uub - us keep their signs
    if (done && nW > 0) {
      if (lane < nW && wi[lane] >= row_u) uvec[wi[lane] - row_u] = ws[lane] > 0 ? p.uub[wi[lane] - row_u] : p.ulb[wi[lane] - row_u];
      __syncwarp();
      u = uvec[lane];
    }
    const bool inp = lane < nu;
    if (inp && done) u = fmin(fmax(u, p.ulb[lane]), p.uub[lane]);
    const bool bad = failed || __any_sync(FULLMASK, xs_bad || (inp && !(fabs(u) <= 1.7e308)));
    if (bad && p.fail && lane == 0) atomicExch(p.fail, 1);
    if (inp) p.us[(long long)b * p.us_stride + lane] = u;
    if (p.iters && lane == 0) p.iters[(long long)b * p.iters_stride] = bad ? -it - 1 : it;
    __syncwarp();
  }
}

int ts_solve_device(nnmpc_ts* h, int B, const double* ysp, long long ysp_stride, const double* d,
                    long long d_stride, double* xs, long long xs_stride, double* us, long long us_stride,
                    int* iters, long long iters_stride, const TsFused* fused, const TsIndex* index,
                    int* fail_flag, cudaStream_t st) {
  if (B <= 0) return 0;
  TsParams p{};
  p.B = B; p.nx = h->nx; p.nu = h->nu; p.ny = h->ny; p.nd = h->nd;
  p.Ht = h->Ht; p.Fy = h->Fy; p.Fd = h->Fd; p.f0 = h->f0; p.Gx = h->Gx; p.Gd = h->Gd; p.ulb = h->ulb; p.uub = h->uub;
  p.ysp = ysp; p.ysp_stride = ysp_stride; p.d = d; p.d_stride = d_stride;
  p.xs = xs; p.xs_stride = xs_stride; p.us = us; p.us_stride = us_stride;
  p.iters = iters; p.iters_stride = iters_stride;
  p.fused = fused ? 1 : 0;
  if (fused) p.f = *fused;
  p.indexed = index ? 1 : 0;
  if (index) p.ix = *index;
  p.fail = fail_flag;
  int blocks = (B + TS_WARPS - 1) / TS_WARPS;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (h->general) {      // the dual active-set kernel solves; the kernel below forms xs (unless reduced) and the fused outputs
    p.nw = h->nw; p.mb = h->mb; p.nR = h->nR; p.rld = h->rld; p.rny = h->rny; p.reduced = h->reduced ? 1 : 0;
    p.Hinv = h->Hinv; p.Abar = h->Abar; p.AH = h->AH; p.Mbar = h->Mbar; p.R = h->R; p.lo0 = h->lo0; p.hi0 = h->hi0;
    p.Kx = h->Kx; p.Ku = h->Ku; p.Zx = h->Zx; p.Zu = h->Zu;
    k_ts_general<<<blocks, TS_WARPS * 32, 0, st>>>(p);
    count_launch();
    NNMPC_CUDA(cudaGetLastError());
    p.given = h->reduced ? 2 : 1;
    if (h->reduced && !fused) return 0;      // xs and us are final
  }
  k_target_selector<<<blocks, TS_WARPS * 32, 0, st>>>(p);
  count_launch();
  NNMPC_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace nnmpc

using namespace nnmpc;

extern "C" {

int nnmpc_ts_create(nnmpc_ts_t** out, int nx, int nu, int ny, int nd, const double* Ht, const double* Fy,
                    const double* Fd, const double* f0, const double* Gx, const double* Gd, const double* ulb,
                    const double* uub, int device) {
  if (!out || !Ht || !Fy || !Fd || !f0 || !Gx || !Gd || !ulb || !uub)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_ts_create: null argument");
  if (nu < 1 || nu > 32) return set_error(NNMPC_ERR_UNSUPPORTED, "nnmpc_ts_create: nu=%d not in [1,32]", nu);
  if (nx < 1 || ny < 1 || nd < 0) return set_error(NNMPC_ERR_BADARG, "nnmpc_ts_create: bad sizes");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return set_error(NNMPC_ERR_CUDA, "nnmpc_ts_create: no CUDA device (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return set_error(NNMPC_ERR_BADARG, "nnmpc_ts_create: bad device %d", device);
  DeviceGuard dg(device);
  nnmpc_ts* h = new (std::nothrow) nnmpc_ts();
  if (!h) return set_error(NNMPC_ERR_NOMEM, "out of host memory");
  h->nx = nx; h->nu = nu; h->ny = ny; h->nd = nd; h->nw = nu; h->device = device;
  int rc = upload(&h->Ht, Ht, (size_t)nu * nu);
  if (rc == 0) rc = upload(&h->Fy, Fy, (size_t)nu * ny);
  if (rc == 0) rc = upload(&h->Fd, Fd, (size_t)nu * (nd > 0 ? nd : 1));
  if (rc == 0) rc = upload(&h->f0, f0, (size_t)nu);
  if (rc == 0) rc = upload(&h->Gx, Gx, (size_t)nx * nu);
  if (rc == 0) rc = upload(&h->Gd, Gd, (size_t)nx * (nd > 0 ? nd : 1));
  if (rc == 0) rc = upload(&h->ulb, ulb, (size_t)nu);
  if (rc == 0) rc = upload(&h->uub, uub, (size_t)nu);
  if (rc == 0 && cudaMalloc((void**)&h->fail, sizeof(int)) != cudaSuccess)
    rc = set_error(NNMPC_ERR_NOMEM, "nnmpc_ts_create: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
  if (rc < 0) {          // a half-built handle is released, not leaked
    nnmpc_ts_destroy(h);
    return rc;
  }
  *out = h;
  return 0;
}

int nnmpc_ts_destroy(nnmpc_ts_t* h) {
  if (!h) return 0;
  DeviceGuard dg(h->device);
  cudaFree(h->Ht); cudaFree(h->Fy); cudaFree(h->Fd); cudaFree(h->f0); cudaFree(h->Gx); cudaFree(h->Gd);
  cudaFree(h->ulb); cudaFree(h->uub);
  cudaFree(h->Hinv); cudaFree(h->Abar); cudaFree(h->AH); cudaFree(h->Mbar); cudaFree(h->R); cudaFree(h->lo0); cudaFree(h->hi0);
  cudaFree(h->Kx); cudaFree(h->Ku); cudaFree(h->Zx); cudaFree(h->Zu);
  if (h->fail) cudaFree(h->fail);
  h->hysp.release(); h->hd.release(); h->hxs.release(); h->hus.release(); h->hiters.release();
  delete h;
  return 0;
}

int nnmpc_ts_set_output_bounds(nnmpc_ts_t* h, const double* Hinv, const double* Abar, const double* AH, const double* Mbar,
                               const double* Ryd, const double* ylb, const double* yub) {
  if (!h || !Hinv || !Abar || !AH || !Mbar || !Ryd || !ylb || !yub)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_ts_set_output_bounds: null argument");
  const int mb = h->ny + h->nu;
  if (mb > TS_MAXC) return set_error(NNMPC_ERR_UNSUPPORTED, "nnmpc_ts_set_output_bounds: ny + nu = %d exceeds %d", mb, TS_MAXC);
  if (h->general) return set_error(NNMPC_ERR_BADARG, "nnmpc_ts_set_output_bounds: already set for this handle");
  DeviceGuard dg(h->device);
  const size_t nu = (size_t)h->nu, ny = (size_t)h->ny, nd = (size_t)(h->nd > 0 ? h->nd : 1);
  NNMPC_TRY(upload(&h->Hinv, Hinv, nu * nu));
  NNMPC_TRY(upload(&h->Abar, Abar, (size_t)mb * nu));
  NNMPC_TRY(upload(&h->AH, AH, (size_t)mb * nu));
  NNMPC_TRY(upload(&h->Mbar, Mbar, (size_t)mb * mb));
  NNMPC_TRY(upload(&h->R, Ryd, ny * nd));
  // row bounds [ylb; ulb], [yub; uub]; only the ny output rows carry an offset, Ryd d
  NNMPC_CUDA(cudaMalloc((void**)&h->lo0, (size_t)mb * 8));
  NNMPC_CUDA(cudaMalloc((void**)&h->hi0, (size_t)mb * 8));
  NNMPC_CUDA(cudaMemcpy(h->lo0, ylb, ny * 8, cudaMemcpyHostToDevice));
  NNMPC_CUDA(cudaMemcpy(h->hi0, yub, ny * 8, cudaMemcpyHostToDevice));
  NNMPC_CUDA(cudaMemcpy(h->lo0 + ny, h->ulb, nu * 8, cudaMemcpyDeviceToDevice));
  NNMPC_CUDA(cudaMemcpy(h->hi0 + ny, h->uub, nu * 8, cudaMemcpyDeviceToDevice));
  h->mb = mb; h->nR = h->ny; h->rld = h->nd; h->rny = 0;
  h->general = true;
  return 0;
}

// Uploads n doubles; an empty array (nw = 0) stays a null device pointer and may be null on the host.
static int upload_opt(double** dst, const double* host, size_t n) {
  if (n == 0) return 0;
  return upload(dst, host, n);
}

int nnmpc_ts_create_reduced(nnmpc_ts_t** out, int nx, int nu, int ny, int nd, int nw, int mb, const double* Hinv,
                            const double* Abar, const double* AH, const double* Mbar, const double* Fy, const double* Fd,
                            const double* f0, const double* R, const double* lo0, const double* hi0, const double* Kx,
                            const double* Ku, const double* Zx, const double* Zu, const double* ulb, const double* uub,
                            int device) {
  if (nu < 1 || nu > 32) return set_error(NNMPC_ERR_UNSUPPORTED, "nnmpc_ts_create_reduced: nu=%d not in [1,32]", nu);
  if (nx < 1 || ny < 1 || nd < 0 || nw < 0 || nw > nu || mb < nu)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_ts_create_reduced: bad sizes");
  if (mb > TS_MAXC) return set_error(NNMPC_ERR_UNSUPPORTED, "nnmpc_ts_create_reduced: mb = %d exceeds %d", mb, TS_MAXC);
  if (!out || !Mbar || !R || !lo0 || !hi0 || !Kx || !Ku || !ulb || !uub ||
      (nw > 0 && (!Hinv || !Abar || !AH || !Fy || !f0 || !Zx || !Zu || (nd > 0 && !Fd))))
    return set_error(NNMPC_ERR_BADARG, "nnmpc_ts_create_reduced: null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return set_error(NNMPC_ERR_CUDA, "nnmpc_ts_create_reduced: no CUDA device (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return set_error(NNMPC_ERR_BADARG, "nnmpc_ts_create_reduced: bad device %d", device);
  DeviceGuard dg(device);
  nnmpc_ts* h = new (std::nothrow) nnmpc_ts();
  if (!h) return set_error(NNMPC_ERR_NOMEM, "out of host memory");
  h->nx = nx; h->nu = nu; h->ny = ny; h->nd = nd; h->nw = nw; h->device = device;
  const size_t w = (size_t)nw, m = (size_t)mb, ns = (size_t)(ny + nd);
  int rc = upload_opt(&h->Hinv, Hinv, w * w);
  if (rc == 0) rc = upload_opt(&h->Abar, Abar, m * w);
  if (rc == 0) rc = upload_opt(&h->AH, AH, m * w);
  if (rc == 0) rc = upload(&h->Mbar, Mbar, m * m);
  if (rc == 0) rc = upload_opt(&h->Fy, Fy, w * ny);
  if (rc == 0) rc = upload_opt(&h->Fd, Fd, w * nd);
  if (rc == 0) rc = upload_opt(&h->f0, f0, w);
  if (rc == 0) rc = upload(&h->R, R, m * ns);
  if (rc == 0) rc = upload(&h->lo0, lo0, m);
  if (rc == 0) rc = upload(&h->hi0, hi0, m);
  if (rc == 0) rc = upload(&h->Kx, Kx, (size_t)nx * ns);
  if (rc == 0) rc = upload(&h->Ku, Ku, (size_t)nu * ns);
  if (rc == 0) rc = upload_opt(&h->Zx, Zx, (size_t)nx * w);
  if (rc == 0) rc = upload_opt(&h->Zu, Zu, (size_t)nu * w);
  if (rc == 0) rc = upload(&h->ulb, ulb, (size_t)nu);
  if (rc == 0) rc = upload(&h->uub, uub, (size_t)nu);
  if (rc == 0 && cudaMalloc((void**)&h->fail, sizeof(int)) != cudaSuccess)
    rc = set_error(NNMPC_ERR_NOMEM, "nnmpc_ts_create_reduced: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
  if (rc < 0) {
    nnmpc_ts_destroy(h);
    return rc;
  }
  h->mb = mb; h->nR = mb; h->rld = ny + nd; h->rny = ny;
  h->general = h->reduced = true;
  *out = h;
  return 0;
}

int nnmpc_ts_solve(nnmpc_ts_t* h, int B, const double* ysp, long long ysp_stride, const double* d,
                   long long d_stride, double* xs, double* us, int* iters, void* stream) {
  if (B == 0 && h) return 0;
  if (!h || !ysp || !d || !xs || !us) return set_error(NNMPC_ERR_BADARG, "nnmpc_ts_solve: null argument");
  if (B < 0) return set_error(NNMPC_ERR_BADARG, "nnmpc_ts_solve: negative batch");
  DeviceGuard dg(h->device);
  return ts_solve_device(h, B, ysp, ysp_stride, d, d_stride, xs, h->nx, us, h->nu, iters, 1, nullptr, nullptr, nullptr,
                         (cudaStream_t)stream);
}

int nnmpc_ts_solve_host(nnmpc_ts_t* h, int B, const double* ysp, const double* d, double* xs, double* us,
                        int* iters) {
  if (B == 0 && h) return 0;
  if (!h || !ysp || !d || !xs || !us) return set_error(NNMPC_ERR_BADARG, "nnmpc_ts_solve_host: null argument");
  if (B <= 0) return B == 0 ? 0 : set_error(NNMPC_ERR_BADARG, "nnmpc_ts_solve_host: negative batch");
  DeviceGuard dg(h->device);
  const size_t b = (size_t)B;
  NNMPC_TRY(h->hysp.ensure(b * h->ny));
  NNMPC_TRY(h->hd.ensure(b * (h->nd > 0 ? h->nd : 1)));
  NNMPC_TRY(h->hxs.ensure(b * h->nx));
  NNMPC_TRY(h->hus.ensure(b * h->nu));
  NNMPC_TRY(h->hiters.ensure(b));
  cudaStream_t st = 0;
  NNMPC_CUDA(cudaMemcpyAsync(h->hysp.p, ysp, b * h->ny * 8, cudaMemcpyHostToDevice, st));
  if (h->nd > 0) NNMPC_CUDA(cudaMemcpyAsync(h->hd.p, d, b * h->nd * 8, cudaMemcpyHostToDevice, st));
  NNMPC_CUDA(cudaMemsetAsync(h->fail, 0, sizeof(int), st));
  NNMPC_TRY(ts_solve_device(h, B, h->hysp.p, h->ny, h->hd.p, h->nd, h->hxs.p, h->nx, h->hus.p, h->nu, h->hiters.p, 1,
                            nullptr, nullptr, h->fail, st));
  int failed = 0;
  NNMPC_CUDA(cudaMemcpyAsync(&failed, h->fail, sizeof(int), cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaMemcpyAsync(xs, h->hxs.p, b * h->nx * 8, cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaMemcpyAsync(us, h->hus.p, b * h->nu * 8, cudaMemcpyDeviceToHost, st));
  if (iters) NNMPC_CUDA(cudaMemcpyAsync(iters, h->hiters.p, b * 4, cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaStreamSynchronize(st));
  return failed ? NNMPC_WARN_TARGET : 0;
}

}  // extern "C"
