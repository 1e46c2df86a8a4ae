// Batched regulator QP of a re-parameterised (open-loop unstable) plant by a primal-dual interior-point method with
// a Riccati recursion per Newton step (Rao, Wright & Rawlings, J. Optim. Theory Appl. 99 (1998) 723-757).
//
// The reference solves, for an unstable A, the condensed QP in v of u = K x + v with general inequalities
// G v <= h(x0) (/root/reference/lib/linearMPC.py:366-382, :476-493).  Its image in u (the box QP the Douglas-Rachford
// path of qp.cu solves) has a Hessian whose condition number grows like rho^2N with the unstable pole rho, while the
// v-space problem stays benign; all the ill-conditioning sits in the map T = I + tK tB.  A first-order method in v
// inherits the u-space rate (DESIGN.md section 2), so this file solves the v-space problem in its stagewise form
//     min  1/2 sum_{k<N} (x_k'Q x_k + v_k'R v_k + 2 x_k'M v_k) + 1/2 x_N'Pf x_N
//     s.t. x_{k+1} = A x_k + B v_k,  x_0 = x0,   lb <= K x_k + v_k <= ub   (per stage, per sample lb/ub)
// with A = A_open + B K stable.  Nothing here forms P_u or T^-1.
//
// Method (per sample): Mehrotra predictor-corrector with slacks s_l = u - lb, s_u = ub - u and multipliers z_l, z_u
// for every finite bound (an infinite bound is absent).  Start: the saturated-LQR roll-out u_k = clip(K x_k), with the
// multipliers that make stationarity exact there (s = max(slack, 1), z = split of mu + 1).  The primal iterate is v;
// x is always the forward roll-out of v on the stable A, so the dynamics hold to rounding.  A Newton step is an LQ
// problem, factorised in the stage's original inputs u = K x + v: weights Q + K'RK - MK - K'M', M - K'R, R + D
// (D = z_l/s_l + z_u/s_u) and dynamics A - BK.  (Written in v the weights are Q + K'DK, M + K'D, R + D, and with
// bounds active over much of the horizon the Riccati update cancels K'DK against S'Re^-1 S to rounding; in u the
// barrier enters only Re.)  One backward Riccati recursion (Cholesky of the nu x nu  R + D + B'P B per stage, gains
// and factors to per-CTA global scratch) serves the predictor and the corrector, each of which then costs one vector
// backward pass and one forward roll-out.
//
// Certificate (the `kkt` output), evaluated in FP64 at the returned point from the adjoint
//     lambda_N = Pf x_N,  lambda_k = Q x_k + M v_k + A'lambda_{k+1} + K'mu_k,   mu = z_u - z_l (net bound multiplier):
//     kkt = max( max|R v_k + M'x_k + B'lambda_{k+1} + mu_k| / g,  max bound violation of u / s_u,
//                max |mu| * (distance of u to the bound mu pushes against) / (g s_u) )
// with g = 1 + the largest magnitude of the four stationarity terms and s_u = 1 + max|u| (a relative measure; the adjoint
// and every roll-out run on the stable A).  A sample stops once kkt <= tol and its mean complementarity s'z / m is at most
// 1e-6 tol g s_u (one or two more iterations of the superlinear end phase, which puts the multipliers of inactive
// bounds at rounding level: a sample with no active bound returns the LQR roll-out, v = 0, to rounding).
//
// cost = the reference's objective 1/2 v'P v + (tq x0)'v, i.e. the stagewise cost of the returned point minus that of
// v = 0, accumulated without that cancellation from the roll-out delta of v from a zero state.  (The Douglas-Rachford
// path reports the u-space value 1/2 u'P_u u + (tq_u x0)'u instead; the two differ by a constant in x0.)
//
// One CTA of IPM_THREADS threads per QP on a grid of one resident wave (occupancy query) that strides over the batch; a sample
// that has stopped leaves its CTA, which takes the next one.  Every reduction has a fixed order, so a sample's result
// is bitwise independent of the batch.  Limits: nxa <= IPM_MAX_NX = 64 and nu <= IPM_MAX_NU = 32 (shared memory of
// the Riccati step).  A sample with lb >= ub somewhere (or a NaN bound) or a non-finite x0 returns NaN with
// iters = max_iter (NNMPC_WARN_MAXITER); so does a sample whose Riccati factorisation breaks down.
#include "qp.cuh"
#include <cmath>

namespace nnmpc {

constexpr int IPM_THREADS = 256;
constexpr int IPM_MAX_NX = 64;
constexpr int IPM_MAX_NU = 32;

struct IpmOps {
  const double *A, *B, *Q, *R, *M, *Pf, *K;   // nx x nx, nx x nu, nx x nx, nu x nu, nx x nu, nx x nx, nu x nx
  // the same stage in the original inputs u = K x + v (Newton-step factorisation): A - B K, Q + K'RK - MK - K'M', M - K'R
  const double *Ao, *Qo, *Mo;
  int nx, nu, N;
};

// per-CTA scratch (doubles), offsets in units of one stage vector
struct IpmScratch {
  double *Kg, *Lc, *kf, *X, *Xf, *DX, *V, *U, *SL, *SU, *ZL, *ZU, *DV, *DSL, *DSU, *DZL, *DZU, *RV, *RPL, *RPU, *D, *E,
      *RCL, *RCU;
};

__host__ __device__ inline long long ipm_scratch_doubles(int nx, int nu, int N) {
  return (long long)N * nu * nx + (long long)N * nu * nu + 3LL * (N + 1) * nx + 19LL * N * nu;
}

__device__ inline IpmScratch ipm_carve(double* base, int nx, int nu, int N) {
  IpmScratch s;
  double* p = base;
  const long long sv = (long long)N * nu;
  s.Kg = p; p += (long long)N * nu * nx;
  s.Lc = p; p += (long long)N * nu * nu;
  s.X = p; p += (long long)(N + 1) * nx;
  s.Xf = p; p += (long long)(N + 1) * nx;
  s.DX = p; p += (long long)(N + 1) * nx;
  double** vecs[] = {&s.kf, &s.V, &s.U, &s.SL, &s.SU, &s.ZL, &s.ZU, &s.DV, &s.DSL, &s.DSU, &s.DZL, &s.DZU, &s.RV,
                     &s.RPL, &s.RPU, &s.D, &s.E, &s.RCL, &s.RCU};
  for (double** v : vecs) { *v = p; p += sv; }
  return s;
}

// deterministic block reductions (fixed tree); `red` holds IPM_THREADS / 32 doubles
__device__ double block_max(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v = nan_max(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = red[0];
  for (int w = 1; w < IPM_THREADS / 32; ++w) r = nan_max(r, red[w]);
  return r;
}
__device__ double block_min(double v, double* red) { return -block_max(-v, red); }
__device__ double block_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = red[0];
  for (int w = 1; w < IPM_THREADS / 32; ++w) r += red[w];
  return r;
}

// X_0 = x0 (or 0), X_{k+1} = A X_k + B v_k (v = null: free response); u = K x + v when U is non-null
__device__ void ipm_rollout(const IpmOps& o, const double* x0, const double* v, double* X, double* U) {
  const int nx = o.nx, nu = o.nu;
  for (int i = threadIdx.x; i < nx; i += blockDim.x) X[i] = x0 ? x0[i] : 0.0;
  __syncthreads();
  for (int k = 0; k < o.N; ++k) {
    const double* xk = X + (long long)k * nx;
    const double* vk = v ? v + (long long)k * nu : nullptr;
    for (int i = threadIdx.x; i < nx; i += blockDim.x) {
      double a = 0.0;
      for (int j = 0; j < nx; ++j) a += o.A[i * nx + j] * xk[j];
      if (vk)
        for (int l = 0; l < nu; ++l) a += o.B[i * nu + l] * vk[l];
      X[(long long)(k + 1) * nx + i] = a;
    }
    __syncthreads();
  }
  if (U) {
    for (int t = threadIdx.x; t < o.N * nu; t += blockDim.x) {
      const int k = t / nu, i = t - k * nu;
      double a = v[t];
      for (int j = 0; j < nx; ++j) a += o.K[i * nx + j] * X[(long long)k * nx + j];
      U[t] = a;
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(IPM_THREADS, 2)
k_ipm(IpmOps o, int Bn, const double* __restrict__ x0g, int x0_ld, const double* __restrict__ lbg,
      const double* __restrict__ ubg, double* __restrict__ Ug, QpOutputs out, double tol, int max_iter,
      double* __restrict__ scratch, long long per_cta, int* __restrict__ flag_maxiter,
      unsigned long long* __restrict__ iter_sum) {
  extern __shared__ double sm[];
  const int nx = o.nx, nu = o.nu, N = o.N;
  const long long nv = (long long)N * nu;
  double* P = sm;                 // nx x nx   cost-to-go Hessian
  double* PA = P + nx * nx;       // nx x nx
  double* PB = PA + nx * nx;      // nx x nu
  double* Re = PB + nx * nu;      // nu x nu   -> its Cholesky factor
  double* Se = Re + nu * nu;      // nu x nx   -> L^-1 Se -> gain
  double* va = Se + nu * nx;      // nx
  double* vb = va + nx;           // nx
  double* se = vb + nx;           // nu
  double* lb = se + nu;           // nu
  double* ub = lb + nu;           // nu
  double* red = ub + nu;          // IPM_THREADS / 32
  __shared__ int s_bad;
  IpmScratch S = ipm_carve(scratch + (long long)blockIdx.x * per_cta, nx, nu, N);
  const int tid = threadIdx.x;

  for (int b = blockIdx.x; b < Bn; b += gridDim.x) {
    const double* x0 = x0g + (long long)b * x0_ld;
    if (tid == 0) s_bad = 0;
    __syncthreads();
    for (int i = tid; i < nu; i += blockDim.x) {
      lb[i] = lbg[(long long)b * nu + i];
      ub[i] = ubg[(long long)b * nu + i];
      if (!(lb[i] < ub[i])) s_bad = 1;
    }
    for (int i = tid; i < x0_ld; i += blockDim.x)
      if (!isfinite(x0[i])) s_bad = 1;
    __syncthreads();
    int m = 0;   // finite bound sides per stage
    for (int i = 0; i < nu; ++i) m += (isinf(lb[i]) ? 0 : 1) + (isinf(ub[i]) ? 0 : 1);
    const double mtot = (double)m * N;
    int it = 0;
    double cert = __longlong_as_double(0x7ff8000000000000ll);
    bool ok = false;
    if (!s_bad) {
      // cold start from the saturated LQR roll-out u_k = clip(K x_k) (v = u - K x, x on the stable A), with the
      // multipliers that make stationarity exact there: mu_k = -(R v_k + M'x_k + B'lambda_{k+1}) along the adjoint.
      // Their scale follows the cost of the roll-out (large where the plant runs away under saturation), which a
      // start at z = 1 would have to climb to with fraction-to-boundary steps.
      for (int i = tid; i < nx; i += blockDim.x) S.X[i] = x0[i];
      __syncthreads();
      for (int k = 0; k < N; ++k) {
        const double* xk = S.X + (long long)k * nx;
        if (tid < nu) {
          double ul = 0.0;
          for (int j = 0; j < nx; ++j) ul += o.K[tid * nx + j] * xk[j];
          const double u = fmin(fmax(ul, lb[tid]), ub[tid]);
          S.U[(long long)k * nu + tid] = u;
          S.V[(long long)k * nu + tid] = u - ul;
        }
        __syncthreads();
        for (int i = tid; i < nx; i += blockDim.x) {
          double a = 0.0;
          for (int j = 0; j < nx; ++j) a += o.A[i * nx + j] * xk[j];
          for (int l = 0; l < nu; ++l) a += o.B[i * nu + l] * S.V[(long long)k * nu + l];
          S.X[(long long)(k + 1) * nx + i] = a;
        }
        __syncthreads();
      }
      {
        double* lam = va;
        double* lam2 = vb;
        for (int i = tid; i < nx; i += blockDim.x) {
          double a = 0.0;
          for (int j = 0; j < nx; ++j) a += o.Pf[i * nx + j] * S.X[(long long)N * nx + j];
          lam[i] = a;
        }
        __syncthreads();
        for (int k = N - 1; k >= 0; --k) {
          const double* xk = S.X + (long long)k * nx;
          const double* vk = S.V + (long long)k * nu;
          if (tid < nu) {
            double g = 0.0;
            for (int j = 0; j < nu; ++j) g += o.R[tid * nu + j] * vk[j];
            for (int j = 0; j < nx; ++j) g += o.M[j * nu + tid] * xk[j] + o.B[j * nu + tid] * lam[j];
            se[tid] = -g;
          }
          __syncthreads();
          for (int i = tid; i < nx; i += blockDim.x) {
            double a = 0.0;
            for (int j = 0; j < nx; ++j) a += o.Q[i * nx + j] * xk[j] + o.A[j * nx + i] * lam[j];
            for (int l = 0; l < nu; ++l) a += o.M[i * nu + l] * vk[l] + o.K[l * nx + i] * se[l];
            lam2[i] = a;
          }
          if (tid < nu) {
            const double mu = se[tid];
            const long long t = (long long)k * nu + tid;
            const bool fl = !isinf(lb[tid]), fu = !isinf(ub[tid]);
            S.SL[t] = fl ? fmax(S.U[t] - lb[tid], 1.0) : 1.0;
            S.SU[t] = fu ? fmax(ub[tid] - S.U[t], 1.0) : 1.0;
            S.ZL[t] = fl ? fmax(-mu, 0.0) + 1.0 : 0.0;
            S.ZU[t] = fu ? fmax(mu, 0.0) + 1.0 : 0.0;
          }
          __syncthreads();
          double* t = lam; lam = lam2; lam2 = t;
        }
      }
      for (it = 0;; ++it) {
        ipm_rollout(o, x0, S.V, S.X, S.U);
        // ---- adjoint pass: stationarity residual r_v and the certificate at (v, x, mu = z_u - z_l)
        double* lam = va;
        double* lam2 = vb;
        for (int i = tid; i < nx; i += blockDim.x) {
          double a = 0.0;
          for (int j = 0; j < nx; ++j) a += o.Pf[i * nx + j] * S.X[(long long)N * nx + j];
          lam[i] = a;
        }
        __syncthreads();
        double gmax = 0.0, rmax = 0.0;
        for (int k = N - 1; k >= 0; --k) {
          const double* xk = S.X + (long long)k * nx;
          const double* vk = S.V + (long long)k * nu;
          const double* zl = S.ZL + (long long)k * nu;
          const double* zu = S.ZU + (long long)k * nu;
          if (tid < nu) {
            const int i = tid;
            double t1 = 0.0, t2 = 0.0, t3 = 0.0;
            for (int j = 0; j < nu; ++j) t1 += o.R[i * nu + j] * vk[j];
            for (int j = 0; j < nx; ++j) t2 += o.M[j * nu + i] * xk[j];
            for (int j = 0; j < nx; ++j) t3 += o.B[j * nu + i] * lam[j];
            const double mu = zu[i] - zl[i];
            const double r = t1 + t2 + t3 + mu;
            S.RV[(long long)k * nu + i] = r;
            rmax = nan_max(rmax, fabs(r));
            gmax = nan_max(gmax, fmax(fmax(fabs(t1), fabs(t2)), fmax(fabs(t3), fabs(mu))));
          } else if (tid >= 32 && tid - 32 < nx) {
            const int i = tid - 32;
            double a = 0.0;
            for (int j = 0; j < nx; ++j) a += o.Q[i * nx + j] * xk[j];
            for (int l = 0; l < nu; ++l) a += o.M[i * nu + l] * vk[l];
            for (int j = 0; j < nx; ++j) a += o.A[j * nx + i] * lam[j];
            for (int l = 0; l < nu; ++l) a += o.K[l * nx + i] * (zu[l] - zl[l]);
            lam2[i] = a;
          }
          __syncthreads();
          double* t = lam; lam = lam2; lam2 = t;
        }
        double umax = 0.0, viol = 0.0, comp = 0.0, gap = 0.0;
        for (long long t = tid; t < nv; t += blockDim.x) {
          const int i = (int)(t % nu);
          const double u = S.U[t], mu = S.ZU[t] - S.ZL[t];
          const bool fl = !isinf(lb[i]), fu = !isinf(ub[i]);
          umax = nan_max(umax, fabs(u));
          if (fl) viol = nan_max(viol, lb[i] - u);
          if (fu) viol = nan_max(viol, u - ub[i]);
          if (mu != 0.0) {
            const bool up = mu > 0.0;
            const double d = up ? (fu ? ub[i] - u : INFINITY) : (fl ? u - lb[i] : INFINITY);
            comp = nan_max(comp, fabs(mu) * fabs(d));
          } else if (mu != mu) {
            comp = mu;
          }
          gap += (fl ? S.SL[t] * S.ZL[t] : 0.0) + (fu ? S.SU[t] * S.ZU[t] : 0.0);
        }
        const double g = 1.0 + block_max(gmax, red);
        const double us = 1.0 + block_max(umax, red);
        const double rm = block_max(rmax, red);
        const double vm = block_max(viol, red);
        const double cm = block_max(comp, red);
        const double mu_avg = mtot > 0 ? block_sum(gap, red) / mtot : 0.0;
        cert = nan_max(nan_max(rm / g, vm / us), cm / (g * us));
        if (cert <= tol && (m == 0 || mu_avg <= 1e-6 * tol * g * us)) { ok = true; break; }
        if (it >= max_iter || !isfinite(cert)) break;

        // ---- Newton system: primal slack residuals and barrier diagonal
        for (long long t = tid; t < nv; t += blockDim.x) {
          const int i = (int)(t % nu);
          const bool fl = !isinf(lb[i]), fu = !isinf(ub[i]);
          S.RPL[t] = fl ? (S.U[t] - lb[i]) - S.SL[t] : 0.0;
          S.RPU[t] = fu ? (ub[i] - S.U[t]) - S.SU[t] : 0.0;
          S.D[t] = S.ZL[t] / S.SL[t] + S.ZU[t] / S.SU[t];
        }
        // ---- backward Riccati recursion (factorisation shared by predictor and corrector)
        for (int t = tid; t < nx * nx; t += blockDim.x) P[t] = o.Pf[t];
        __syncthreads();
        for (int k = N - 1; k >= 0; --k) {
          const double* Dk = S.D + (long long)k * nu;
          for (int t = tid; t < nx * (nx + nu); t += blockDim.x) {
            if (t < nx * nx) {
              const int i = t / nx, j = t - i * nx;
              double a = 0.0;
              for (int l = 0; l < nx; ++l) a += P[i * nx + l] * o.Ao[l * nx + j];
              PA[t] = a;
            } else {
              const int r = t - nx * nx, i = r / nu, j = r - i * nu;
              double a = 0.0;
              for (int l = 0; l < nx; ++l) a += P[i * nx + l] * o.B[l * nu + j];
              PB[r] = a;
            }
          }
          __syncthreads();
          for (int t = tid; t < nu * (nu + nx); t += blockDim.x) {
            if (t < nu * nu) {
              const int i = t / nu, j = t - i * nu;
              double a = o.R[t] + (i == j ? Dk[i] : 0.0);
              for (int l = 0; l < nx; ++l) a += o.B[l * nu + i] * PB[l * nu + j];
              Re[t] = a;
            } else {
              const int r = t - nu * nu, i = r / nx, j = r - i * nx;
              double a = o.Mo[j * nu + i];
              for (int l = 0; l < nx; ++l) a += o.B[l * nu + i] * PA[l * nx + j];
              Se[r] = a;
            }
          }
          __syncthreads();
          if (tid < 32) {   // Cholesky Re = L L' by one warp, lane i owns row i (lower triangle)
            const int i = tid;
            for (int c = 0; c < nu; ++c) {
              if (i == c) {
                const double d = Re[c * nu + c];
                if (!(d > 0.0)) s_bad = 1;
                Re[c * nu + c] = sqrt(d);
              }
              __syncwarp();
              if (i > c && i < nu) Re[i * nu + c] /= Re[c * nu + c];
              __syncwarp();
              if (i > c && i < nu)
                for (int j = c + 1; j <= i; ++j) Re[i * nu + j] -= Re[i * nu + c] * Re[j * nu + c];
              __syncwarp();
            }
          }
          __syncthreads();
          double* Lk = S.Lc + (long long)k * nu * nu;
          for (int t = tid; t < nu * nu; t += blockDim.x) Lk[t] = Re[t];
          for (int j = tid; j < nx; j += blockDim.x) {   // Y = L^-1 Se, column by column in place
            for (int i = 0; i < nu; ++i) {
              double a = Se[i * nx + j];
              for (int l = 0; l < i; ++l) a -= Re[i * nu + l] * Se[l * nx + j];
              Se[i * nx + j] = a / Re[i * nu + i];
            }
          }
          __syncthreads();
          // P_k = Q + K'DK + A'PA - Y'Y  (upper triangle computed, mirrored: symmetric by construction)
          for (int t = tid; t < nx * nx; t += blockDim.x) {
            const int i = t / nx, j = t - i * nx;
            if (j < i) continue;
            double a = o.Qo[t];
            for (int l = 0; l < nx; ++l) a += o.Ao[l * nx + i] * PA[l * nx + j];
            for (int l = 0; l < nu; ++l) a -= Se[l * nx + i] * Se[l * nx + j];
            P[i * nx + j] = a;
            P[j * nx + i] = a;
          }
          __syncthreads();
          double* Kk = S.Kg + (long long)k * nu * nx;
          for (int j = tid; j < nx; j += blockDim.x) {   // gain = -L'^-1 Y
            for (int i = nu - 1; i >= 0; --i) {
              double a = Se[i * nx + j];
              for (int l = i + 1; l < nu; ++l) a -= Re[l * nu + i] * Se[l * nx + j];
              Se[i * nx + j] = a / Re[i * nu + i];
              Kk[i * nx + j] = -Se[i * nx + j];
            }
          }
          __syncthreads();
        }
        if (s_bad) break;

        // ---- one right-hand side: e from (RCL, RCU); direction (DV, DX) and (DSL, DSU, DZL, DZU)
        auto direction = [&]() {
          for (long long t = tid; t < nv; t += blockDim.x)
            S.E[t] = (S.RCL[t] + S.ZL[t] * S.RPL[t]) / S.SL[t] - (S.RCU[t] + S.ZU[t] * S.RPU[t]) / S.SU[t];
          for (int i = tid; i < nx; i += blockDim.x) va[i] = 0.0;
          __syncthreads();
          double* p = va;
          double* p2 = vb;
          for (int k = N - 1; k >= 0; --k) {
            const double* ek = S.E + (long long)k * nu;
            const double* Kk = S.Kg + (long long)k * nu * nx;
            if (tid < nu) {
              double a = S.RV[(long long)k * nu + tid] + ek[tid];
              for (int l = 0; l < nx; ++l) a += o.B[l * nu + tid] * p[l];
              se[tid] = a;
            }
            __syncthreads();
            if (tid == 0) {   // feed-forward -Re^-1 se through the stored factor
              const double* L = S.Lc + (long long)k * nu * nu;
              double* kf = S.kf + (long long)k * nu;
              for (int i = 0; i < nu; ++i) {
                double a = se[i];
                for (int l = 0; l < i; ++l) a -= L[i * nu + l] * kf[l];
                kf[i] = a / L[i * nu + i];
              }
              for (int i = nu - 1; i >= 0; --i) {
                double a = kf[i];
                for (int l = i + 1; l < nu; ++l) a -= L[l * nu + i] * kf[l];
                kf[i] = a / L[i * nu + i];
              }
              for (int i = 0; i < nu; ++i) kf[i] = -kf[i];
            } else if (tid >= 32 && tid - 32 < nx) {
              const int i = tid - 32;
              double a = 0.0;
              for (int l = 0; l < nu; ++l) a -= o.K[l * nx + i] * S.RV[(long long)k * nu + l];
              for (int l = 0; l < nx; ++l) a += o.Ao[l * nx + i] * p[l];
              for (int l = 0; l < nu; ++l) a += Kk[l * nx + i] * se[l];
              p2[i] = a;
            }
            __syncthreads();
            double* t = p; p = p2; p2 = t;
          }
          // forward: du_k = Kk dx_k + kf_k, dv_k = du_k - K dx_k, dx_{k+1} = (A - BK) dx_k + B du_k
          for (int i = tid; i < nx; i += blockDim.x) S.DX[i] = 0.0;
          __syncthreads();
          for (int k = 0; k < N; ++k) {
            const double* dxk = S.DX + (long long)k * nx;
            if (tid < nu) {
              const double* Kk = S.Kg + (long long)k * nu * nx;
              double a = S.kf[(long long)k * nu + tid];
              double kx = 0.0;
              for (int j = 0; j < nx; ++j) {
                a += Kk[tid * nx + j] * dxk[j];
                kx += o.K[tid * nx + j] * dxk[j];
              }
              se[tid] = a;
              S.DV[(long long)k * nu + tid] = a - kx;
            }
            __syncthreads();
            for (int i = tid; i < nx; i += blockDim.x) {
              double a = 0.0;
              for (int j = 0; j < nx; ++j) a += o.Ao[i * nx + j] * dxk[j];
              for (int l = 0; l < nu; ++l) a += o.B[i * nu + l] * se[l];
              S.DX[(long long)(k + 1) * nx + i] = a;
            }
            __syncthreads();
          }
          for (long long t = tid; t < nv; t += blockDim.x) {
            const int k = (int)(t / nu), i = (int)(t - (long long)k * nu);
            const bool fl = !isinf(lb[i]), fu = !isinf(ub[i]);
            double du = S.DV[t];
            for (int j = 0; j < nx; ++j) du += o.K[i * nx + j] * S.DX[(long long)k * nx + j];
            const double dsl = fl ? du + S.RPL[t] : 0.0;
            const double dsu = fu ? -du + S.RPU[t] : 0.0;
            S.DSL[t] = dsl;
            S.DSU[t] = dsu;
            S.DZL[t] = fl ? -(S.RCL[t] + S.ZL[t] * dsl) / S.SL[t] : 0.0;
            S.DZU[t] = fu ? -(S.RCU[t] + S.ZU[t] * dsu) / S.SU[t] : 0.0;
          }
          __syncthreads();
        };
        // largest step in (0, 1] that keeps s and z non-negative
        auto max_step = [&]() -> double {
          double a = 1.0;
          for (long long t = tid; t < nv; t += blockDim.x) {
            if (S.DSL[t] < 0.0) a = fmin(a, -S.SL[t] / S.DSL[t]);
            if (S.DSU[t] < 0.0) a = fmin(a, -S.SU[t] / S.DSU[t]);
            if (S.DZL[t] < 0.0) a = fmin(a, -S.ZL[t] / S.DZL[t]);
            if (S.DZU[t] < 0.0) a = fmin(a, -S.ZU[t] / S.DZU[t]);
          }
          return block_min(a, red);
        };
        double alpha = 1.0;
        if (m > 0) {
          // predictor (affine scaling): rc = s z
          for (long long t = tid; t < nv; t += blockDim.x) {
            S.RCL[t] = S.SL[t] * S.ZL[t];
            S.RCU[t] = S.SU[t] * S.ZU[t];
          }
          direction();
          const double aa = max_step();
          double ga = 0.0;
          for (long long t = tid; t < nv; t += blockDim.x)
            ga += (S.SL[t] + aa * S.DSL[t]) * (S.ZL[t] + aa * S.DZL[t]) + (S.SU[t] + aa * S.DSU[t]) * (S.ZU[t] + aa * S.DZU[t]);
          const double mu_aff = block_sum(ga, red) / mtot;
          const double ratio = mu_aff / mu_avg;
          const double sigmu = ratio * ratio * ratio * mu_avg;
          // corrector: rc = s z + ds_aff dz_aff - sigma mu  (absent sides keep z = 0, ds = dz = 0)
          for (long long t = tid; t < nv; t += blockDim.x) {
            const int i = (int)(t % nu);
            const bool fl = !isinf(lb[i]), fu = !isinf(ub[i]);
            S.RCL[t] = fl ? S.SL[t] * S.ZL[t] + S.DSL[t] * S.DZL[t] - sigmu : 0.0;
            S.RCU[t] = fu ? S.SU[t] * S.ZU[t] + S.DSU[t] * S.DZU[t] - sigmu : 0.0;
          }
          direction();
          alpha = fmin(1.0, 0.995 * max_step());
        } else {
          for (long long t = tid; t < nv; t += blockDim.x) S.RCL[t] = S.RCU[t] = 0.0;
          direction();
        }
        for (long long t = tid; t < nv; t += blockDim.x) {
          S.V[t] += alpha * S.DV[t];
          S.SL[t] += alpha * S.DSL[t];
          S.SU[t] += alpha * S.DSU[t];
          S.ZL[t] += alpha * S.DZL[t];
          S.ZU[t] += alpha * S.DZU[t];
        }
        __syncthreads();
      }
    }
    // ---- outputs: the last iterate (certified when ok); NaN for bad input or a breakdown
    double* Ub = Ug + (long long)b * nv;
    if (!s_bad && isfinite(cert)) {
      for (long long t = tid; t < nv; t += blockDim.x) Ub[t] = S.U[t];
      if (out.cost) {
        // 1/2 v'Pv + (tq x0)'v = sum_k [1/2 d_k'Q (x_k + f_k) + 1/2 v_k'R v_k + x_k'M v_k] + 1/2 d_N'Pf (x_N + f_N)
        // with f the free response of x0 and d = x - f the response of v from a zero state
        ipm_rollout(o, x0, nullptr, S.Xf, nullptr);
        ipm_rollout(o, nullptr, S.V, S.DX, nullptr);
        double acc = 0.0;
        for (long long t = tid; t < (long long)(N + 1) * nx; t += blockDim.x) {
          const int k = (int)(t / nx), i = (int)(t - (long long)k * nx);
          const double* W = k < N ? o.Q : o.Pf;
          double a = 0.0;
          for (int j = 0; j < nx; ++j)
            a += W[i * nx + j] * (S.X[(long long)k * nx + j] + S.Xf[(long long)k * nx + j]);
          acc += 0.5 * S.DX[t] * a;
          if (k < N)
            for (int l = 0; l < nu; ++l) acc += S.X[t] * o.M[i * nu + l] * S.V[(long long)k * nu + l];
        }
        for (long long t = tid; t < nv; t += blockDim.x) {
          const int k = (int)(t / nu), i = (int)(t - (long long)k * nu);
          double a = 0.0;
          for (int l = 0; l < nu; ++l) a += o.R[i * nu + l] * S.V[(long long)k * nu + l];
          acc += 0.5 * S.V[t] * a;
        }
        const double c = block_sum(acc, red);
        if (tid == 0) out.cost[(long long)b * out.stride] = c;
      }
    } else {
      const double qnan = __longlong_as_double(0x7ff8000000000000ll);
      for (long long t = tid; t < nv; t += blockDim.x) Ub[t] = qnan;
      if (out.cost && tid == 0) out.cost[(long long)b * out.stride] = qnan;
      cert = qnan;
    }
    if (!ok) it = max_iter;
    if (tid == 0) {
      if (out.kkt) out.kkt[(long long)b * out.stride] = cert;
      if (out.iters) out.iters[(long long)b * out.stride] = it;
      atomicAdd(iter_sum, (unsigned long long)it);
      if (!ok) atomicExch(flag_maxiter, 1);
    }
    __syncthreads();
  }
}

inline size_t ipm_smem_bytes(int nx, int nu) {
  return (size_t)(2 * nx * nx + 2 * nx * nu + nu * nu + 2 * nx + 3 * nu + IPM_THREADS / 32) * sizeof(double);
}

int ipm_solve_device(nnmpc_qp* h, int B, const double* x0, const double* lb, const double* ub, double* u,
                     QpOutputs out, double tol, int max_iter, cudaStream_t st, long long* iter_sum_out) {
  if (B <= 0) return 0;
  if (max_iter < 1) max_iter = 1;
  const int nx = h->nxa, nu = h->nu, N = h->N;
  const long long per_cta = (ipm_scratch_doubles(nx, nu, N) + 31) & ~31LL;
  const size_t smem = ipm_smem_bytes(nx, nu);
  if (smem > 48 * 1024)
    NNMPC_CUDA(cudaFuncSetAttribute(k_ipm, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // one resident wave of CTAs (the occupancy of k_ipm at this shared-memory size), fewer if the per-CTA scratch would
  // pass 4 GiB in total
  int dev = 0, sms = 0, per_sm = 0;
  NNMPC_CUDA(cudaGetDevice(&dev));
  NNMPC_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  NNMPC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_ipm, IPM_THREADS, smem));
  long long grid = (long long)sms * (per_sm > 0 ? per_sm : 1);
  if (grid > B) grid = B;
  const long long mem_cap = (4LL << 30) / (per_cta * (long long)sizeof(double));
  if (grid > mem_cap) grid = mem_cap < 1 ? 1 : mem_cap;
  NNMPC_TRY(h->ipm_scr.ensure((size_t)(grid * per_cta)));
  NNMPC_CUDA(cudaMemsetAsync(h->counts, 0, 4 * sizeof(int), st));
  NNMPC_CUDA(cudaMemsetAsync(h->iter_sum, 0, sizeof(unsigned long long), st));
  IpmOps o{h->iA, h->iB, h->iQ, h->iR, h->iM, h->iPf, h->iK, h->iAo, h->iQo, h->iMo, nx, nu, N};
  k_ipm<<<(unsigned)grid, IPM_THREADS, smem, st>>>(o, B, x0, nx, lb, ub, u, out, tol, max_iter, h->ipm_scr.p, per_cta,
                                                  h->counts + 2, h->iter_sum);
  count_launch();
  NNMPC_CUDA(cudaGetLastError());
  NNMPC_CUDA(cudaMemcpyAsync(h->h_pinned, h->counts, 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaMemcpyAsync(h->h_pinned + 4, h->iter_sum, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaStreamSynchronize(st));
  unsigned long long isum;
  memcpy(&isum, h->h_pinned + 4, sizeof(isum));
  if (iter_sum_out) *iter_sum_out = (long long)isum;
  return h->h_pinned[2] ? NNMPC_WARN_MAXITER : 0;
}

}  // namespace nnmpc

using namespace nnmpc;

extern "C" {

int nnmpc_qp_create_ipm(nnmpc_qp_t** out, int nxa_ld, int nu, int N, const double* A_host, const double* B_host,
                        const double* Q_host, const double* R_host, const double* M_host, const double* Pf_host,
                        const double* K_host, int device) {
  if (!out || !A_host || !B_host || !Q_host || !R_host || !M_host || !Pf_host || !K_host)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_qp_create_ipm: null argument");
  if (nxa_ld <= 0 || nu <= 0 || N <= 0) return set_error(NNMPC_ERR_BADARG, "nnmpc_qp_create_ipm: sizes must be positive");
  if (nxa_ld > IPM_MAX_NX || nu > IPM_MAX_NU)
    return set_error(NNMPC_ERR_UNSUPPORTED, "nnmpc_qp_create_ipm: nxa = %d, nu = %d: the interior-point kernel holds "
                     "nxa <= %d and nu <= %d", nxa_ld, nu, IPM_MAX_NX, IPM_MAX_NU);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return set_error(NNMPC_ERR_CUDA, "nnmpc_qp_create_ipm: no CUDA device (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return set_error(NNMPC_ERR_BADARG, "nnmpc_qp_create_ipm: bad device %d", device);
  DeviceGuard dg(device);
  nnmpc_qp* h = new (std::nothrow) nnmpc_qp();
  if (!h) return set_error(NNMPC_ERR_NOMEM, "out of host memory");
  h->ipm = 1;
  h->n = N * nu; h->nxa = nxa_ld; h->nu = nu; h->N = N; h->device = device; h->alpha = 1.0;
  const size_t nx = (size_t)nxa_ld;
  int rc = upload(&h->iA, A_host, nx * nx);
  if (rc == 0) rc = upload(&h->iB, B_host, nx * nu);
  if (rc == 0) rc = upload(&h->iQ, Q_host, nx * nx);
  if (rc == 0) rc = upload(&h->iR, R_host, (size_t)nu * nu);
  if (rc == 0) rc = upload(&h->iM, M_host, nx * nu);
  if (rc == 0) rc = upload(&h->iPf, Pf_host, nx * nx);
  if (rc == 0) rc = upload(&h->iK, K_host, (size_t)nu * nx);
  if (rc == 0) {   // the stage in the original inputs: A - BK, Q + K'RK - MK - K'M', M - K'R
    double* Ao = new (std::nothrow) double[nx * nx];
    double* Qo = new (std::nothrow) double[nx * nx];
    double* Mo = new (std::nothrow) double[nx * nu];
    if (!Ao || !Qo || !Mo) {
      rc = set_error(NNMPC_ERR_NOMEM, "out of host memory");
    } else {
      for (size_t i = 0; i < nx; ++i) {
        for (size_t j = 0; j < nx; ++j) {
          double a = A_host[i * nx + j], q = Q_host[i * nx + j];
          for (int l = 0; l < nu; ++l) {
            a -= B_host[i * nu + l] * K_host[l * nx + j];
            q -= M_host[i * nu + l] * K_host[l * nx + j] + K_host[l * nx + i] * M_host[j * nu + l];
            for (int r = 0; r < nu; ++r) q += K_host[l * nx + i] * R_host[l * nu + r] * K_host[r * nx + j];
          }
          Ao[i * nx + j] = a;
          Qo[i * nx + j] = q;
        }
        for (int j = 0; j < nu; ++j) {
          double m = M_host[i * nu + j];
          for (int l = 0; l < nu; ++l) m -= K_host[l * nx + i] * R_host[l * nu + j];
          Mo[i * nu + j] = m;
        }
      }
      for (size_t i = 0; i < nx; ++i)      // symmetric by construction; remove the rounding asymmetry
        for (size_t j = i + 1; j < nx; ++j) Qo[i * nx + j] = Qo[j * nx + i] = 0.5 * (Qo[i * nx + j] + Qo[j * nx + i]);
      rc = upload(&h->iAo, Ao, nx * nx);
      if (rc == 0) rc = upload(&h->iQo, Qo, nx * nx);
      if (rc == 0) rc = upload(&h->iMo, Mo, nx * nu);
    }
    delete[] Ao; delete[] Qo; delete[] Mo;
  }
  if (rc == 0 && (cudaMalloc((void**)&h->counts, 4 * sizeof(int)) != cudaSuccess ||
                  cudaMalloc((void**)&h->iter_sum, sizeof(unsigned long long)) != cudaSuccess ||
                  cudaMallocHost((void**)&h->h_pinned, 8 * sizeof(int)) != cudaSuccess))
    rc = set_error(NNMPC_ERR_NOMEM, "nnmpc_qp_create_ipm: allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
  if (rc < 0) {
    cudaGetLastError();
    nnmpc_qp_destroy(h);
    return rc;
  }
  *out = h;
  return 0;
}

}  // extern "C"
