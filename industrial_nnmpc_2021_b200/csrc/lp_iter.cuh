// Mixed-precision Douglas-Rachford iteration of the regulator QP: epilogues for the tcgen05
// split-operator GEMM (lp_gemm.cuh) and the small FP64 kernels around the FP64 anchors.
//
// State per sample (row), all FP64 unless noted:
//   V     Douglas-Rachford state v                      X     x = Top w_lp - c  (tracked incrementally)
//   E     fp32: w - w_lp, the part of the operand the fp16 increments have not delivered yet
//   D     fp16: scaled increment s_row (w_lp+ - w_lp) = the A operand of the next tensor-core pass
// One pass:  x += (T1 + T2) dq / (s_T s_row);  d = x - clip(v);  v += alpha d;
//            dw = (2 clip(v) - v) - w_lp;  dq = fp16(s_row' dw);  w_lp += dq / s_row'
// Deferred second operator term (s_mode != 0): the pass multiplies T1 only, and the 2^-11-relative correction T2 dq is
// delivered every m-th pass for all increments since the last delivery at once - T2 is linear, so nothing is lost,
// only delayed (like E): S (fp16, laid out like D, own per-row power-of-two scale sS) holds the pending sum
// sum_j dq_j, a one-term GEMM  x += T2 S / (s_T sS)  (EpiAddX) delivers it, and the next pass starts a new sum.
// MMA work per pass falls from 2 to 1 + 1/m products; the board is power capped in this kernel
// (profiles/r02n_pass_energy_diagnosis.md), so joules are what the pass time is made of.
// Fixed points are exactly those of the FP64 iteration in qp.cu (E -> 0, dq -> 0).  What the fp16
// operator split and the fp32 accumulation lose is proportional to |w_lp - w_anchor|; an FP64
// anchor GEMM (x = Top w - c with w_lp := w, E := 0) resets it, and every returned point is
// checked with P in FP64, so the reference tolerances (/root/repo/BASELINE.json north_star:
// KKT <= 1e-8) are certified by FP64 arithmetic, not by the fp16 path.
#pragma once
#include "lp.cuh"
#include "lp_gemm.cuh"

namespace nnmpc {

// probe variants (tools/probes/lp_pass_split.py): drop the state loads / the state stores of the epilogue
#ifndef NNMPC_EPI_PREFETCH
#define NNMPC_EPI_PREFETCH 1
#endif
#ifndef NNMPC_PROBE_NOLOAD
#define NNMPC_PROBE_NOLOAD 0
#endif
#ifndef NNMPC_PROBE_NOSTORE
#define NNMPC_PROBE_NOSTORE 0
#endif
// (ring depths: 192 KB of operand stages next to the epilogue's staging blocks; the 16-warp build - twice the staging
//  blocks - runs one stage shallower)
constexpr int LP_SH = lp::EPI_WARPS == 16 ? 1 : 0;
using LpTileN128 = lp::LpTile<128, 4 - LP_SH>;
using LpTileM256 = lp::LpTile<128, 3 - LP_SH, 2>;     // 256 x 128 outputs per CTA tile: operator bytes per flop halved
// one operator term per pass (deferred second term): a stage is A + B1
using LpTile1N128 = lp::LpTile<128, 6 - LP_SH, 1, 1>;
using LpTile1M256 = lp::LpTile<128, 4 - LP_SH, 2, 1>;

// one element of the Douglas-Rachford delta update (shared by the tensor-core epilogue and k_dr_first)
__device__ __forceinline__ void dr_delta_one(double& x, double& v, double wl, double l, double u, double alpha,
                                             double& dw, double& dabs) {
  const double z0 = clipd(v, l, u);
  const double d = x - z0;
  v += alpha * d;
  const double z1 = clipd(v, l, u);
  dw = (2.0 * z1 - v) - wl;
  dabs = fabs(d);
}
__device__ __forceinline__ __half quantise_dw(double dw, double s, double inv_s, float& e) {
  double t = dw * s;
  t = fmin(fmax(t, -60000.0), 60000.0);          // saturate: the residual e carries what did not fit
  const __half q = __double2half(t);
  e = (float)(dw - (double)__half2float(q) * inv_s);
  return q;
}

// The tensor-core epilogue is bound by instruction issue (8 warps, ~100 instructions per element before this
// form): fmin/fmax on doubles expand into DSETP + four selects + NaN fix-ups each, so the epilogue clips with
// compare/select (a NaN stays a NaN and is caught by the residual check) and clamps the quantised value in fp32.
__device__ __forceinline__ double clip_sel(double v, double l, double u) {
  const double r = v < l ? l : v;
  return r > u ? u : r;
}
__device__ __forceinline__ void dr_delta_fast(double& x, double& v, double z0, double wl, double l, double u, double alpha,
                                              double& dw, double& dabs) {
  const double d = x - z0;
  v += alpha * d;
  const double z1 = clip_sel(v, l, u);
  dw = (2.0 * z1 - v) - wl;
  dabs = fabs(d);
}
__device__ __forceinline__ __half quantise_dw_fast(double dw, double s, double inv_s, float& e) {
  float tf = (float)(dw * s);
  tf = fminf(fmaxf(tf, -60000.f), 60000.f);      // saturate: the residual e carries what did not fit
  const __half q = __float2half_rn(tf);          // any rounding will do: e is formed from the q actually sent
  e = (float)(dw - (double)__half2float(q) * inv_s);
  return q;
}

// ---- epilogue of the tensor-core pass: the whole iteration on the accumulator registers ----------
// Warp-collective (see lp_gemm.cuh): the warp owns 32 rows; TMEM hands lane l the CW accumulators of row l, the
// block is transposed through shared memory, and lane (rg = l / LPR, cp = l % LPR), LPR = CW / 2 lanes per row,
// then updates the column pair {2cp, 2cp + 1} of rows rg, rg + RG, rg + 2 RG, ... (RG = 32 / LPR rows per
// instruction).  With CW = 16 one warp instruction touches 4 rows x one full 128-byte line of FP64 state each (round
// 1 touched 8 rows x 64 bytes: twice the L1 wavefronts per request - the LSU data pipe ran at 45 %), every access is
// whole 32-byte sectors, and all loads of a step are in flight before the first use.
struct EpiDelta {
  struct Params {
    double* X;
    double* V;
    float* E;
    __half* Dn;          // next operand (the TMA reads the current one)
    long long ldd;       // row stride of Dn (elements)
    const double* lb;
    const double* ub;    // B x nu
    const int* state;    // row takes part iff state[row] == iter_state
    int iter_state;
    const int* list_r;   // position (row of the operand the TMA reads) -> sample row; null = identity
    const int* pos_w;    // sample row -> position in the operand written now; null = identity
    const double* sc_in;   // scale the current operand row was quantised with
    const double* sc_out;  // scale for the operand written now
    unsigned long long* dres;  // per row: max |d| (bit pattern of a non-negative double)
    // deferred second term (s_mode: 0 = off, 1 = add this pass's increment to the pending sum, 2 = start a new sum)
    const __half* Sc;    // pending sums, laid out like the operand the TMA reads
    __half* Sn;          // ... like the operand written now
    double* sS;          // per sample row: scale of its pending sum
    int s_mode;
    int n, nu;
    double alpha;
    double inv_sT;       // 1 / operator scale
  };
  static constexpr int LPR = lp::CW / 2;     // lanes per row
  static constexpr int RG = 32 / LPR;        // rows per warp instruction
  static constexpr int NI = 32 / RG;         // row iterations = column pairs per lane
  Params p;
  lp::EpiWarpSmem* sm;
  int lane, rg, cp;
  int pos0;                // operand position of the warp's first row in this tile
  float dmax[NI];          // per row: max |d| (fp32 is plenty for a trigger; NaN survives)
  __device__ EpiDelta(const Params& p_, lp::EpiWarpSmem* sm_, int lane_)
      : p(p_), sm(sm_), lane(lane_), rg(lane_ / LPR), cp(lane_ % LPR) {}
  __device__ void begin_tile(int pos0_, int M) {
    pos0 = pos0_;
    const int pos = pos0 + lane;
    lp::EpiRowInfo ri;
    ri.row = -1; ri.pw = 0; ri.inv_in = 0.0; ri.s_out = 0.0; ri.inv_out = 0.0; ri.g = 0.f; ri.boff = 0; ri.xoff = 0; ri.doff = 0;
    if (pos < M) {
      const int row = p.list_r ? p.list_r[pos] : pos;
      if (p.state[row] == p.iter_state) {
        ri.row = row;
        ri.pw = p.pos_w ? p.pos_w[row] : row;
        ri.inv_in = p.inv_sT / p.sc_in[row];
        ri.s_out = p.sc_out[row];
        ri.inv_out = 1.0 / ri.s_out;
        // a new sum is kept at 1/8 of the operand scale: head room for the increments that follow
        if (p.s_mode == 2) ri.g = 0.125f;
        else if (p.s_mode == 1) ri.g = (float)(p.sS[row] * ri.inv_out);
        ri.boff = row * p.nu;
        ri.xoff = (long long)row * p.n;
        ri.doff = (long long)ri.pw * p.ldd;
      }
    }
    __syncwarp();            // the previous tile's last reads of info[] are done
    sm->info[lane] = ri;
#pragma unroll
    for (int i = 0; i < NI; ++i) dmax[i] = 0.f;
    __syncwarp();
  }
  // one column pair of one row
  __device__ __forceinline__ void pair(double2& x, double2& v, float2& e, float a0, float a1, double2 l, double2 u,
                                       const lp::EpiRowInfo& ri, __half2& q, float& dm, bool valid = true) {
    x.x += (double)a0 * ri.inv_in;
    x.y += (double)a1 * ri.inv_in;
    const double z00 = clip_sel(v.x, l.x, u.x), z01 = clip_sel(v.y, l.y, u.y);
    const double wl0 = (2.0 * z00 - v.x) - (double)e.x;
    const double wl1 = (2.0 * z01 - v.y) - (double)e.y;
    double dw0, dw1, d0, d1;
    dr_delta_fast(x.x, v.x, z00, wl0, l.x, u.x, p.alpha, dw0, d0);
    dr_delta_fast(x.y, v.y, z01, wl1, l.y, u.y, p.alpha, dw1, d1);
    const __half q0 = quantise_dw_fast(dw0, ri.s_out, ri.inv_out, e.x);
    const __half q1 = quantise_dw_fast(dw1, ri.s_out, ri.inv_out, e.y);
    q = __halves2half2(q0, q1);
    // a NaN in d, or a non-finite residual e (v or E not finite while d is), makes the row's residual NaN (0 e = +-0
    // otherwise, and a + +-0 = a for a >= 0: finite residuals are unchanged)
    const float a = fmaf(0.f, e.x, fmaf(0.f, e.y, nan_max((float)d0, (float)d1)));
    if (valid) dm = nan_max(dm, a);                      // lanes that ran on a stand-in row must not touch the residual
  }

  // ---- the chunk as a software pipeline over QUARTERS (QR = NI / 4 row iterations = 2 rows x 2 columns per lane) ----
  // The loads of a quarter (state, pending sum, bounds: 38 registers) are issued one quarter ahead of their use, across
  // chunk boundaries, so every DRAM / L2 round trip is covered by the arithmetic of the quarter before it; an L2
  // prefetch runs one chunk ahead of that.  History (profiles/r02n_pass_energy_diagnosis.md, r02p_*): the per-row loop
  // of round 2h paid one exposed bounds round trip per row; loads under `if (row >= 0)` were serialised by the
  // compiler's placement of the conversions; with everything loaded at the top of the chunk the pass was still one
  // exposed round trip per chunk and warp (epilogue alone 0.88 ms against 0.47 ms without its loads).
  // Rows that do not take part (and lanes beyond N) read row 0 / column 0 and are dropped at the stores.
  static constexpr int QR = NI / 4;
  struct QLoad {
    double2 x[QR], v[QR], l[QR], u[QR];
    float2 e[QR];
    __half2 so[QR];
  };
  QLoad qa;                // the quarter(s) in flight between two chunk() calls
#ifndef NNMPC_EPI_DEPTH
#define NNMPC_EPI_DEPTH 1   // quarters the loads run ahead of their use (2: three quarters of registers in flight)
#endif
#if NNMPC_EPI_DEPTH == 2
  QLoad qn;
#endif
  template <int QI>
  __device__ __forceinline__ void issue(int col0, int N, QLoad& q) const {
    const int cbase = col0 + 2 * cp;       // n is even: the pair is inside when its first column is
    const int cb = cbase < N ? cbase : 0;
    // the chunk (col0 is a multiple of CW) lies inside one stage when the stage width is a multiple of CW
    const int k0 = cb % p.nu;
    const int k1 = (k0 + 1 == p.nu) ? 0 : k0 + 1;          // wraps to stage input 0 when nu is odd
    const bool vec = (p.nu & 1) == 0 && ((reinterpret_cast<uintptr_t>(p.lb) | reinterpret_cast<uintptr_t>(p.ub)) & 15) == 0;
#pragma unroll
    for (int j = 0; j < QR; ++j) {
      const int r = rg + RG * (QI * QR + j);
      const long long base = sm->info[r].xoff + cb;
#if NNMPC_PROBE_NOLOAD
      q.x[j] = make_double2(0.0, (double)base * 1e-300);
      q.v[j] = make_double2(0.0, 0.0);
      q.e[j] = make_float2(0.f, 0.f);
#else
      q.x[j] = __ldcs(reinterpret_cast<const double2*>(p.X + base));
      q.v[j] = __ldcs(reinterpret_cast<const double2*>(p.V + base));
      q.e[j] = __ldcs(reinterpret_cast<const float2*>(p.E + base));
#endif
      // pending sum of this row and column pair (operand position = tile row; the buffers are padded to whole tiles)
      q.so[j] = __float2half2_rn(0.f);
      if (p.s_mode == 1) q.so[j] = *reinterpret_cast<const __half2*>(p.Sc + (long long)(pos0 + r) * p.ldd + cb);
      const double* lbr = p.lb + sm->info[r].boff;
      const double* ubr = p.ub + sm->info[r].boff;
      if (vec) {
        q.l[j] = __ldg(reinterpret_cast<const double2*>(lbr + k0));
        q.u[j] = __ldg(reinterpret_cast<const double2*>(ubr + k0));
      } else {
        q.l[j] = make_double2(__ldg(lbr + k0), __ldg(lbr + k1));
        q.u[j] = make_double2(__ldg(ubr + k0), __ldg(ubr + k1));
      }
    }
  }
  template <int QI>
  __device__ __forceinline__ void update_store(int col0, int N, QLoad& q) {
    const int cbase = col0 + 2 * cp;
    const bool in = cbase < N;
    __half2 qh[QR];
    // no branch around the arithmetic: the rows of a quarter interleave
#pragma unroll
    for (int j = 0; j < QR; ++j) {
      const int r = rg + RG * (QI * QR + j);
      const lp::EpiRowInfo ri = sm->info[r];
      pair(q.x[j], q.v[j], q.e[j], sm->stg[(2 * cp) * lp::STG_LD + r], sm->stg[(2 * cp + 1) * lp::STG_LD + r], q.l[j], q.u[j],
           ri, qh[j], dmax[QI * QR + j], in && ri.row >= 0);
    }
#pragma unroll
    for (int j = 0; j < QR; ++j) {
      const int r = rg + RG * (QI * QR + j);
      if (!in || sm->info[r].row < 0 || (NNMPC_PROBE_NOSTORE && q.x[j].x != 123.456)) continue;
      const long long base = sm->info[r].xoff + cbase;
      __stcs(reinterpret_cast<double2*>(p.X + base), q.x[j]);
      __stcs(reinterpret_cast<double2*>(p.V + base), q.v[j]);
      __stcs(reinterpret_cast<float2*>(p.E + base), q.e[j]);
      const long long o = sm->info[r].doff + cbase;
      *reinterpret_cast<__half2*>(p.Dn + o) = qh[j];       // the fp16 increment goes straight to the operand the next pass reads
      if (p.s_mode) {      // pending sum of the second operator term: S+ = S + g dq, saturating (what saturates is lost to
                           // the fp16 path only: the exact check certifies every returned point)
        const float g = sm->info[r].g;
        const float2 so = __half22float2(q.so[j]), qf = __half22float2(qh[j]);
        const float s0 = fminf(fmaxf(fmaf(qf.x, g, so.x), -65504.f), 65504.f);
        const float s1 = fminf(fmaxf(fmaf(qf.y, g, so.y), -65504.f), 65504.f);
        *reinterpret_cast<__half2*>(p.Sn + o) = __floats2half2_rn(s0, s1);
      }
    }
  }
  // start of a row block: the first quarter of its first chunk
#if NNMPC_EPI_DEPTH == 2
  __device__ __forceinline__ void prime(int col0, int N) {
    issue<0>(col0, N, qa);
    issue<1>(col0, N, qn);
  }
  __device__ void chunk(int col0, const uint32_t (&acc)[lp::CW], int N, int next_col0) {
#pragma unroll
    for (int c = 0; c < lp::CW; ++c) sm->stg[c * lp::STG_LD + lane] = __uint_as_float(acc[c]);
    __syncwarp();
    // on entry quarter 0 is in qa and quarter 1 in qn; on exit the next chunk's quarters 0 and 1 are
    QLoad qc;
    issue<2>(col0, N, qc);
    update_store<0>(col0, N, qa);
    issue<3>(col0, N, qa);
    update_store<1>(col0, N, qn);
    if (next_col0 >= 0) issue<0>(next_col0, N, qn);
    update_store<2>(col0, N, qc);
    if (next_col0 >= 0) issue<1>(next_col0, N, qc);
    update_store<3>(col0, N, qa);
    qa = qn;
    qn = qc;
    __syncwarp();            // stg is rewritten by the next step
  }
#else
  __device__ __forceinline__ void prime(int col0, int N) { issue<0>(col0, N, qa); }
  __device__ void chunk(int col0, const uint32_t (&acc)[lp::CW], int N, int next_col0) {
    // transpose: stg[c][r], leading dimension STG_LD: conflict-free writes and reads
#pragma unroll
    for (int c = 0; c < lp::CW; ++c) sm->stg[c * lp::STG_LD + lane] = __uint_as_float(acc[c]);
    __syncwarp();
    QLoad qb;
    issue<1>(col0, N, qb);
    update_store<0>(col0, N, qa);
    issue<2>(col0, N, qa);
    update_store<1>(col0, N, qb);
    issue<3>(col0, N, qb);
    update_store<2>(col0, N, qa);
    if (next_col0 >= 0) issue<0>(next_col0, N, qa);
    update_store<3>(col0, N, qb);
    __syncwarp();            // stg is rewritten by the next step
  }
#endif
  // L2 prefetch of the state of the NEXT chunk of this warp (lane = row): the loads of a chunk are one exposed DRAM round
  // trip per chunk and warp, and with two warps per scheduler nothing else covers it.  No registers held.
  __device__ __forceinline__ void prefetch(int col0, int N) const {
#if NNMPC_EPI_PREFETCH
    const int row = sm->info[lane].row;
    if (row < 0 || col0 >= N) return;
    const long long base = (long long)row * p.n + col0;
    const int last = (col0 + lp::CW <= N ? lp::CW : N - col0) - 1;
    const char* px = reinterpret_cast<const char*>(p.X + base);
    const char* pv = reinterpret_cast<const char*>(p.V + base);
    const char* pe = reinterpret_cast<const char*>(p.E + base);
    asm volatile("prefetch.global.L2 [%0];" ::"l"(px));
    asm volatile("prefetch.global.L2 [%0];" ::"l"(pv));
    asm volatile("prefetch.global.L2 [%0];" ::"l"(pe));
    if ((reinterpret_cast<uintptr_t>(px) & 127) + 8 * last >= 128) {       // rows that are not 128-byte aligned straddle lines
      asm volatile("prefetch.global.L2 [%0];" ::"l"(px + 8 * last));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(pv + 8 * last));
    }
    if ((reinterpret_cast<uintptr_t>(pe) & 127) + 4 * last >= 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(pe + 4 * last));
#endif
  }
  __device__ void end_tile() {
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      float m = dmax[i];
      // the LPR lanes of a row group hold disjoint columns of the same rows; NaN must survive the reduction
#pragma unroll
      for (int o = 1; o < LPR; o <<= 1) {
        m = nan_max(m, __shfl_xor_sync(0xffffffffu, m, o));
      }
      const int row = sm->info[rg + RG * i].row;
      if (cp == 0 && row >= 0) {
        // (every column tile of the row writes the same value)
        if (p.s_mode == 2) p.sS[row] = 0.125 * sm->info[rg + RG * i].s_out;
        double md = (double)m;
        if (!(m <= 3.0e38f)) md = __longlong_as_double(0x7ff0000000000000ll);   // NaN/Inf must not look converged
        atomicMax(p.dres + row, (unsigned long long)__double_as_longlong(md));
      }
    }
  }
};

// ---- delivery of the deferred second operator term:  x += T2 S / (s_T sS)  for the iterating rows ----------------
// Same warp-collective shape as EpiDelta (transpose through shared memory, one warp instruction = 4 rows x 128 bytes).
struct EpiAddX {
  struct Params {
    double* X;
    const int* state;
    int iter_state;
    const int* list_r;   // operand position -> sample row; null = identity
    const double* sS;    // per sample row: scale of its pending sum
    int n;
    double inv_sT;
  };
  static constexpr int LPR = lp::CW / 2, RG = 32 / LPR, NI = 32 / RG;
  Params p;
  lp::EpiWarpSmem* sm;
  int lane, rg, cp;
  __device__ EpiAddX(const Params& p_, lp::EpiWarpSmem* sm_, int lane_)
      : p(p_), sm(sm_), lane(lane_), rg(lane_ / LPR), cp(lane_ % LPR) {}
  __device__ void begin_tile(int pos0, int M) {
    const int pos = pos0 + lane;
    lp::EpiRowInfo ri;
    ri.row = -1; ri.pw = 0; ri.inv_in = 0.0; ri.s_out = 0.0; ri.inv_out = 0.0; ri.g = 0.f; ri.boff = 0; ri.xoff = 0; ri.doff = 0;
    if (pos < M) {
      const int row = p.list_r ? p.list_r[pos] : pos;
      if (p.state[row] == p.iter_state) {
        ri.row = row;
        ri.inv_in = p.inv_sT / p.sS[row];
      }
    }
    __syncwarp();
    sm->info[lane] = ri;
    __syncwarp();
  }
  __device__ void chunk(int col0, const uint32_t (&acc)[lp::CW], int N) {
#pragma unroll
    for (int c = 0; c < lp::CW; ++c) sm->stg[c * lp::STG_LD + lane] = __uint_as_float(acc[c]);
    __syncwarp();
    const int cbase = col0 + 2 * cp;
    const bool in = cbase < N;
    double2 x[NI];
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int row = in ? sm->info[rg + RG * i].row : -1;
      x[i] = *reinterpret_cast<const double2*>(p.X + (long long)(row >= 0 ? row : 0) * p.n + (in ? cbase : 0));
    }
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int r = rg + RG * i;
      const int row = in ? sm->info[r].row : -1;
      const double inv = sm->info[r].inv_in;
      x[i].x += (double)sm->stg[(2 * cp) * lp::STG_LD + r] * inv;
      x[i].y += (double)sm->stg[(2 * cp + 1) * lp::STG_LD + r] * inv;
      if (row >= 0) *reinterpret_cast<double2*>(p.X + (long long)row * p.n + cbase) = x[i];
    }
    __syncwarp();
  }
  __device__ void end_tile() {}
};

// plain store (self test): C = scale * acc
struct EpiLpStore {
  struct Params {
    double* C;
    long long ldc;
    double scale;
  };
  Params p;
  int lane, row;
  bool ok;
  __device__ EpiLpStore(const Params& p_, lp::EpiWarpSmem*, int lane_) : p(p_), lane(lane_), row(0), ok(false) {}
  __device__ void begin_tile(int pos0, int M) {
    row = pos0 + lane;
    ok = row < M;
  }
  __device__ void chunk(int col0, const uint32_t (&acc)[lp::CW], int N) {
    if (!ok) return;
#pragma unroll
    for (int j = 0; j < lp::CW; ++j)
      if (col0 + j < N) p.C[(long long)row * p.ldc + col0 + j] = (double)__uint_as_float(acc[j]) * p.scale;
  }
  __device__ void end_tile() {}
};

// ---- FP64 anchor: x = Top w - c on the accumulators of the DMMA GEMM ---------------------------
struct EpiAnchor {
  struct Params {
    double* X;
    const double* C;
    int n;
  };
  Params p;
  __device__ EpiAnchor(const Params& p_, int, int) : p(p_) {}
  __device__ void begin_row() {}
  __device__ void apply(int pr, int, int col, double a0, double a1, bool ok0, bool ok1) {
    if (!ok0) return;
    const long long off = (long long)pr * p.n + col;
    if (ok1) {
      const double2 c = *reinterpret_cast<const double2*>(p.C + off);
      *reinterpret_cast<double2*>(p.X + off) = make_double2(a0 - c.x, a1 - c.y);
    } else {
      p.X[off] = a0 - p.C[off];
    }
  }
  __device__ void finish_row(int, int, int, bool) {}
};

// operator split: T1 = fp16(s Top), T2 = fp16(s Top - T1)  (same scale: both products share one accumulator)
__global__ void k_split_f16(const double* __restrict__ T, int n, long long ldh, double s, __half* __restrict__ T1,
                            __half* __restrict__ T2) {
  const long long total = (long long)n * ldh;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const long long r = i / ldh;
    const int c = (int)(i - r * ldh);
    double t = c < n ? T[r * n + c] * s : 0.0;
    const __half h1 = __double2half(t);
    const __half h2 = __double2half(t - (double)__half2float(h1));
    T1[i] = h1;
    T2[i] = h2;
  }
}

// anchor rows: the FP64 operand w = 2 clip(v) - v, nothing outstanding (E = 0)
__global__ void k_anchor_prep(const int* __restrict__ rows, const int* __restrict__ count, const double* __restrict__ V,
                              double* __restrict__ W, float* __restrict__ E, const double* __restrict__ lb,
                              const double* __restrict__ ub, int n, int nu) {
  const int cnt = *count;
  for (int li = blockIdx.x; li < cnt; li += gridDim.x) {
    const long long s = rows[li];
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
      const int k = j % nu;
      const double v = V[s * n + j];
      W[s * n + j] = 2.0 * clipd(v, lb[s * nu + k], ub[s * nu + k]) - v;
      E[s * n + j] = 0.f;
    }
  }
}

// anchor rows after the FP64 GEMM: one full-precision Douglas-Rachford step from the exact x, then the
// first fp16 increment with a scale taken from the row's own max |dw| (one CTA per row)
__global__ void __launch_bounds__(256)
k_dr_first(const int* __restrict__ rows, const int* __restrict__ count, double* __restrict__ X, double* __restrict__ V,
           double* __restrict__ W, float* __restrict__ E, __half* __restrict__ D, long long ldd,
           const double* __restrict__ lb, const double* __restrict__ ub, double* __restrict__ sc_in,
           double* __restrict__ sc_out, int* __restrict__ state, int* __restrict__ it, int iter_state, int n, int nu,
           double alpha, const int* __restrict__ pos_r, unsigned char* __restrict__ need2, __half* __restrict__ S,
           double* __restrict__ sS) {
  __shared__ double red[2][8];
  const int cnt = *count;
  for (int li = blockIdx.x; li < cnt; li += gridDim.x) {
  const long long s = rows[li];
  double dmax = 0.0, wmax = 0.0;
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    const int k = j % nu;
    const double l = lb[s * nu + k], u = ub[s * nu + k];
    double x = X[s * n + j], v = V[s * n + j], dw, a;
    dr_delta_one(x, v, W[s * n + j], l, u, alpha, dw, a);
    V[s * n + j] = v;
    W[s * n + j] = dw;                    // staged for the second pass
    dmax = nan_max(dmax, a);
    wmax = nan_max(wmax, fabs(dw));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    dmax = nan_max(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
    wmax = nan_max(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
  }
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = dmax;
    red[1][threadIdx.x >> 5] = wmax;
  }
  __syncthreads();
  dmax = red[0][0];
  wmax = red[1][0];
  for (int w = 1; w < 8; ++w) {
    dmax = nan_max(dmax, red[0][w]);
    wmax = nan_max(wmax, red[1][w]);
  }
  const double sq = pow2_scale(wmax), inv = 1.0 / sq;
  const long long dpos = pos_r ? pos_r[s] : s;      // row of the operand buffer the next pass reads for this sample
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    float e;
    const __half q = quantise_dw(W[s * n + j], sq, inv, e);
    if (dpos >= 0) D[dpos * ldd + j] = q;
    if (S && dpos >= 0) S[dpos * ldd + j] = __float2half_rn(0.125f * __half2float(q));    // deferred second term: the pending sum starts
    E[s * n + j] = e;
  }
  if (threadIdx.x == 0) {
    if (sS) sS[s] = 0.125 * sq;
    sc_in[s] = sq;
    sc_out[s] = pow2_scale(3.0 * alpha * dmax);
    state[s] = iter_state;
    it[s] += 1;
    if (need2 && dpos >= 0) need2[dpos >> 7] = 1;     // a QP starts with large increments: both operator terms
  }
  __syncthreads();          // red[] is reused by the next row
  }
}

// ---- re-anchoring from a failed exact check (no FP64 anchor GEMM) -------------------------------
// The check computes g = P z + q in FP64 for z = clip(v).  With w_lp := z + g / rho the tracked quantity
// x = Top w_lp - c = (P + D)^-1 (D z + P z) = z holds EXACTLY, so the check itself re-anchors the fp16 path:
// x := z, and what is left to deliver is w - w_lp = (z - v) - g / rho, which vanishes at the solution - the
// operator-split and fp32-accumulation errors of delivering it are relative to a vanishing quantity.
__global__ void k_reanchor(const int* __restrict__ rows, const int* __restrict__ count, const int* __restrict__ state,
                           int emit_state, const double* __restrict__ Z, double* __restrict__ GW,
                           const double* __restrict__ rinv, double* __restrict__ X, int n) {
  const int cnt = *count;
  for (int li = blockIdx.x; li < cnt; li += gridDim.x) {
    const long long s = rows[li];
    if (state[s] != emit_state) continue;
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
      const double z = Z[s * n + j];
      GW[s * n + j] = z + GW[s * n + j] * rinv[j];          // g -> w_lp
      X[s * n + j] = z;
    }
  }
}

// Rows in `emit_state` (one CTA per row): first fp16 increment from the exactly anchored (x, w_lp):
//   dw = (2 clip(v) - v) - w_lp  -> operand row of the next tensor-core pass, quantisation residual into E.
// The scale of the operand the next pass WRITES is a guess from the ||d|| that triggered the check plus the
// increment itself (k_select takes over from the measured ||d|| after that pass; a guess that is too small only
// saturates the increment, whose remainder E carries forward).
__global__ void __launch_bounds__(256)
k_lp_emit(const int* __restrict__ rows, const int* __restrict__ count, int* __restrict__ state, int emit_state,
          int iter_state, const double* __restrict__ V, double* __restrict__ WL, float* __restrict__ E,
          __half* __restrict__ D, long long ldd, const double* __restrict__ lb, const double* __restrict__ ub,
          double* __restrict__ sc_in, double* __restrict__ sc_out, const double* __restrict__ dtrig, int n, int nu,
          double alpha, const int* __restrict__ pos_r, unsigned char* __restrict__ need2, __half* __restrict__ S,
          double* __restrict__ sS) {
  __shared__ double red[8];
  const int cnt = *count;
  for (int li = blockIdx.x; li < cnt; li += gridDim.x) {
  const long long s = rows[li];
  if (state[s] != emit_state) continue;          // uniform over the CTA
  double wmax = 0.0;
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    const int k = j % nu;
    const double v = V[s * n + j];
    const double z = clipd(v, lb[s * nu + k], ub[s * nu + k]);
    const double dw = (2.0 * z - v) - WL[s * n + j];
    WL[s * n + j] = dw;                   // staged for the second pass
    wmax = nan_max(wmax, fabs(dw));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) wmax = nan_max(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = wmax;
  __syncthreads();
  wmax = red[0];
  for (int w = 1; w < 8; ++w) wmax = nan_max(wmax, red[w]);
  const double sq = pow2_scale(wmax), inv = 1.0 / sq;
  const long long dpos = pos_r ? pos_r[s] : s;      // row of the operand buffer the next pass reads for this sample
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    float e;
    const __half q = quantise_dw(WL[s * n + j], sq, inv, e);
    if (dpos >= 0) D[dpos * ldd + j] = q;
    if (S && dpos >= 0) S[dpos * ldd + j] = __float2half_rn(0.125f * __half2float(q));
    E[s * n + j] = e;
  }
  if (threadIdx.x == 0) {
    if (sS) sS[s] = 0.125 * sq;
    sc_in[s] = sq;
    sc_out[s] = pow2_scale(3.0 * alpha * (dtrig[s] + wmax));
    state[s] = iter_state;
    // a re-anchored row restarts from the gradient of a failed check: its first increments are not small
    if (need2 && dpos >= 0) need2[dpos >> 7] = 1;
  }
  __syncthreads();          // red[] is reused by the next row
  }
}

}  // namespace nnmpc
