// Closed-loop offline data generation for B trajectories at once, as a continuously batched engine.
//
// Replaces simulate_offline (/root/reference/lib/linearMPC.py:827-880) run in one OS process per
// trajectory chunk (:803-825).  Every trajectory ("slot") repeats, at its own pace,
//     target selector (:851) -> regulator QP (:853) -> u = useq[0:nu] (:856) -> x+ = Ax+Bu+Bd d (:860)
// and the only coupling between slots is that they share the dense operators.  The reference (and a
// lock-step batch) waits for the slowest QP of a step; here a slot whose QP has converged
// immediately advances to its next time step and keeps iterating in place, so the iteration GEMM
// always runs over every live trajectory (full tiles) and the cost per sample is the MEAN iteration
// count, not the maximum over the batch.
//
// One engine loop (all launches stream ordered, row lists and their lengths live on the device):
//   1. iteration GEMM over the active list (EpiAdmm: DR update + ||d||_inf per row); in mixed precision the
//      tcgen05 fp16 pass (lp_gemm.cuh), preceded on full loops by the exact anchors of the rows that start a QP
//   2. k_select:   rows with kappa*||d||_inf <= tol (or at max_iter) become candidates
//   3. k_make_z + verification GEMM on the candidates: exact KKT residual with P (FP64 DMMA, or the INT8-sliced
//      FP64-accurate tensor-core apply of oz_gemm.cuh in mixed precision)
//   4. k_retire:   candidates that pass are done (iters/kkt rows written), the rest keep iterating (mixed precision:
//      re-anchored from the gradient the check just computed)
//   5. k_advance_plant on the done rows: dataset row u and the plant step x+ = [A|B|Bd][x|u|d], one fused kernel
//   6. k_step:     t += 1; finished trajectories leave; the rest form the renew list
//   7. target selector (fused: dataset rows x,uprev,xs,us; x0, lb, ub; warm-start shift dus),
//      q-build GEMMs (c = Mtq x0, q = tq x0) and k_warm_shift on the renew rows
// The host only polls a finished-trajectories counter with a two-loop lag, so the GPU never waits
// for it.  Per-row results do not depend on which other rows are in the batch: every GEMM tile
// shape accumulates in the same order and every decision uses the row's own data.
#include "qp.cuh"
#include "ts.cuh"
#include "lp.cuh"

namespace nnmpc {
int qp_ensure_scratch(nnmpc_qp* h, long long B);

// SLOT_EMIT (mixed mode): x and w_lp are exact (re-anchored by an exact check), the first fp16 increment is pending
enum SlotState { SLOT_IDLE = 0, SLOT_ITER = 1, SLOT_CAND = 2, SLOT_DONE = 3, SLOT_RENEW = 4, SLOT_ANCHOR = 5, SLOT_EMIT = 6 };
enum Counter { N_ACTIVE = 0, N_CAND = 1, N_DONE = 2, N_RENEW = 3, N_FINISHED = 4, F_MAXITER = 5, N_ANCHOR = 6,
               // mixed mode: effective row counts of this loop's launches (0 switches a launch off on the device)
               E_ANCHOR = 7, E_LP = 8, E_TAIL = 9, LP_LEN0 = 10, LP_LEN1 = 11,
               // chunk queue: slots that finished a trajectory chunk this loop, cold (re)starts, next chunk to hand out
               N_SWAP = 12, N_COLD = 13, NEXT_CHUNK = 14,
               // a target-selector solve that did not reach its optimum (active-set stall or non-finite data)
               F_TS_FAIL = 15, N_COUNTERS = 16 };
constexpr int POLL_RING = 4;
}  // namespace nnmpc

struct nnmpc_sim {
  nnmpc_qp* qp;
  nnmpc_ts* ts;
  int nx, nu, nd, ny, device;
  int kin_ld;    // nx+nu+nd rounded up to even
  int nxa_ld;    // = qp->nxa
  double* ABd;   // device nx x kin_ld
  double kappa0, kappa_max;
  long long cap;
  long long warm_B;   // batch size whose solver state (V, us_prev, kappa) is valid for `resume`; 0 = none
  nnmpc::DevBuf<double> x0, lb, ub, us_prev, dus, V, Z, xcur, upcur, kappa, dtrig;
  nnmpc::DevBuf<int> state, tcur, it, lists;   // lists: 9 x cap (active, cand, done, renew, anchor, cold, swap, swap_old, swap_new)
  nnmpc::DevBuf<int> chunk, cold;              // per slot: the trajectory chunk it works on; cold (re)start pending
  int slot_cap;                                // most trajectories advanced concurrently (further chunks queue up)
  int cadence;                                 // mixed mode: the FP64 phases run every cadence-th loop
  // mixed-precision iteration (tcgen05 fp16 increments + FP64-accurate anchors / checks), see lp_iter.cuh, oz_gemm.cuh
  int mixed;
  int tail_rows;                    // live rows at or below which the mixed mode finishes in FP64 (-1 = auto)
  nnmpc::LpState lps;
  int exact_oz;                     // mixed mode: anchors and exact checks on the INT8 tensor cores (oz_gemm.cuh) instead of DMMA
  nnmpc::OzRows ozr;
  nnmpc::DevBuf<int> lp_layout;     // 2 x cap operand layouts (position -> row) + 2 x cap inverses (row -> position)
  nnmpc::DevBuf<double> dlast;      // last ||d|| per slot
  nnmpc::DevBuf<unsigned char> need2;   // per 128-row operand tile: both operator terms needed in the next pass
  double t2_factor;                 // a row is "late" when ||d|| <= t2_factor * tol (0: never skip the second term)
  int t2_every;                     // mixed mode: second fp16 operator term delivered every t2_every-th pass (0: every pass, fused)
  bool t2_auto;                     // not set by the caller: deferred only where the MMAs weigh (n >= T2_AUTO_MIN_N)
  unsigned long long* tile_stat;    // device: tensor-core tiles run with [0] one, [1] both operator terms, [2] second-term delivery tiles (cumulative)
  unsigned long long* stats;        // device: [0] anchors, [1] exact KKT checks, [2] QPs whose optimum has active bounds, [3] active bounds in total
  long long tot_rowiters, tot_anchors, tot_verifies, tot_qps, tot_qps_active, tot_active;   // since create (host)
  nnmpc::DevBuf<unsigned long long> dres, kres;
  int* counts;                      // device, N_COUNTERS ints
  unsigned long long* rowiters;     // device: [0] total row-iterations executed (flop accounting), [1] of which in the FP64 tail
  int* pin;                         // pinned: POLL_RING x N_COUNTERS ints + 2 x u64
  cudaEvent_t poll_ev[nnmpc::POLL_RING];
  // staging for the host entry point
  nnmpc::DevBuf<double> h_sp, h_dist, h_x, h_uprev, h_xs, h_us, h_u, h_kkt, h_xio, h_upio;
  nnmpc::DevBuf<int> h_iters;
  // optional sinks of the next runs (nnmpc_sim_set_capture): full optimal sequence and optimal cost of every QP
  double* cap_useq;                 // device [B][T][n] or null
  double* cap_cost;                 // device [B][T] or null
  nnmpc::DevBuf<double> gcap;       // f64 mode with capture: the gradient g = P z + q of the last check per slot
};

namespace nnmpc {

// ---- single-block list builders --------------------------------------------------------------
// Ordered (ascending position) compaction by one 1024-thread block: entries with keep != 0 are
// appended to out[] in input order; returns the new length to every thread.
__device__ int block_append(bool keep, int value, int* out, int base) {
  __shared__ int warp_tot[32];
  __shared__ int total;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned m = __ballot_sync(0xffffffffu, keep);
  if (lane == 0) warp_tot[warp] = __popc(m);
  __syncthreads();
  if (warp == 0) {
    int v = warp_tot[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += t;
    }
    warp_tot[lane] = v;   // inclusive
    if (lane == 31) total = v;
  }
  __syncthreads();
  const int woff = warp ? warp_tot[warp - 1] : 0;
  if (keep) out[base + woff + __popc(m & ((1u << lane) - 1u))] = value;
  const int t = total;
  __syncthreads();
  return base + t;
}

struct EngineArrays {
  int* state; int* tcur; int* it;
  double* kappa; double* dtrig;
  unsigned long long* dres; unsigned long long* kres;
  int* l_active; int* l_cand; int* l_done; int* l_renew; int* l_anchor;
  int* l_cold; int* l_swap; int* swap_old; int* swap_new; int* chunk; int* cold; int n_chunks;
  int* counts; unsigned long long* rowiters;
  // mixed-precision mode
  int mixed; double* sc_in; double* sc_out; unsigned long long* stats; double alpha;
  int* lp_list; int* lp_pos;   // [2][S] each
  int tail_rows;
  // one-term tensor-core tiles (lp_gemm.cuh LpShape::need2): last ||d|| per row, threshold below which a row is in
  // its late phase, per-128-row-tile flags for the next pass (null: every tile runs both operator terms)
  double* dlast; double t2_thr; unsigned char* need2;
};

// exclusive prefix of a per-thread count over one 1024-thread block; total to every thread
__device__ int block_excl_scan(int c, int& total_out) {
  __shared__ int warp_tot[32];
  __shared__ int total;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int v = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  if (lane == 31) warp_tot[warp] = v;
  __syncthreads();
  if (warp == 0) {
    int w = warp_tot[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += t;
    }
    warp_tot[lane] = w;   // inclusive over warps
    if (lane == 31) total = w;
  }
  __syncthreads();
  const int excl = v - c + (warp ? warp_tot[warp - 1] : 0);
  total_out = total;
  __syncthreads();
  return excl;
}

// after an iteration: bump iteration counters, pick the rows worth an exact KKT check
// (append: candidates of earlier passes are still waiting for their exact check - the FP64 phases of the mixed
//  mode run every `cadence`-th loop - so the list grows instead of starting over).
// Four consecutive list entries per thread and round: the dependent loads of a row (list -> state -> residual)
// overlap across the four, and the candidate list keeps the order of the live list.
// Several 1024-thread blocks share the live list (it is the one kernel between two tensor-core passes, so its latency
// is exposed): every block scans its slices and reserves a range of the candidate list with one atomicAdd per slice,
// hence the ORDER of the candidate list - not its content - varies from run to run; nothing downstream depends on
// it.  N_CAND is reset by the host-side launcher when a new list starts.  With one-term tiles enabled (need2) the
// kernel runs as a single block, because the tile flags are cleared before they are raised.
__global__ void __launch_bounds__(1024) k_select(EngineArrays e, double tol, int max_iter, int full,
                                                 const int* __restrict__ pos_next, int S) {
  constexpr int RPT = 4;
  const int na = e.counts[N_ACTIVE];
  int iterated = 0;
  // tile flags of the NEXT pass start from "one term is enough"; rows that are not in their late phase raise them
  if (e.need2)
    for (int i = threadIdx.x; i < (S + 127) / 128 + 1; i += 1024) e.need2[i] = 0;
  __syncthreads();
  __shared__ int s_base;
  for (int i0 = blockIdx.x * 1024 * RPT; i0 < na; i0 += gridDim.x * 1024 * RPT) {
    int s[RPT];
    bool live[RPT], cand[RPT];
#pragma unroll
    for (int r = 0; r < RPT; ++r) {
      const int i = i0 + threadIdx.x * RPT + r;
      s[r] = i < na ? e.l_active[i] : -1;
    }
#pragma unroll
    for (int r = 0; r < RPT; ++r) live[r] = s[r] >= 0 && e.state[s[r]] == SLOT_ITER;   // rows waiting for an exact phase did not iterate
    int nc = 0;
#pragma unroll
    for (int r = 0; r < RPT; ++r) {
      cand[r] = false;
      if (live[r]) {
        const int row = s[r];
        ++iterated;
        const int it = e.it[row] + 1;
        e.it[row] = it;
        const double d = __longlong_as_double((long long)e.dres[row]);
        e.dres[row] = 0ull;
        if (e.mixed) {   // the operand written by this pass was quantised with sc_out; pick the next scale from ||d||
          e.sc_in[row] = e.sc_out[row];
          e.sc_out[row] = pow2_scale(3.0 * e.alpha * d);
        }
        cand[r] = (e.kappa[row] * d <= tol) || it >= max_iter;
        if (e.mixed) e.dlast[row] = d;
        if (e.need2 && !cand[r] && !(d <= e.t2_thr)) {
          const int pos = pos_next[row];
          if (pos >= 0) e.need2[pos >> 7] = 1;
        }
        if (cand[r]) {
          e.state[row] = SLOT_CAND;
          e.dtrig[row] = d;
          e.kres[row] = 0ull;
          ++nc;
        }
      }
    }
    int total;
    const int excl = block_excl_scan(nc, total);
    if (threadIdx.x == 0) s_base = total ? atomicAdd(e.counts + N_CAND, total) : 0;
    __syncthreads();
    int off = s_base + excl;
#pragma unroll
    for (int r = 0; r < RPT; ++r)
      if (cand[r]) e.l_cand[off++] = s[r];
    __syncthreads();
  }
  // block-wide count of the rows that iterated
  int tot_it;
  block_excl_scan(iterated, tot_it);
  if (threadIdx.x == 0) {
    if (tot_it) {
      atomicAdd(e.rowiters, (unsigned long long)tot_it);
      if (e.mixed && e.counts[E_TAIL] > 0) atomicAdd(e.rowiters + 1, (unsigned long long)tot_it);   // of which: FP64 tail iterations
    }
    if (blockIdx.x == 0 && e.mixed && full) e.stats[0] += (unsigned long long)e.counts[E_ANCHOR];   // anchors served at the top of this loop
  }
}

// z = clip(v) for the candidate rows (one CTA per row)
__global__ void k_make_z(const int* __restrict__ rows, const int* __restrict__ count, const double* __restrict__ V,
                         double* __restrict__ Z, const double* __restrict__ lb, const double* __restrict__ ub,
                         int n, int nu) {
  const int cnt = *count;
  for (int li = blockIdx.x; li < cnt; li += gridDim.x) {
    const long long s = rows[li];
    const double* v = V + s * n;
    double* z = Z + s * n;
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
      const int k = j % nu;
      z[j] = clipd(v[j], lb[s * nu + k], ub[s * nu + k]);
    }
  }
}

// candidates whose exact KKT residual passes (or that ran out of iterations) are done
__global__ void __launch_bounds__(1024) k_retire(EngineArrays e, double tol, int max_iter, int T, int* out_iters,
                                                 double* out_kkt, double kappa_max) {
  const int nc = e.counts[N_CAND];
  int base = 0;
  for (int i0 = 0; i0 < nc; i0 += 1024) {
    const int i = i0 + threadIdx.x;
    bool done = false;
    int s = 0;
    if (i < nc) {
      s = e.l_cand[i];
      const double r = __longlong_as_double((long long)e.kres[s]);
      const double d = e.dtrig[s];
      const int it = e.it[s];
      // recalibrate this trajectory's trigger from what the exact check saw (consecutive QPs are alike)
      done = r <= tol || it >= max_iter;
      if (d > 1e-300 && r <= 1.7e308) {
        double k = fmax(1.3 * r / d, 0.7 * e.kappa[s]);
        // mixed mode: a failed check may be drift of the fp16 path (removed by the anchor that follows),
        // not a trigger that is too loose, so the trigger tightens by at most 2x per failure
        if (e.mixed && !done) k = fmin(k, 2.0 * e.kappa[s]);
        e.kappa[s] = fmin(fmax(k, 1e-6), kappa_max);
      }
      if (done) {
        e.state[s] = SLOT_DONE;
        const long long o = (long long)e.chunk[s] * T + e.tcur[s];
        if (out_iters) out_iters[o] = it;
        if (out_kkt) out_kkt[o] = r;
        if (!(r <= tol)) e.counts[F_MAXITER] = 1;
      } else {
        // mixed mode: the exact check re-anchors x (k_reanchor), the row goes on once k_lp_emit has issued
        // its first increment - no FP64 anchor GEMM
        e.state[s] = e.mixed ? SLOT_EMIT : SLOT_ITER;
      }
    }
    base = block_append(done, s, e.l_done, base);
  }
  if (threadIdx.x == 0) {
    e.counts[N_DONE] = base;
    e.counts[N_ANCHOR] = 0;   // k_step appends the rows that start a QP
    if (e.mixed) e.stats[1] += (unsigned long long)nc;   // failed checks = checks - QPs
  }
}

// First move, dataset row u and the plant step x+ = A x + B u + Bd d of the done rows, fused (linearMPC.py:856-866).
// A CTA takes ADV_ROWS done rows at a time: it stages their [x | u | d] in shared memory (writing the dataset row
// u and the new uprev on the way), then every warp streams rows of [A | B | Bd] once per group - coalesced, 8 rows
// of reuse - and reduces the dot products with shuffles.  The summation order of a row does not depend on which
// other rows share its group.  With capture sinks also the whole optimal sequence (deviation variables + us per
// stage, as DenseQPRegulator.solve returns it through get_control_sequence, linearMPC.py:689) and the optimal cost
// 1/2 z'Pz + q'z = 1/2 z'(g + q) from the gradient g = P z + q of the check that certified z.
constexpr int ADV_ROWS = 8;
constexpr int T2_AUTO_MIN_N = 1536;
constexpr int ADV_THREADS = 1024;   // 32 warps share the rows of [A|B|Bd]: the dot products are latency bound (8 warps: 32 rows each)
__global__ void __launch_bounds__(ADV_THREADS)
k_advance_plant(const int* __restrict__ rows, const int* __restrict__ count, const int* __restrict__ tcur,
                const int* __restrict__ chunk, int T, const double* __restrict__ Z, const double* __restrict__ us,
                double* __restrict__ xcur, const double* __restrict__ dist, double* __restrict__ row_u,
                double* __restrict__ upcur, const double* __restrict__ ABd, int n, int nx, int nu, int nd, int kin_ld,
                const double* __restrict__ G, const double* __restrict__ Ql, double* __restrict__ cap_useq,
                double* __restrict__ cap_cost, const double* __restrict__ lb, const double* __restrict__ ub,
                unsigned long long* __restrict__ stats) {
  extern __shared__ double adv_in[];          // ADV_ROWS x kin_ld
  __shared__ double red[ADV_THREADS / 32];
  __shared__ int row_act[ADV_ROWS];
  const int cnt = *count;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int g0 = blockIdx.x * ADV_ROWS; g0 < cnt; g0 += gridDim.x * ADV_ROWS) {
    const int nr = cnt - g0 < ADV_ROWS ? cnt - g0 : ADV_ROWS;
    for (int idx = threadIdx.x; idx < nr * kin_ld; idx += blockDim.x) {
      const int r = idx / kin_ld, c = idx - r * kin_ld;
      const long long s = rows[g0 + r];
      const long long o = (long long)chunk[s] * T + tcur[s];
      double v;
      if (c < nx) {
        v = xcur[s * nx + c];
      } else if (c < nx + nu) {
        const int k = c - nx;
        v = Z[s * n + k] + us[o * nu + k];
        row_u[o * nu + k] = v;
        upcur[s * nu + k] = v;
      } else if (c < nx + nu + nd) {
        v = dist[o * nd + (c - nx - nu)];
      } else {
        v = 0.0;
      }
      adv_in[idx] = v;
    }
    {  // workload statistics: how constrained the optimum is (z = clip(v) sits exactly on an active bound).  One flat
       // loop over the group's rows x n elements: independent, coalesced loads (a per-row loop with a block-wide vote
       // per row serialised 8 x 18 dependent load rounds and was most of this kernel's time)
      if (threadIdx.x < ADV_ROWS) row_act[threadIdx.x] = 0;
      __syncthreads();
      int na = 0;
      const int total = nr * n;
#pragma unroll 4
      for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
        const int r = idx / n, j = idx - r * n;
        const long long s = rows[g0 + r];
        const double z = Z[s * n + j];
        const bool act = z <= lb[s * nu + (j % nu)] || z >= ub[s * nu + (j % nu)];
        if (act) { ++na; row_act[r] = 1; }
      }
      na = __reduce_add_sync(0xffffffffu, na);
      if (lane == 0 && na > 0) atomicAdd(stats + 3, (unsigned long long)na);
      __syncthreads();
      if (threadIdx.x == 0) {
        int nrow = 0;
        for (int r = 0; r < nr; ++r) nrow += row_act[r];
        if (nrow) atomicAdd(stats + 2, (unsigned long long)nrow);
      }
    }
    for (int r = 0; r < nr && (cap_useq || cap_cost); ++r) {
      const long long s = rows[g0 + r];
      const long long o = (long long)chunk[s] * T + tcur[s];
      if (cap_useq)
        for (int j = threadIdx.x; j < n; j += blockDim.x) cap_useq[o * n + j] = Z[s * n + j] + us[o * nu + (j % nu)];
      if (cap_cost) {
        double acc = 0.0;
        for (int j = threadIdx.x; j < n; j += blockDim.x) acc += Z[s * n + j] * (G[s * n + j] + Ql[s * n + j]);
#pragma unroll
        for (int o2 = 16; o2 > 0; o2 >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o2);
        if (lane == 0) red[warp] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
          double t = 0.0;
          for (int w = 0; w < nwarps; ++w) t += red[w];
          cap_cost[o] = 0.5 * t;
        }
        __syncthreads();
      }
    }
    __syncthreads();                           // inputs staged (and xcur read) before any x+ is written
    for (int i = warp; i < nx; i += nwarps) {
      const double* arow = ABd + (long long)i * kin_ld;
      double acc[ADV_ROWS];
#pragma unroll
      for (int r = 0; r < ADV_ROWS; ++r) acc[r] = 0.0;
      for (int c = lane; c < kin_ld; c += 32) {
        const double a = arow[c];
#pragma unroll
        for (int r = 0; r < ADV_ROWS; ++r) acc[r] += a * adv_in[r * kin_ld + c];   // rows beyond nr hold stale finite data
      }
#pragma unroll
      for (int r = 0; r < ADV_ROWS; ++r) {
        double t = acc[r];
#pragma unroll
        for (int o2 = 16; o2 > 0; o2 >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o2);
        if (lane == 0 && r < nr) xcur[(long long)rows[g0 + r] * nx + i] = t;
      }
    }
    __syncthreads();                           // adv_in is rewritten by the next group
  }
}

// done rows move to their next time step; finished trajectories leave; rebuild renew + active lists
__global__ void __launch_bounds__(1024) k_step(EngineArrays e, int T, int S, int wbuf) {
  const int nd = e.counts[N_DONE];
  int base = 0, fin = 0;
  const int na0 = e.mixed ? e.counts[N_ANCHOR] : 0;
  int nanch = na0;
  __syncthreads();
  int nsw = 0, ncold = 0;
  for (int i0 = 0; i0 < nd; i0 += 1024) {
    const int i = i0 + threadIdx.x;
    bool renew = false, swap = false;
    int s = 0;
    if (i < nd) {
      s = e.l_done[i];
      const int t = e.tcur[s] + 1;
      e.tcur[s] = t;
      renew = t < T;
      swap = !renew;
      e.state[s] = renew ? SLOT_RENEW : SLOT_IDLE;
    }
    base = block_append(renew, s, e.l_renew, base);
    if (e.mixed) nanch = block_append(renew, s, e.l_anchor, nanch);
    nsw = block_append(swap, s, e.l_swap, nsw);
  }
  fin = nsw;
  // slots that finished their chunk take the next queued chunk (cold start at its t = 0), if any is left
  const int next0 = e.counts[NEXT_CHUNK];
  const int left = e.n_chunks - next0;
  const int ntake = nsw < left ? nsw : (left > 0 ? left : 0);
  __syncthreads();
  for (int i0 = 0; i0 < nsw; i0 += 1024) {
    const int i = i0 + threadIdx.x;
    const bool take = i < ntake;
    int s = 0;
    if (i < nsw) {
      s = e.l_swap[i];
      e.swap_old[i] = e.chunk[s];
      e.swap_new[i] = take ? next0 + i : -1;
      if (take) {
        e.chunk[s] = next0 + i;
        e.tcur[s] = 0;
        e.cold[s] = 1;
        e.state[s] = SLOT_RENEW;
      }
    }
    base = block_append(take, s, e.l_renew, base);
    if (e.mixed) nanch = block_append(take, s, e.l_anchor, nanch);
    ncold = block_append(take, s, e.l_cold, ncold);
  }
  int na = 0;
  if (e.need2) {
    // sorted by phase: rows in the late phase of their QP first, so that whole 128-row operand tiles of the next
    // layout can run with one operator term (rows only move early -> late until the next rebuild)
    for (int pass = 0; pass < 2; ++pass)
      for (int i0 = 0; i0 < S; i0 += 1024) {
        const int s = i0 + threadIdx.x;
        bool live = false, late = false;
        if (s < S) {
          const int st = e.state[s];
          live = st == SLOT_ITER || st == SLOT_RENEW || st == SLOT_ANCHOR || st == SLOT_EMIT;
          // the layout built here is read 5 to 8 passes from now: rows whose residual is within ~two decades of
          // the threshold will be late by then (rows that finish in between idle until a later rebuild)
          late = st == SLOT_ITER && e.dlast[s] <= 64.0 * e.t2_thr;
        }
        na = block_append(live && (late == (pass == 0)), s, e.l_active, na);
      }
  } else if (nd > 0) {   // only a finished chunk changes the live list, but rebuilding is cheap
    for (int i0 = 0; i0 < S; i0 += 1024) {
      const int s = i0 + threadIdx.x;
      const bool live = s < S && (e.state[s] == SLOT_ITER || e.state[s] == SLOT_RENEW || e.state[s] == SLOT_ANCHOR ||
                                  e.state[s] == SLOT_EMIT);
      na = block_append(live, s, e.l_active, na);
    }
  } else {
    na = e.counts[N_ACTIVE];
  }
  if (e.mixed) {
    // Operand layout for the pass after next = the live list of the next loop (the tensor-core operand is
    // rewritten every pass, so it is re-compacted for free, one pass behind the live list).
    int* L = e.lp_list + (long long)wbuf * S;
    int* Pp = e.lp_pos + (long long)wbuf * S;
    for (int i = threadIdx.x; i < S; i += 1024) Pp[i] = -1;
    __syncthreads();
    for (int i = threadIdx.x; i < na; i += 1024) {
      const int s = e.l_active[i];
      L[i] = s;
      Pp[s] = i;
    }
  }
  if (threadIdx.x == 0) {
    e.counts[N_RENEW] = base;
    e.counts[N_FINISHED] += fin;
    e.counts[N_ACTIVE] = na;
    e.counts[N_SWAP] = nsw;
    e.counts[N_COLD] = ncold;
    e.counts[NEXT_CHUNK] = next0 + ntake;
    if (e.mixed) {
      e.counts[N_ANCHOR] = nanch;
      e.counts[LP_LEN0 + wbuf] = na;
      const bool tail = na <= e.tail_rows;     // few live rows: skinny FP64 GEMMs beat a tensor-core pass
      e.counts[E_ANCHOR] = tail ? 0 : nanch;
      e.counts[E_LP] = tail ? 0 : e.counts[LP_LEN0 + (wbuf ^ 1)];
      e.counts[E_TAIL] = tail ? na : 0;
    }
  }
}

// mixed mode, tail: the live rows iterate in FP64; the operand is rebuilt from v every loop.  Rows waiting for an
// exact phase (candidates, re-anchored rows) sit the pass out exactly as they do in a tensor-core pass.
__global__ void k_tail_prep(const int* __restrict__ rows, const int* __restrict__ count, int* __restrict__ state,
                            const double* __restrict__ V, double* __restrict__ W, const double* __restrict__ lb,
                            const double* __restrict__ ub, int n, int nu) {
  const int cnt = *count;
  for (int li = blockIdx.x; li < cnt; li += gridDim.x) {
    const long long s = rows[li];
    const int st = state[s];
    __syncthreads();                                   // every thread has read the state before thread 0 may change it
    if (st != SLOT_ITER && st != SLOT_ANCHOR) continue;
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
      const int k = j % nu;
      const double v = V[s * n + j];
      W[s * n + j] = 2.0 * clipd(v, lb[s * nu + k], ub[s * nu + k]) - v;
    }
    if (threadIdx.x == 0 && st == SLOT_ANCHOR) state[s] = SLOT_ITER;
  }
}

// slots that finished a chunk: hand its final state back, load the initial state of the chunk taken next
__global__ void k_chunk_swap(const int* __restrict__ rows, const int* __restrict__ count, const int* __restrict__ c_old,
                             const int* __restrict__ c_new, double* __restrict__ xcur, double* __restrict__ upcur,
                             double* __restrict__ x_io, double* __restrict__ uprev_io, double* __restrict__ us_prev,
                             double* __restrict__ kappa, double kappa0, int nx, int nu) {
  const int cnt = *count;
  for (int li = blockIdx.x; li < cnt; li += gridDim.x) {
    const long long s = rows[li];
    const long long co = c_old[li], cn = c_new[li];
    if (x_io) {                                   // (null in batched-QP mode: chunks carry no plant state)
      for (int j = threadIdx.x; j < nx; j += blockDim.x) {
        x_io[co * nx + j] = xcur[s * nx + j];
        if (cn >= 0) xcur[s * nx + j] = x_io[cn * nx + j];
      }
      for (int j = threadIdx.x; j < nu; j += blockDim.x) {
        uprev_io[co * nu + j] = upcur[s * nu + j];
        if (cn >= 0) {
          upcur[s * nu + j] = uprev_io[cn * nu + j];
          us_prev[s * nu + j] = 0.0;
        }
      }
    }
    // a new chunk starts like a fresh trajectory: results do not depend on which slot serves it
    if (threadIdx.x == 0 && cn >= 0) kappa[s] = kappa0;
  }
}

// renew rows: v <- shifted previous solution re-centred on the new target (or the cold-start law
// already in V), w = 2 clip(v) - v into the operand buffer the next iteration reads
__global__ void k_warm_shift(const int* __restrict__ rows, const int* __restrict__ count, int* __restrict__ state,
                             int* __restrict__ it, unsigned long long* __restrict__ dres, double* __restrict__ V,
                             double* __restrict__ Zs, double* __restrict__ W, const double* __restrict__ dus,
                             const double* __restrict__ lb, const double* __restrict__ ub, int n, int nu,
                             int* __restrict__ cold_flag, int next_state, int write_w) {
  const int cnt = *count;
  for (int li = blockIdx.x; li < cnt; li += gridDim.x) {
  const long long s = rows[li];
  const int cold = cold_flag[s];   // cold start: V already holds the unconstrained law of this QP
  double* v = V + s * n;
  double* z = Zs + s * n;
  double* w = W + s * n;
  if (!cold) {
    // v_new[j] = v_old[j+nu] + dus[j % nu] (last stage repeated), staged through the free z row
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
      const int js = j + nu < n ? j + nu : j;
      z[j] = v[js] + dus[s * nu + (j % nu)];
    }
    __syncthreads();
  }
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    const double vn = cold ? v[j] : z[j];
    const int k = j % nu;
    if (!cold) v[j] = vn;
    if (write_w) w[j] = 2.0 * clipd(vn, lb[s * nu + k], ub[s * nu + k]) - vn;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    cold_flag[s] = 0;
    state[s] = next_state;
    it[s] = 0;
    dres[s] = 0ull;
  }
  __syncthreads();          // thread 0 has cleared the cold flag: nobody may still be reading it
  }
}

__global__ void k_engine_init(EngineArrays e, int S, int keep_kappa, double kappa0, int cold_all) {
  if (blockIdx.x * blockDim.x + threadIdx.x < S) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    e.chunk[i] = i;
    e.cold[i] = cold_all;
    e.l_cold[i] = i;
  }
  if (e.mixed && blockIdx.x * blockDim.x + threadIdx.x < S) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    e.l_anchor[i] = i;
    e.lp_list[i] = e.lp_list[S + i] = i;
    e.lp_pos[i] = e.lp_pos[S + i] = i;
  }
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < S) {
    e.state[s] = SLOT_RENEW;
    e.tcur[s] = 0;
    e.it[s] = 0;
    e.dres[s] = 0ull;
    e.kres[s] = 0ull;
    e.dtrig[s] = 0.0;
    if (!keep_kappa) e.kappa[s] = kappa0;
    e.l_active[s] = s;
    e.l_renew[s] = s;
  }
  if (s == 0) {
    e.counts[N_ACTIVE] = S;
    e.counts[N_CAND] = 0;
    e.counts[N_DONE] = 0;
    e.counts[N_RENEW] = S;
    e.counts[N_FINISHED] = 0;
    e.counts[F_MAXITER] = 0;
    e.counts[F_TS_FAIL] = 0;
    e.counts[N_ANCHOR] = e.mixed ? S : 0;
    e.counts[N_SWAP] = 0;
    e.counts[N_COLD] = cold_all ? S : 0;
    e.counts[NEXT_CHUNK] = S;
    const bool tail = S <= e.tail_rows;
    e.counts[LP_LEN0] = e.counts[LP_LEN1] = S;
    e.counts[E_ANCHOR] = (e.mixed && !tail) ? S : 0;
    e.counts[E_LP] = (e.mixed && !tail) ? S : 0;
    e.counts[E_TAIL] = (e.mixed && tail) ? S : 0;
    e.rowiters[0] = e.rowiters[1] = 0ull;
    e.stats[0] = e.stats[1] = e.stats[2] = e.stats[3] = 0ull;
  }
}

// Batched-QP mode of the engine (nnmpc_sim_solve_qps): every "trajectory chunk" is one regulator QP with its own
// x0 and bounds, one step long; the continuous batching, the tensor-core tiers and the exact certification are
// those of the closed loop, the target selector and the plant step drop out.
struct QpBatch {
  const double* X0;   // Btot x nxa_ld
  const double* LB;   // Btot x nu
  const double* UB;
  double* U;          // Btot x n
  double* cost;       // Btot, nullable
};

// renew rows in batched-QP mode: regulator inputs of the chunk (= QP) the slot now works on
__global__ void k_qp_load(const int* __restrict__ rows, const int* __restrict__ count, const int* __restrict__ chunk,
                          QpBatch qb, double* __restrict__ x0, double* __restrict__ lb, double* __restrict__ ub,
                          double* __restrict__ dus, int nxa_ld, int nu) {
  const int cnt = *count;
  for (int li = blockIdx.x; li < cnt; li += gridDim.x) {
    const long long s = rows[li], c = chunk[s];
    for (int j = threadIdx.x; j < nxa_ld; j += blockDim.x) x0[s * nxa_ld + j] = qb.X0[c * nxa_ld + j];
    for (int j = threadIdx.x; j < nu; j += blockDim.x) {
      lb[s * nu + j] = qb.LB[c * nu + j];
      ub[s * nu + j] = qb.UB[c * nu + j];
      dus[s * nu + j] = 0.0;
    }
  }
}

// done rows in batched-QP mode: minimiser, optimal cost 1/2 z'(g + q) and the workload statistics
__global__ void __launch_bounds__(256)
k_qp_store(const int* __restrict__ rows, const int* __restrict__ count, const int* __restrict__ chunk, QpBatch qb,
           const double* __restrict__ Z, const double* __restrict__ G, const double* __restrict__ Ql,
           const double* __restrict__ lb, const double* __restrict__ ub, unsigned long long* __restrict__ stats, int n,
           int nu) {
  __shared__ double red[8];
  const int cnt = *count;
  for (int li = blockIdx.x; li < cnt; li += gridDim.x) {
    const long long s = rows[li], c = chunk[s];
    double acc = 0.0;
    int na = 0;
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
      const double z = Z[s * n + j];
      qb.U[c * n + j] = z;
      if (qb.cost) acc += z * (G[s * n + j] + Ql[s * n + j]);
      na += (z <= lb[s * nu + (j % nu)] || z >= ub[s * nu + (j % nu)]) ? 1 : 0;
    }
    if (__syncthreads_or(na > 0)) {
      na = __reduce_add_sync(0xffffffffu, na);
      if ((threadIdx.x & 31) == 0 && na > 0) atomicAdd(stats + 3, (unsigned long long)na);
      if (threadIdx.x == 0) atomicAdd(stats + 2, 1ull);
    }
    if (qb.cost) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
      __syncthreads();
      if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w];
        qb.cost[c] = 0.5 * t;
      }
      __syncthreads();
    }
  }
}

static int sim_ensure(nnmpc_sim* h, long long B) {
  if (B <= h->cap) return 0;
  const long long n = h->qp->n;
  h->warm_B = 0;
  NNMPC_TRY(h->x0.ensure(B * h->nxa_ld));
  NNMPC_TRY(h->lb.ensure(B * h->nu));
  NNMPC_TRY(h->ub.ensure(B * h->nu));
  NNMPC_TRY(h->us_prev.ensure(B * h->nu));
  NNMPC_TRY(h->dus.ensure(B * h->nu));
  NNMPC_TRY(h->V.ensure(B * n));
  NNMPC_TRY(h->Z.ensure(B * n));
  NNMPC_TRY(h->xcur.ensure(B * h->nx));
  NNMPC_TRY(h->upcur.ensure(B * h->nu));
  NNMPC_TRY(h->kappa.ensure(B));
  NNMPC_TRY(h->dtrig.ensure(B));
  NNMPC_TRY(h->state.ensure(B));
  NNMPC_TRY(h->tcur.ensure(B));
  NNMPC_TRY(h->it.ensure(B));
  NNMPC_TRY(h->lists.ensure(9 * B));
  NNMPC_TRY(h->chunk.ensure(B));
  NNMPC_TRY(h->cold.ensure(B));
  NNMPC_TRY(h->lp_layout.ensure(4 * B));
  NNMPC_TRY(h->dlast.ensure(B));
  NNMPC_TRY(h->need2.ensure((B + 127) / 128 + 2));
  NNMPC_TRY(h->dres.ensure(B));
  NNMPC_TRY(h->kres.ensure(B));
  h->cap = B;
  return 0;
}

// ---- lock-step engine of an interior-point regulator handle (nnmpc_qp_create_ipm) ------------------------------------
// The continuously batched engine above is built on Douglas-Rachford internals (operand buffers, anchors, per-row
// triggers).  With an interior-point regulator every step runs over the whole batch, as the online loop does:
//     target selector (fused regulator inputs) -> interior-point QPs (ipm.cu) -> dataset rows and plant step.
// Precision, slots, cadence, tail, exact-GEMM and second-term options have no effect on it.

// one CTA per trajectory: u = first move + target, dataset row, uprev, optional capture, x+ = [A|B|Bd][x|u|d]
__global__ void __launch_bounds__(128)
k_ipm_plant(int B, int T, int t, const double* __restrict__ U, int n, const double* __restrict__ us,
            double* __restrict__ xcur, double* __restrict__ upcur, const double* __restrict__ dist,
            double* __restrict__ row_u, const double* __restrict__ ABd, int nx, int nu, int nd, int kin_ld,
            double* __restrict__ cap_useq) {
  extern __shared__ double kin[];   // kin_ld
  for (int s = blockIdx.x; s < B; s += gridDim.x) {
    const long long o = (long long)s * T + t;
    for (int c = threadIdx.x; c < kin_ld; c += blockDim.x) {
      double v = 0.0;
      if (c < nx) {
        v = xcur[(long long)s * nx + c];
      } else if (c < nx + nu) {
        const int k = c - nx;
        v = U[(long long)s * n + k] + us[o * nu + k];
        row_u[o * nu + k] = v;
        upcur[(long long)s * nu + k] = v;
      } else if (c < nx + nu + nd) {
        v = dist[o * nd + (c - nx - nu)];
      }
      kin[c] = v;
    }
    if (cap_useq)
      for (int j = threadIdx.x; j < n; j += blockDim.x) cap_useq[o * n + j] = U[(long long)s * n + j] + us[o * nu + (j % nu)];
    __syncthreads();
    for (int i = threadIdx.x; i < nx; i += blockDim.x) {
      double a = 0.0;
      for (int c = 0; c < kin_ld; ++c) a += ABd[(long long)i * kin_ld + c] * kin[c];
      xcur[(long long)s * nx + i] = a;
    }
    __syncthreads();
  }
}

static int sim_run_ipm(nnmpc_sim* h, int B, int T, double* x_io, double* uprev_io, const double* sp, const double* dist,
                       double* ox, double* ouprev, double* oxs, double* ous, double* ou, int* oiters, double* okkt,
                       double tol, int max_iter, cudaStream_t st, const QpBatch* qb) {
  nnmpc_qp* q = h->qp;
  long long isum = 0;
  int warn = 0;
  if (qb) {
    warn = ipm_solve_device(q, B, qb->X0, qb->LB, qb->UB, qb->U, QpOutputs{qb->cost, okkt, oiters, 1}, tol, max_iter, st,
                            &isum);
    if (warn < 0) return warn;
  } else {
    const int nx = h->nx, nu = h->nu, nd = h->nd, ny = h->ny, n = q->n, nxa = h->nxa_ld;
    const size_t b = (size_t)B;
    NNMPC_TRY(h->x0.ensure(b * nxa));
    NNMPC_TRY(h->lb.ensure(b * nu));
    NNMPC_TRY(h->ub.ensure(b * nu));
    NNMPC_TRY(h->us_prev.ensure(b * nu));
    NNMPC_TRY(h->dus.ensure(b * nu));
    NNMPC_TRY(h->xcur.ensure(b * nx));
    NNMPC_TRY(h->upcur.ensure(b * nu));
    NNMPC_TRY(h->Z.ensure(b * n));
    NNMPC_CUDA(cudaMemsetAsync(h->counts, 0, N_COUNTERS * sizeof(int), st));
    NNMPC_CUDA(cudaMemsetAsync(h->x0.p, 0, b * nxa * 8, st));   // padding column of x0
    NNMPC_CUDA(cudaMemsetAsync(h->us_prev.p, 0, b * nu * 8, st));
    NNMPC_CUDA(cudaMemcpyAsync(h->xcur.p, x_io, b * nx * 8, cudaMemcpyDeviceToDevice, st));
    NNMPC_CUDA(cudaMemcpyAsync(h->upcur.p, uprev_io, b * nu * 8, cudaMemcpyDeviceToDevice, st));
    const size_t smem = (size_t)h->kin_ld * sizeof(double);
    if (smem > 48 * 1024) return set_error(NNMPC_ERR_UNSUPPORTED, "plant step: nx + nu + nd = %d is too large", h->kin_ld);
    for (int t = 0; t < T; ++t) {
      TsFused F{};
      F.x = h->xcur.p; F.uprev = h->upcur.p; F.x0 = h->x0.p; F.nxa_ld = nxa; F.lb = h->lb.p; F.ub = h->ub.p;
      F.us_prev = h->us_prev.p; F.dus = h->dus.p;
      F.row_x = ox + (size_t)t * nx; F.row_uprev = ouprev + (size_t)t * nu;
      F.row_stride_x = (long long)T * nx; F.row_stride_u = (long long)T * nu;
      NNMPC_TRY(ts_solve_device(h->ts, B, sp + (size_t)t * ny, (long long)T * ny, dist + (size_t)t * nd, (long long)T * nd,
                                oxs + (size_t)t * nx, (long long)T * nx, ous + (size_t)t * nu, (long long)T * nu, nullptr, 0,
                                &F, nullptr, h->counts + F_TS_FAIL, st));
      long long it = 0;
      const int rc = ipm_solve_device(q, B, h->x0.p, h->lb.p, h->ub.p, h->Z.p,
                                      QpOutputs{h->cap_cost ? h->cap_cost + t : nullptr, okkt ? okkt + t : nullptr,
                                                oiters ? oiters + t : nullptr, T},
                                      tol, max_iter, st, &it);
      if (rc < 0) return rc;
      warn |= rc;
      isum += it;
      k_ipm_plant<<<row_grid(B), 128, smem, st>>>(B, T, t, h->Z.p, n, ous, h->xcur.p, h->upcur.p, dist, ou, h->ABd, nx, nu, nd,
                                                  h->kin_ld, h->cap_useq);
      count_launch();
    }
    NNMPC_CUDA(cudaMemcpyAsync(x_io, h->xcur.p, b * nx * 8, cudaMemcpyDeviceToDevice, st));
    NNMPC_CUDA(cudaMemcpyAsync(uprev_io, h->upcur.p, b * nu * 8, cudaMemcpyDeviceToDevice, st));
    NNMPC_CUDA(cudaMemcpyAsync(h->pin, h->counts, N_COUNTERS * sizeof(int), cudaMemcpyDeviceToHost, st));
    NNMPC_CUDA(cudaStreamSynchronize(st));
    NNMPC_CUDA(cudaGetLastError());
    if (h->pin[F_TS_FAIL]) warn |= NNMPC_WARN_TARGET;
  }
  h->tot_rowiters += isum;
  h->tot_qps += (long long)B * (qb ? 1 : T);
  return warn;
}

static int sim_run_device(nnmpc_sim* h, int Btot, int T, double* x_io, double* uprev_io, const double* sp,
                          const double* dist, double* ox, double* ouprev, double* oxs, double* ous, double* ou,
                          int* oiters, double* okkt, double tol, int max_iter, int resume, cudaStream_t st,
                          const QpBatch* qb = nullptr) {
  if (Btot <= 0 || T <= 0) return 0;
  if (h->qp->ipm) return sim_run_ipm(h, Btot, T, x_io, uprev_io, sp, dist, ox, ouprev, oxs, ous, ou, oiters, okkt, tol, max_iter,
                                     st, qb);
  if (max_iter < 1) max_iter = 1;
  // B trajectory slots advance concurrently; with more chunks than slots the rest queue up and a slot that
  // finishes its chunk takes the next one (cold start), so the batch stays full until the queue is empty
  const int B = Btot < h->slot_cap ? Btot : h->slot_cap;
  NNMPC_TRY(sim_ensure(h, B));
  nnmpc_qp* q = h->qp;
  NNMPC_TRY(qp_ensure_scratch(q, B));
  const bool cont = resume && h->warm_B == Btot && Btot == B;   // solver state is kept per slot
  h->warm_B = 0;
  const int nx = h->nx, nu = h->nu, nd = h->nd, ny = h->ny, n = q->n, nxa = h->nxa_ld;
  const int mixed = h->mixed;
  if (mixed) {
    if (!q->rinv)
      return set_error(NNMPC_ERR_BADARG, "mixed precision needs the ADMM penalty vector: call nnmpc_qp_set_penalty first");
    if (!q->lpop.ready) NNMPC_TRY(lp_split_operator(q->Top, n, q->top_max, &q->lpop, st));
    // (one-term tiles by row phase are the other, older scheme.)  Small QPs keep both terms in every pass: at n = 540 the
    // MMAs are 15 % of a pass and the pending sums only add epilogue traffic (probe: 0.167 ms fused, 0.189 ms deferred)
    h->lps.defer2 = h->t2_every > 0 && !(h->t2_factor > 0.0) && (!h->t2_auto || n >= T2_AUTO_MIN_N);
    NNMPC_TRY(lp_state_ensure(&h->lps, h->cap, n, st));
    if (h->exact_oz) {
      if (!q->ozP.ready) NNMPC_TRY(oz_slice_operator(q->P, n, n, &q->ozP, st));
      if (!q->ozTop.ready) NNMPC_TRY(oz_slice_operator(q->Top, n, n, &q->ozTop, st));
      NNMPC_TRY(oz_rows_ensure(&h->ozr, h->cap, n, st));
    }
  }
  const bool oz = mixed && h->exact_oz;
  // gradient g = P z + q of the exact check: the mixed mode re-anchors from it; the cost capture needs it in any mode
  const bool want_g = h->cap_cost || (qb && qb->cost);
  if (!mixed && want_g) NNMPC_TRY(h->gcap.ensure((size_t)h->cap * n));
  double* gbuf = mixed ? h->lps.Wl.p : (want_g ? h->gcap.p : nullptr);
  if (!qb) {
    NNMPC_CUDA(cudaMemcpyAsync(h->xcur.p, x_io, (size_t)B * nx * 8, cudaMemcpyDeviceToDevice, st));
    NNMPC_CUDA(cudaMemcpyAsync(h->upcur.p, uprev_io, (size_t)B * nu * 8, cudaMemcpyDeviceToDevice, st));
  }
  if (!cont) NNMPC_CUDA(cudaMemsetAsync(h->us_prev.p, 0, (size_t)B * nu * 8, st));

  EngineArrays e{};
  e.state = h->state.p; e.tcur = h->tcur.p; e.it = h->it.p; e.kappa = h->kappa.p; e.dtrig = h->dtrig.p;
  e.dres = h->dres.p; e.kres = h->kres.p;
  e.l_active = h->lists.p; e.l_cand = h->lists.p + B; e.l_done = h->lists.p + 2 * (long long)B;
  e.l_renew = h->lists.p + 3 * (long long)B; e.l_anchor = h->lists.p + 4 * (long long)B;
  e.counts = h->counts; e.rowiters = h->rowiters;
  e.l_cold = h->lists.p + 5 * (long long)B; e.l_swap = h->lists.p + 6 * (long long)B;
  e.swap_old = h->lists.p + 7 * (long long)B; e.swap_new = h->lists.p + 8 * (long long)B;
  e.chunk = h->chunk.p; e.cold = h->cold.p; e.n_chunks = Btot;
  e.lp_list = h->lp_layout.p; e.lp_pos = h->lp_layout.p + 2 * (long long)B;
  // automatic tail: below ~B/256 live rows skinny FP64 GEMMs beat a tensor-core pass (measured on B200, round 2c:
  // B/16 spends 5.5 % of the step in the tail, B/64 2.3 %, B/256 1.5 %)
  e.tail_rows = h->tail_rows >= 0 ? h->tail_rows : (B / 256 > 48 ? B / 256 : 48);
  const bool t2skip = mixed && h->t2_factor > 0.0;
  e.dlast = h->dlast.p; e.t2_thr = h->t2_factor * tol; e.need2 = t2skip ? h->need2.p : nullptr;
  if (t2skip) NNMPC_CUDA(cudaMemsetAsync(h->need2.p, 1, (size_t)((B + 127) / 128 + 2), st));   // first pass: both terms everywhere
  NNMPC_CUDA(cudaMemsetAsync(h->dlast.p, 0x7f, (size_t)B * sizeof(double), st));              // large: nothing is late yet
  e.mixed = mixed; e.sc_in = h->lps.sc_in.p; e.sc_out = h->lps.sc_out.p; e.stats = h->stats; e.alpha = q->alpha;
  k_engine_init<<<(B + 255) / 256, 256, 0, st>>>(e, B, cont ? 1 : 0, h->kappa0, cont ? 0 : 1);
  count_launch();

  const size_t adv_smem = (size_t)ADV_ROWS * h->kin_ld * sizeof(double);
  if (adv_smem > 200 * 1024) return set_error(NNMPC_ERR_UNSUPPORTED, "plant step: nx + nu + nd = %d does not fit the staging buffer", h->kin_ld);
  if (adv_smem > 48 * 1024)
    NNMPC_CUDA(cudaFuncSetAttribute(k_advance_plant, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)adv_smem));
  double* Wc = q->W0.p;   // operand the next iteration reads
  double* Wn = q->W1.p;
  int lay = 0;            // mixed mode: operand layout buffer the next tensor-core pass reads

  // target selector + regulator inputs + solver (re)start for the rows of the renew list
  auto renew = [&](int first) -> int {
    TsFused F{};
    F.x = h->xcur.p; F.uprev = h->upcur.p; F.x0 = h->x0.p; F.nxa_ld = nxa; F.lb = h->lb.p; F.ub = h->ub.p;
    F.us_prev = h->us_prev.p; F.dus = h->dus.p;
    F.row_x = ox; F.row_uprev = ouprev; F.row_stride_x = nx; F.row_stride_u = nu;
    TsIndex ix{e.l_renew, e.counts + N_RENEW, e.tcur, T, e.chunk};
    if (qb) {
      k_qp_load<<<row_grid(B), 128, 0, st>>>(e.l_renew, e.counts + N_RENEW, e.chunk, *qb, h->x0.p, h->lb.p, h->ub.p, h->dus.p, nxa, nu);
      count_launch();
    } else {
      NNMPC_TRY(ts_solve_device(h->ts, B, sp, ny, dist, nd, oxs, nx, ous, nu, nullptr, 0, &F, &ix, e.counts + F_TS_FAIL, st));
    }
    GemmOperands g{};
    g.A = h->x0.p; g.lda = nxa; g.ldb = nxa; g.M = B; g.N = n; g.K = nxa; g.rows = e.l_renew;
    g.m_count = e.counts + N_RENEW;
    g.Bt = q->Mtq;
    cudaError_t ce = launch_gemm<TileMid, EpiStore>(g, EpiStore::Params{q->C.p, n, nullptr, 0}, st);
    g.Bt = q->tq;
    if (ce == cudaSuccess) ce = launch_gemm<TileMid, EpiStore>(g, EpiStore::Params{q->Ql.p, n, nullptr, 0}, st);
    if (ce == cudaSuccess && (first ? !cont : Btot > B)) {   // cold starts: the unconstrained (LQR) law v0 = Kunc x0
      g.Bt = q->Kunc; g.rows = e.l_cold; g.m_count = e.counts + N_COLD;
      ce = launch_gemm<TileMid, EpiStore>(g, EpiStore::Params{h->V.p, n, nullptr, 0}, st);
      count_launch();
    }
    count_launch(2);
    if (ce != cudaSuccess) return set_error(NNMPC_ERR_CUDA, "gemm launch failed: %s", cudaGetErrorString(ce));
    // mixed mode: a QP starts from an FP64 anchor GEMM at the top of the next full loop.  (Measured on B200:
    // starting it instead from the x the previous QP's last check anchored, with the change of the operand as
    // the first fp16 increment, makes nearly every first check fail - the stage shift is an O(1e-2) increment
    // whose fp32-accumulation error is far above the 1e-10 the trigger needs - and costs 2 checks + 53
    // iterations per QP instead of 1.1 + 30.)
    k_warm_shift<<<row_grid(B), 256, 0, st>>>(e.l_renew, e.counts + N_RENEW, e.state, e.it, e.dres, h->V.p, h->Z.p, Wc,
                                    h->dus.p, h->lb.p, h->ub.p, n, nu, e.cold, mixed ? SLOT_ANCHOR : SLOT_ITER,
                                    mixed ? 0 : 1);
    count_launch();
    return 0;
  };

  NNMPC_TRY(renew(1));

  // mixed mode: the FP64 phases (exact checks, plant step, next targets, cold-start anchors) run every cad-th loop
  // over the rows that accumulated meanwhile - those rows sit out at most cad-1 tensor-core passes, and the FP64
  // GEMMs and the small kernels around them see cad times longer row lists
  const int cad = mixed ? (h->cadence > 1 ? h->cadence : 1) : 1;
  // deferred second operator term: delivery passes fall on full loops (right after the anchors of new QPs, whose first
  // - largest - increment is then corrected in the same loop), every m2-th loop
  const int m2 = (mixed && h->lps.defer2) ? (h->t2_every + cad - 1) / cad * cad : 0;
  long long polls = 0;
  const long long max_loops = ((long long)T * ((long long)max_iter + 2) * ((Btot + B - 1) / B) + 8) * cad;
  int rc_warn = 0;
  bool finished = false;
  long long loop = 0;
  for (; loop < max_loops && !finished; ++loop) {
    // 1. one Douglas-Rachford iteration for every live trajectory
    const bool full = (loop % cad) == 0;
    const int* pos_next = e.lp_pos;      // mixed mode: layout the NEXT pass reads (set below)
    if (mixed) {
      // 1a. exact anchors for the rows that start a QP: x = Top w - c (INT8-sliced tensor-core apply, or the
      //     DMMA kernel), one full-precision step, first fp16 increment
      int* cnt = e.counts + E_ANCHOR;
      const int rbuf = lay;
      const int* list_r = e.lp_list + (long long)rbuf * B;
      const int* pos_r = e.lp_pos + (long long)rbuf * B;
      // a full loop ends with k_step, which publishes the next live list: write the operand in that layout
      const int* pos_w = e.lp_pos + (long long)(full ? rbuf ^ 1 : rbuf) * B;
      ProfSpan span64;
      if (full) {
        const bool prof64 = prof_begin(&span64, st);
        NNMPC_TRY(lp_anchor_prep(e.l_anchor, cnt, B, h->V.p, q->W0.p, &h->lps, h->lb.p, h->ub.p, nu, st));
        if (oz) NNMPC_TRY(oz_anchor(&q->ozTop, &h->ozr, e.l_anchor, cnt, B, q->W0.p, q->C.p, h->lps.X.p, n, h->device, st));
        else NNMPC_TRY(lp_anchor_gemm(e.l_anchor, cnt, B, q->W0.p, q->Top, q->C.p, h->lps.X.p, n, st));
        NNMPC_TRY(lp_dr_first(e.l_anchor, cnt, B, &h->lps, h->V.p, q->W0.p, h->lb.p, h->ub.p, e.state, e.it, SLOT_ITER,
                              nu, q->alpha, pos_r, st, e.need2));
        if (prof64) prof_end(span64, st, 0.0, 1, 1);
      }
      // 1b. tensor-core pass (tcgen05, fp16 increments of the operand, state in FP64) over every live row
      ProfSpan span;
      const bool prof = prof_begin(&span, st);
      int s_mode = 0;
      if (m2) {
        s_mode = 1;
        if (loop % m2 == 0) {
          NNMPC_TRY(lp_correct(&q->lpop, &h->lps, B, list_r, e.counts + E_LP, e.state, SLOT_ITER, h->device, st, h->tile_stat + 2));
          s_mode = 2;
        }
      }
      NNMPC_TRY(lp_iterate(&q->lpop, &h->lps, B, list_r, e.counts + E_LP, pos_w, h->V.p, h->lb.p, h->ub.p, e.state,
                           SLOT_ITER, e.dres, nu, q->alpha, h->device, st, e.need2, h->tile_stat, s_mode));
      pos_next = pos_w;
      if (prof) prof_end(span, st, 0.0, 1);
      // 1c. tail: with few live rows left the same update runs as skinny FP64 GEMMs (counts[E_TAIL] rows, else 0)
      const bool prof64b = prof_begin(&span64, st);
      // at most tail_rows rows are ever listed here (E_TAIL is 0 above that)
      const int tail_grid = e.tail_rows < B ? (e.tail_rows > 0 ? e.tail_rows : 1) : B;
      k_tail_prep<<<row_grid(tail_grid), 256, 0, st>>>(e.l_active, e.counts + E_TAIL, e.state, h->V.p, q->W0.p, h->lb.p, h->ub.p, n, nu);
      count_launch();
      GemmOperands gi{};
      gi.A = q->W0.p; gi.lda = n; gi.Bt = q->Top; gi.ldb = n; gi.M = e.tail_rows < B ? (e.tail_rows > 0 ? e.tail_rows : 1) : B;
      gi.N = n; gi.K = n; gi.rows = e.l_active; gi.m_count = e.counts + E_TAIL;
      EpiAdmm::Params ept{h->V.p, q->C.p, q->W1.p, nullptr, h->lb.p, h->ub.p, n, nu, q->alpha, 0, e.dres, e.state, SLOT_ITER};
      NNMPC_TRY(gemm_by_count<EpiAdmm>(gi, ept, st));
      if (prof64b) prof_end(span64, st, 0.0, 1, 2);
    } else {
      GemmOperands gi{};
      gi.A = Wc; gi.lda = n; gi.Bt = q->Top; gi.ldb = n; gi.M = B; gi.N = n; gi.K = n; gi.rows = e.l_active;
      gi.m_count = e.counts + N_ACTIVE;
      EpiAdmm::Params ep{h->V.p, q->C.p, Wn, nullptr, h->lb.p, h->ub.p, n, nu, q->alpha, 0, e.dres, nullptr, 0};
      ProfSpan span;
      const bool prof = prof_begin(&span, st);
      NNMPC_TRY(gemm_by_count<EpiAdmm>(gi, ep, st));
      if (prof) prof_end(span, st, 0.0, 1);
      double* t = Wc; Wc = Wn; Wn = t;
    }
    // 2-4. candidates -> exact KKT check -> done list
    if (!(cad > 1 && (loop % cad) != 1 % cad))      // a new candidate list starts (otherwise this pass appends to it)
      NNMPC_CUDA(cudaMemsetAsync(e.counts + N_CAND, 0, sizeof(int), st));
    {
      int sel_blocks = e.need2 ? 1 : (B + 4095) / 4096;
      if (sel_blocks > 16) sel_blocks = 16;
      k_select<<<sel_blocks, 1024, 0, st>>>(e, tol, max_iter, full ? 1 : 0, pos_next, B);
    }
    if (!full) {
      count_launch();
      continue;
    }
    k_make_z<<<row_grid(B), 256, 0, st>>>(e.l_cand, e.counts + N_CAND, h->V.p, h->Z.p, h->lb.p, h->ub.p, n, nu);
    count_launch(2);
    {
      GemmOperands gv{};
      gv.A = h->Z.p; gv.lda = n; gv.Bt = q->P; gv.ldb = n; gv.M = B; gv.N = n; gv.K = n; gv.rows = e.l_cand;
      gv.m_count = e.counts + N_CAND;
      EpiVerifyMax::Params ev{h->Z.p, q->Ql.p, h->lb.p, h->ub.p, e.kres, n, nu, gbuf};
      ProfSpan span64;
      const bool prof64 = mixed && prof_begin(&span64, st);
      if (oz) NNMPC_TRY(oz_verify(&q->ozP, &h->ozr, e.l_cand, e.counts + N_CAND, B, h->Z.p, q->Ql.p, h->lb.p, h->ub.p,
                                  e.kres, h->lps.Wl.p, n, nu, h->device, st));
      else NNMPC_TRY(gemm_by_count<EpiVerifyMax>(gv, ev, st));
      if (prof64) prof_end(span64, st, 0.0, 1, 1);
    }
    ProfSpan span_rest;
    const bool prof_rest = mixed && prof_begin(&span_rest, st);
    k_retire<<<1, 1024, 0, st>>>(e, tol, max_iter, T, oiters, okkt, h->kappa_max);
    if (mixed) {
      // a failed exact check re-anchors the fp16 path from its own gradient (no FP64 anchor GEMM): x := z exactly
      // for w_lp = z + g / rho; the row goes on with the first increment of what is left to deliver
      NNMPC_TRY(lp_reanchor(e.l_cand, e.counts + N_CAND, B, e.state, SLOT_EMIT, h->Z.p, q->rinv, &h->lps, st));
      NNMPC_TRY(lp_emit(e.l_cand, e.counts + N_CAND, B, e.state, SLOT_EMIT, SLOT_ITER, &h->lps, h->V.p, h->lb.p,
                        h->ub.p, e.dtrig, nu, q->alpha, e.lp_pos + (long long)(lay ^ 1) * B, st, e.need2));
    }
    // 5. first move, dataset row, plant step for the done rows
    if (qb)
      k_qp_store<<<row_grid(B), 256, 0, st>>>(e.l_done, e.counts + N_DONE, e.chunk, *qb, h->Z.p, gbuf, q->Ql.p, h->lb.p, h->ub.p,
                                              h->stats, n, nu);
    else
      k_advance_plant<<<row_grid((B + ADV_ROWS - 1) / ADV_ROWS), ADV_THREADS, adv_smem, st>>>(
          e.l_done, e.counts + N_DONE, e.tcur, e.chunk, T, h->Z.p, ous, h->xcur.p, dist, ou, h->upcur.p, h->ABd, n, nx, nu, nd,
          h->kin_ld, gbuf, q->Ql.p, h->cap_useq, h->cap_cost, h->lb.p, h->ub.p, h->stats);
    count_launch(2);
    // 6-7. next time step for the done rows
    k_step<<<1, 1024, 0, st>>>(e, T, B, lay);
    lay ^= 1;
    k_chunk_swap<<<row_grid(B), 128, 0, st>>>(e.l_swap, e.counts + N_SWAP, e.swap_old, e.swap_new, h->xcur.p, h->upcur.p, qb ? nullptr : x_io,
                                    uprev_io, h->us_prev.p, h->kappa.p, h->kappa0, nx, nu);
    count_launch(2);
    NNMPC_TRY(renew(0));
    if (prof_rest) prof_end(span_rest, st, 0.0, 1, 3);
    // poll the finished counter with a two-loop lag (the GPU never waits for the host)
    const int slot = (int)(polls % POLL_RING);
    NNMPC_CUDA(cudaMemcpyAsync(h->pin + slot * N_COUNTERS, h->counts, N_COUNTERS * sizeof(int),
                               cudaMemcpyDeviceToHost, st));
    NNMPC_CUDA(cudaEventRecord(h->poll_ev[slot], st));
    ++polls;
    if (polls >= 3) {
      const int k = (int)((polls - 3) % POLL_RING);
      NNMPC_CUDA(cudaEventSynchronize(h->poll_ev[k]));
      if (h->pin[k * N_COUNTERS + N_FINISHED] >= Btot) finished = true;
    }
  }
  // drain: the last loops may not have been polled yet
  unsigned long long* pin64 = reinterpret_cast<unsigned long long*>(h->pin + POLL_RING * N_COUNTERS);
  for (int i = 0; i < 8; ++i) pin64[i] = 0ull;
  NNMPC_CUDA(cudaMemcpyAsync(h->pin, h->counts, N_COUNTERS * sizeof(int), cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaMemcpyAsync(pin64 + 5, h->rowiters, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaMemcpyAsync(pin64 + 1, h->stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaStreamSynchronize(st));   // final states were handed back chunk by chunk (k_chunk_swap)
  NNMPC_CUDA(cudaGetLastError());
  if (h->pin[N_FINISHED] < Btot)
    return set_error(NNMPC_ERR_CUDA, "closed-loop engine stopped with %d of %d trajectories finished", h->pin[N_FINISHED], Btot);
  if (h->pin[F_MAXITER]) rc_warn |= NNMPC_WARN_MAXITER;
  if (h->pin[F_TS_FAIL]) rc_warn |= NNMPC_WARN_TARGET;
  pin64[0] = pin64[5];
  g_iterations.fetch_add((long long)*pin64, std::memory_order_relaxed);
  // each channel's flops belong to the kernels whose time it records: tensor-core passes (0), FP64 tail (2)
  prof_add_flops(2.0 * n * (double)n * (double)(pin64[5] - pin64[6]));                // iteration passes
  prof_add_flops(2.0 * n * (double)n * (double)pin64[6], 2);                          // FP64 tail iterations
  prof_add_flops(2.0 * n * (double)n * (double)(pin64[1] + pin64[2]), 1);             // exact anchors + checks (FP64-equivalent)
  h->tot_rowiters += (long long)pin64[0];
  h->tot_anchors += (long long)pin64[1];
  h->tot_verifies += (long long)pin64[2];
  h->tot_qps += (long long)Btot * T;
  h->tot_qps_active += (long long)pin64[3];
  h->tot_active += (long long)pin64[4];
  h->warm_B = (Btot == B && !qb) ? Btot : 0;
  return rc_warn;
}

}  // namespace nnmpc

using namespace nnmpc;

extern "C" {

int nnmpc_sim_create(nnmpc_sim_t** out, nnmpc_qp_t* qp, nnmpc_ts_t* ts, int nx, int nu, int nd, int ny,
                     const double* ABd_host, int device) {
  // ts == NULL (with ABd_host == NULL): a handle for nnmpc_sim_solve_qps only
  if (!out || !qp || (ts && !ABd_host)) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_create: null argument");
  if (qp->device != device || (ts && ts->device != device))
    return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_create: handles live on different devices");
  if (qp->nu != nu || qp->nxa < nx + nu || (ts && (ts->nu != nu || ts->nx != nx || ts->nd != nd || ts->ny != ny)))
    return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_create: inconsistent sizes");
  DeviceGuard dg(device);
  nnmpc_sim* h = new (std::nothrow) nnmpc_sim();
  if (!h) return set_error(NNMPC_ERR_NOMEM, "out of host memory");
  h->qp = qp; h->ts = ts; h->nx = nx; h->nu = nu; h->nd = nd; h->ny = ny; h->device = device;
  h->nxa_ld = qp->nxa;
  const int kin = nx + nu + nd;
  h->kin_ld = (kin + 1) & ~1;
  h->cap = 0;
  h->warm_B = 0;
  h->ABd = nullptr; h->counts = nullptr; h->rowiters = nullptr; h->stats = nullptr; h->pin = nullptr;
  for (int i = 0; i < POLL_RING; ++i) h->poll_ev[i] = nullptr;
  h->mixed = 0;
  h->tail_rows = -1;
  h->slot_cap = 8192;
  h->cadence = 4;
  h->exact_oz = 1;
  h->cap_useq = h->cap_cost = nullptr;
  h->t2_auto = true;
  h->t2_every = 8;          // measured (profiles/r02o/p): 4 -> +12 %, 8 -> +16 %, 12 -> +17 %, 16 -> +11 % sim-steps/s over the fused form;
                            // iterations and exact checks per QP are unchanged up to 8 and start to grow at 12
  h->t2_factor = 0.0;       // one-term tiles off: measured share of such tiles 0.4 - 6 % (rows restart inside late tiles), no gain
  h->tile_stat = nullptr;
  h->tot_rowiters = h->tot_anchors = h->tot_verifies = h->tot_qps = h->tot_qps_active = h->tot_active = 0;
  h->kappa0 = 0.25 * qp->p_norm_inf;
  h->kappa_max = 8.0 * qp->p_norm_inf;
  // pad [A|B|Bd] rows to an even leading dimension for the 16-byte operand loader
  int rc = 0;
  if (ABd_host) {
    double* tmp = new (std::nothrow) double[(size_t)nx * h->kin_ld];
    if (!tmp) {
      delete h;
      return set_error(NNMPC_ERR_NOMEM, "out of host memory");
    }
    for (int r = 0; r < nx; ++r) {
      for (int c = 0; c < kin; ++c) tmp[(size_t)r * h->kin_ld + c] = ABd_host[(size_t)r * kin + c];
      for (int c = kin; c < h->kin_ld; ++c) tmp[(size_t)r * h->kin_ld + c] = 0.0;
    }
    rc = upload(&h->ABd, tmp, (size_t)nx * h->kin_ld);
    delete[] tmp;
  }
  auto cu = [&](cudaError_t e, const char* what) {
    if (rc == 0 && e != cudaSuccess) rc = set_error(NNMPC_ERR_CUDA, "nnmpc_sim_create: %s: %s", what, cudaGetErrorString(e));
  };
  if (rc == 0) cu(cudaMalloc((void**)&h->counts, N_COUNTERS * sizeof(int)), "cudaMalloc");
  if (rc == 0) cu(cudaMalloc((void**)&h->rowiters, 2 * sizeof(unsigned long long)), "cudaMalloc");
  if (rc == 0) cu(cudaMalloc((void**)&h->stats, 4 * sizeof(unsigned long long)), "cudaMalloc");
  if (rc == 0) cu(cudaMemset(h->stats, 0, 4 * sizeof(unsigned long long)), "cudaMemset");
  if (rc == 0) cu(cudaMalloc((void**)&h->tile_stat, 4 * sizeof(unsigned long long)), "cudaMalloc");
  if (rc == 0) cu(cudaMemset(h->tile_stat, 0, 4 * sizeof(unsigned long long)), "cudaMemset");
  if (rc == 0) cu(cudaMallocHost((void**)&h->pin, POLL_RING * N_COUNTERS * sizeof(int) + 8 * sizeof(unsigned long long)), "cudaMallocHost");
  for (int i = 0; i < POLL_RING && rc == 0; ++i) cu(cudaEventCreateWithFlags(&h->poll_ev[i], cudaEventDisableTiming), "cudaEventCreate");
  if (rc < 0) {          // a half-built handle is released, not leaked
    cudaGetLastError();
    nnmpc_sim_destroy(h);
    return rc;
  }
  *out = h;
  return 0;
}

int nnmpc_sim_destroy(nnmpc_sim_t* h) {
  if (!h) return 0;
  DeviceGuard dg(h->device);
  if (h->ABd) cudaFree(h->ABd);
  if (h->counts) cudaFree(h->counts);
  if (h->rowiters) cudaFree(h->rowiters);
  if (h->stats) cudaFree(h->stats);
  if (h->tile_stat) cudaFree(h->tile_stat);
  if (h->pin) cudaFreeHost(h->pin);
  h->lps.release();
  h->ozr.release();
  h->lp_layout.release();
  h->dlast.release();
  h->need2.release();
  for (int i = 0; i < POLL_RING; ++i)
    if (h->poll_ev[i]) cudaEventDestroy(h->poll_ev[i]);
  h->x0.release(); h->lb.release(); h->ub.release(); h->us_prev.release(); h->dus.release(); h->V.release();
  h->Z.release(); h->xcur.release(); h->upcur.release(); h->kappa.release(); h->dtrig.release();
  h->chunk.release(); h->cold.release();
  h->state.release(); h->tcur.release(); h->it.release(); h->lists.release(); h->dres.release(); h->kres.release();
  h->h_sp.release(); h->h_dist.release(); h->h_x.release(); h->h_uprev.release(); h->h_xs.release();
  h->h_us.release(); h->h_u.release(); h->h_kkt.release(); h->h_xio.release(); h->h_upio.release();
  h->h_iters.release();
  h->gcap.release();
  delete h;
  return 0;
}

int nnmpc_sim_set_precision(nnmpc_sim_t* h, int mode) {
  if (!h) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_set_precision: null handle");
  if (mode != NNMPC_PRECISION_F64 && mode != NNMPC_PRECISION_MIXED)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_set_precision: unknown mode %d", mode);
  if (h->mixed != (mode == NNMPC_PRECISION_MIXED)) h->warm_B = 0;   // solver state is not shared between the modes
  h->mixed = mode == NNMPC_PRECISION_MIXED;
  return 0;
}

int nnmpc_sim_set_slots(nnmpc_sim_t* h, int slots) {
  if (!h) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_set_slots: null handle");
  if (slots < 1) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_set_slots: need at least one slot");
  h->slot_cap = slots;
  h->warm_B = 0;
  return 0;
}

int nnmpc_sim_set_cadence(nnmpc_sim_t* h, int cadence) {
  if (!h) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_set_cadence: null handle");
  if (cadence < 1 || cadence > 8) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_set_cadence: cadence must be in 1..8");
  h->cadence = cadence;
  return 0;
}

int nnmpc_sim_set_tail_rows(nnmpc_sim_t* h, int rows) {
  if (!h) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_set_tail_rows: null handle");
  h->tail_rows = rows < 0 ? -1 : rows;
  return 0;
}

int nnmpc_sim_set_exact_gemm(nnmpc_sim_t* h, int mode) {
  if (!h) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_set_exact_gemm: null handle");
  if (mode != 0 && mode != 1) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_set_exact_gemm: mode must be 0 (DMMA) or 1 (INT8 slices)");
  h->exact_oz = mode;
  return 0;
}

int nnmpc_sim_set_capture(nnmpc_sim_t* h, double* useq_dev, double* cost_dev) {
  if (!h) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_set_capture: null handle");
  h->cap_useq = useq_dev;
  h->cap_cost = cost_dev;
  return 0;
}

int nnmpc_sim_set_one_term_threshold(nnmpc_sim_t* h, double factor) {
  if (!h) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_set_one_term_threshold: null handle");
  if (!(factor >= 0.0) || !(factor <= 1e12)) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_set_one_term_threshold: factor must be in [0, 1e12]");
  h->t2_factor = factor;
  return 0;
}

int nnmpc_sim_tile_stats(nnmpc_sim_t* h, long long* out3) {
  if (!h || !out3) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_tile_stats: null argument");
  DeviceGuard dg(h->device);
  unsigned long long t[3] = {0, 0, 0};
  NNMPC_CUDA(cudaMemcpy(t, h->tile_stat, sizeof(t), cudaMemcpyDeviceToHost));
  out3[0] = (long long)t[0]; out3[1] = (long long)t[1]; out3[2] = (long long)t[2];
  return 0;
}

int nnmpc_sim_set_second_term_cadence(nnmpc_sim_t* h, int every) {
  if (!h) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_set_second_term_cadence: null handle");
  if (every < 0 || every > 64) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_set_second_term_cadence: need 0 <= every <= 64");
  h->t2_every = every;
  h->t2_auto = false;
  h->warm_B = 0;        // the next run starts from cold operand buffers (pending sums are allocated on demand)
  return 0;
}

int nnmpc_sim_active_stats(nnmpc_sim_t* h, long long* out2) {
  if (!h || !out2) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_active_stats: null argument");
  out2[0] = h->tot_qps_active; out2[1] = h->tot_active;
  return 0;
}

int nnmpc_sim_stats(nnmpc_sim_t* h, long long* out4) {
  if (!h || !out4) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_stats: null argument");
  out4[0] = h->tot_rowiters; out4[1] = h->tot_anchors; out4[2] = h->tot_verifies; out4[3] = h->tot_qps;
  return 0;
}

int nnmpc_sim_run(nnmpc_sim_t* h, int B, int T, double* x_io, double* uprev_io, const double* setpoints,
                  const double* disturbances, double* x, double* uprev, double* xs, double* us, double* u, int* iters,
                  double* kkt, double tol, int max_iter, int resume, void* stream) {
  if ((B == 0 || T == 0) && h) return 0;
  if (!h || !x_io || !uprev_io || !setpoints || !disturbances || !x || !uprev || !xs || !us || !u)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_run: null argument");
  if (B < 0 || T < 0) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_run: negative size");
  if (!h->ts) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_run: this handle was created without a target selector (batched-QP use only)");
  DeviceGuard dg(h->device);
  return sim_run_device(h, B, T, x_io, uprev_io, setpoints, disturbances, x, uprev, xs, us, u, iters, kkt, tol,
                        max_iter, resume, (cudaStream_t)stream);
}

int nnmpc_sim_solve_qps(nnmpc_sim_t* h, int B, const double* x0, const double* lb, const double* ub, double* u, double* cost,
                        double* kkt, int* iters, double tol, int max_iter, void* stream) {
  if (B == 0 && h) return 0;
  if (!h || !x0 || !lb || !ub || !u) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_solve_qps: null argument");
  if (B < 0) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_solve_qps: negative batch");
  DeviceGuard dg(h->device);
  QpBatch qb{x0, lb, ub, u, cost};
  return sim_run_device(h, B, 1, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, iters, kkt,
                        tol, max_iter, 0, (cudaStream_t)stream, &qb);
}

int nnmpc_sim_run_host(nnmpc_sim_t* h, int B, int T, double* x_io, double* uprev_io, const double* setpoints,
                       const double* disturbances, double* x, double* uprev, double* xs, double* us, double* u,
                       int* iters, double* kkt, double tol, int max_iter, int resume) {
  if ((B == 0 || T == 0) && h) return 0;
  if (!h || !x_io || !uprev_io || !setpoints || !disturbances || !x || !uprev || !xs || !us || !u)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_run_host: null argument");
  if (B <= 0 || T <= 0) return (B == 0 || T == 0) ? 0 : set_error(NNMPC_ERR_BADARG, "nnmpc_sim_run_host: negative size");
  if (!h->ts) return set_error(NNMPC_ERR_BADARG, "nnmpc_sim_run_host: this handle was created without a target selector");
  DeviceGuard dg(h->device);
  const size_t bt = (size_t)B * T;
  const int nx = h->nx, nu = h->nu, nd = h->nd, ny = h->ny;
  NNMPC_TRY(h->h_sp.ensure(bt * ny));
  NNMPC_TRY(h->h_dist.ensure(bt * (nd > 0 ? nd : 1)));
  NNMPC_TRY(h->h_x.ensure(bt * nx));
  NNMPC_TRY(h->h_xs.ensure(bt * nx));
  NNMPC_TRY(h->h_uprev.ensure(bt * nu));
  NNMPC_TRY(h->h_us.ensure(bt * nu));
  NNMPC_TRY(h->h_u.ensure(bt * nu));
  NNMPC_TRY(h->h_kkt.ensure(bt));
  NNMPC_TRY(h->h_iters.ensure(bt));
  NNMPC_TRY(h->h_xio.ensure((size_t)B * nx));
  NNMPC_TRY(h->h_upio.ensure((size_t)B * nu));
  cudaStream_t st = 0;
  NNMPC_CUDA(cudaMemcpyAsync(h->h_sp.p, setpoints, bt * ny * 8, cudaMemcpyHostToDevice, st));
  if (nd > 0) NNMPC_CUDA(cudaMemcpyAsync(h->h_dist.p, disturbances, bt * nd * 8, cudaMemcpyHostToDevice, st));
  NNMPC_CUDA(cudaMemcpyAsync(h->h_xio.p, x_io, (size_t)B * nx * 8, cudaMemcpyHostToDevice, st));
  NNMPC_CUDA(cudaMemcpyAsync(h->h_upio.p, uprev_io, (size_t)B * nu * 8, cudaMemcpyHostToDevice, st));
  double* const keep_useq = h->cap_useq;
  double* const keep_cost = h->cap_cost;
  h->cap_useq = h->cap_cost = nullptr;       // the capture sinks belong to the device entry point
  int rc = sim_run_device(h, B, T, h->h_xio.p, h->h_upio.p, h->h_sp.p, h->h_dist.p, h->h_x.p, h->h_uprev.p, h->h_xs.p,
                          h->h_us.p, h->h_u.p, h->h_iters.p, h->h_kkt.p, tol, max_iter, resume, st);
  h->cap_useq = keep_useq;
  h->cap_cost = keep_cost;
  if (rc < 0) return rc;
  NNMPC_CUDA(cudaMemcpyAsync(x, h->h_x.p, bt * nx * 8, cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaMemcpyAsync(xs, h->h_xs.p, bt * nx * 8, cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaMemcpyAsync(uprev, h->h_uprev.p, bt * nu * 8, cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaMemcpyAsync(us, h->h_us.p, bt * nu * 8, cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaMemcpyAsync(u, h->h_u.p, bt * nu * 8, cudaMemcpyDeviceToHost, st));
  if (iters) NNMPC_CUDA(cudaMemcpyAsync(iters, h->h_iters.p, bt * 4, cudaMemcpyDeviceToHost, st));
  if (kkt) NNMPC_CUDA(cudaMemcpyAsync(kkt, h->h_kkt.p, bt * 8, cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaMemcpyAsync(x_io, h->h_xio.p, (size_t)B * nx * 8, cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaMemcpyAsync(uprev_io, h->h_upio.p, (size_t)B * nu * 8, cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaStreamSynchronize(st));
  return rc;
}

}  // extern "C"
