/* nnmpc.h — C ABI of libnnmpc.so: the B200 (sm_100a) linear-MPC / structured-NN hot path.
 *
 * The reference (pratyushkumar211/industrial_nnmpc_2021) is pure Python and has no FFI; its
 * boundary for this path is the Python object API of lib/linearMPC.py and lib/LinearMPCLayers.py.
 * Each entry point below names the reference method it replaces (file:line in /root/reference).
 * The Python drop-ins in industrial_nnmpc_2021_b200/ bind these with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - all matrices are float64, row-major, contiguous unless a stride is named;
 *  - "host" pointers are ordinary CPU memory, "dev" pointers are CUDA device memory on the
 *    handle's device (e.g. torch.Tensor.data_ptr()); `stream` is a cudaStream_t (NULL = default);
 *  - every function returns 0 on success, a negative nnmpc_status on error (message through
 *    nnmpc_last_error(), thread-local) and a positive bit mask of warnings otherwise:
 *    NNMPC_WARN_MAXITER (some regulator QP hit max_iter), NNMPC_WARN_TARGET (some target-selector
 *    solve did not reach its optimum);
 *  - the caller owns every buffer it passes; handles own only the replicated operators and
 *    scratch, released by *_destroy; one device per handle.
 *  - threading: the OPERATORS of a handle never change after create (nnmpc_qp_set_penalty and
 *    nnmpc_ts_set_output_bounds complete the create of a regulator / target-selector handle and are called
 *    once, before the first solve; the one exception is nnmpc_mlp_train_step, which updates the weights
 *    of a network handle in place - that is its purpose), but a handle also
 *    owns solver SCRATCH and, for nnmpc_sim, the run options of the nnmpc_sim_set_* calls: one call
 *    at a time per handle (the reference's objects are single-threaded too, lib/linearMPC.py:685-686
 *    mutates the regulator on every call).  Different handles are independent and may be driven from
 *    different host threads / streams concurrently; nothing is global except the launch counters and
 *    the optional profiling spans of nnmpc_prof_* (mutex protected, off by default).
 */
#ifndef NNMPC_H
#define NNMPC_H
#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  NNMPC_OK = 0,
  NNMPC_WARN_MAXITER = 1,
  NNMPC_WARN_TARGET = 2,
  NNMPC_ERR_BADARG = -1,
  NNMPC_ERR_CUDA = -2,
  NNMPC_ERR_NOMEM = -3,
  NNMPC_ERR_UNSUPPORTED = -4
} nnmpc_status;

typedef struct nnmpc_qp nnmpc_qp_t;    /* condensed regulator QP operators + solver scratch */
typedef struct nnmpc_ts nnmpc_ts_t;    /* target-selector operators */
typedef struct nnmpc_sim nnmpc_sim_t;  /* closed-loop offline data generator */
typedef struct nnmpc_mlp nnmpc_mlp_t;  /* structured-network weights */
typedef struct nnmpc_online nnmpc_online_t;  /* batched online closed loop (filter + controller + plant) */

int nnmpc_version(void);
const char* nnmpc_last_error(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
long long nnmpc_launch_count(void);
/* sum over all solved samples of the Douglas-Rachford iterations they used (for flop accounting) */
long long nnmpc_iteration_count(void);
/* Live timing of the dominant kernel (the regulator-QP iteration GEMM) for bench.py's roofline:
 * when enabled, every group of back-to-back iteration launches is bracketed by CUDA events on the
 * stream it is launched on.  nnmpc_prof_read synchronises those events and returns the summed
 * device time [ms], the algorithmic flops (active samples x 2 n^2 per launch) and the number of
 * launches since the last reset.  Disabled by default (no events are recorded). */
int nnmpc_prof_enable(int on);
int nnmpc_prof_read(double* ms, double* flops, long long* launches, int reset);
/* Same with two channels (arrays of 2): [0] the iteration passes (FP64 DMMA GEMM, or the tcgen05 pass
 * of the mixed-precision mode), [1] the FP64 anchor / exact-check GEMMs of the mixed-precision mode. */
int nnmpc_prof_read2(double* ms, double* flops, long long* launches, int reset);
/* up to 4 channels: 0 iteration passes, 1 exact anchors / KKT checks, 2 FP64 tail iterations, 3 rest of a full engine loop */
int nnmpc_prof_readn(int nchan, double* ms, double* flops, long long* launches, int reset);

/* ---- regulator QP:  DenseQPRegulator (lib/linearMPC.py:321-517) -------------------------------
 *   min_u 1/2 u'Pu + (tq x0)'u   s.t.  lb <= u_k <= ub  for every stage k     (box path, :481)
 * Operators (host, uploaded once; built by industrial_nnmpc_2021_b200.condense):
 *   P     n x n      Hessian (:472)                       tq    n x nxa   linear-term map (:473)
 *   Top   n x n      (P + diag(rho))^-1 diag(rho)          Mtq   n x nxa   (P + diag(rho))^-1 tq
 *   Kunc  n x nxa    -P^-1 tq  (unconstrained law; equals the LQR sequence, :356)
 *   n = N*nu must be even, nxa even (pad with a zero column otherwise). */
int nnmpc_qp_create(nnmpc_qp_t** out, int n, int nxa, int nu, int N,
                    const double* P_host, const double* tq_host, const double* Top_host,
                    const double* Mtq_host, const double* Kunc_host, double alpha, int device);
/* Regulator of a re-parameterised (open-loop unstable) plant, u = K x + v, solved in v by a primal-dual interior-point
 * method (Mehrotra predictor-corrector, one Riccati recursion per Newton step; industrial_nnmpc_2021_b200/csrc/ipm.cu)
 * on the stagewise form of the reference's general-G QP (lib/linearMPC.py:366-382, :476-493):
 *   min 1/2 sum_{k<N} (x_k'Q x_k + v_k'R v_k + 2 x_k'M v_k) + 1/2 x_N'Pf x_N
 *   s.t. x_{k+1} = A x_k + B v_k,  x_0 = x0,  lb <= K x_k + v_k <= ub      (A = A_open + B K stable)
 * Host arrays, row-major, padded with zeros to nxa_ld states: A, Q, Pf nxa_ld x nxa_ld, B, M nxa_ld x nu, R nu x nu,
 * K nu x nxa_ld.  nxa_ld <= 64 and nu <= 32 (NNMPC_ERR_UNSUPPORTED otherwise).  The handle is an ordinary regulator:
 * nnmpc_qp_solve[_host], nnmpc_online_run and nnmpc_sim_* accept it.  Through it u = K x + v along the forward roll-out
 * (the reference's output, :507-509); v_state / warm are ignored (every solve starts cold); kkt is the relative KKT
 * certificate of ipm.cu at the returned point; cost is the reference's objective 1/2 v'Pv + (tq x0)'v (not the u-space
 * value the Douglas-Rachford path reports); iters counts interior-point iterations.  A sample with lb >= ub somewhere,
 * a NaN bound or a non-finite x0 returns NaN with iters = max_iter (NNMPC_WARN_MAXITER); a bound at +-Inf is absent.
 * nnmpc_qp_set_penalty refuses the handle (NNMPC_ERR_BADARG).  nnmpc_sim_create builds a lock-step engine on it
 * (per step: target selector, interior-point QPs, dataset rows and plant step over the whole batch); the precision,
 * slots, cadence, tail, exact-GEMM, one-term and second-term setters are accepted and have no effect, and
 * nnmpc_sim_stats reports interior-point iterations as row-iterations. */
int nnmpc_qp_create_ipm(nnmpc_qp_t** out, int nxa_ld, int nu, int N, const double* A_host, const double* B_host,
                        const double* Q_host, const double* R_host, const double* M_host, const double* Pf_host,
                        const double* K_host, int device);
/* The ADMM penalty vector rho (host, n doubles, all > 0) behind Top = (P + diag(rho))^-1 diag(rho).  Needed by the
 * mixed-precision closed loop (nnmpc_sim_set_precision), which re-anchors x = Top w - c from the exact gradient
 * g = P z + q of its KKT checks:  w := z + g / rho  gives  x = z  exactly. */
int nnmpc_qp_set_penalty(nnmpc_qp_t* h, const double* rho_host);
int nnmpc_qp_destroy(nnmpc_qp_t* h);

/* Batched solve; replaces one DenseQPRegulator.solve(x0) per sample (:495-512) with the bounds
 * mutation of LinearMPCController.get_control_sequence (:685-686) passed per sample instead.
 *   x0     dev B x nxa   deviation state [x-xs; uprev-us] (:688)
 *   lb,ub  dev B x nu    per-sample stage bounds ulb-us, uub-us
 *   u      dev B x n     out: minimiser (deviation variables; caller adds us, :689)
 *   v_state dev B x n    in/out Douglas-Rachford state for warm starts, or NULL;  warm != 0 uses it
 *   cost,kkt dev B       out (nullable): optimal value 1/2u'Pu+q'u and ||u-clip(u-(Pu+q))||_inf
 *   iters  dev B int     out (nullable): iterations used per sample
 * Stops each sample when its true KKT residual (evaluated with P in FP64) <= tol. */
int nnmpc_qp_solve(nnmpc_qp_t* h, int B, const double* x0, const double* lb, const double* ub,
                   double* u, double* v_state, int warm, double* cost, double* kkt, int* iters,
                   double tol, int max_iter, void* stream);
/* Same with HOST buffers (copies in/out inside the call); the end-to-end entry point. */
int nnmpc_qp_solve_host(nnmpc_qp_t* h, int B, const double* x0, const double* lb, const double* ub,
                        double* u, double* cost, double* kkt, int* iters, double tol, int max_iter);

/* ---- target selector:  TargetSelector.solve (lib/linearMPC.py:298-311) -------------------------
 * nnmpc_ts_create: H empty and I - A invertible.
 * Reduced exactly to the nu-dim box QP  min 1/2 us'Ht us + (Fy ysp + Fd d + f0)'us,
 * xs = Gx us + Gd d  (Gx = (I-A)^-1 B, Gd = (I-A)^-1 Bd).  nu <= 32. */
int nnmpc_ts_create(nnmpc_ts_t** out, int nx, int nu, int ny, int nd, const double* Ht_host,
                    const double* Fy_host, const double* Fd_host, const double* f0_host,
                    const double* Gx_host, const double* Gd_host, const double* ulb_host,
                    const double* uub_host, int device);
/* Output-constrained targets, ylb <= C xs + Cd dhat <= yub next to the input box (the ylb/yub branch of
 * TargetSelector, lib/linearMPC.py:242-248, :284-288).  Host arrays, row-major, built by the caller from the same
 * reduction as nnmpc_ts_create (xs = Gx us + Gd dhat):  Hinv = Ht^-1 (nu x nu), Abar = [C Gx; I] ((ny + nu) x nu),
 * AH = Abar Hinv, Mbar = Abar Hinv Abar' ((ny + nu)^2), Ryd = C Gd + Cd (ny x nd), ylb, yub (ny).  From then on every
 * solve through this handle (nnmpc_ts_solve*, the closed-loop engine, the online loop) runs an exact dual active-set
 * method (one warp per sample) over the ny + nu two-sided rows; an infeasible sample raises NNMPC_WARN_TARGET and carries
 * a negative iteration count.  ny + nu <= 160.  Call once, before the first solve. */
int nnmpc_ts_set_output_bounds(nnmpc_ts_t* h, const double* Hinv_host, const double* Abar_host, const double* AH_host,
                               const double* Mbar_host, const double* Ryd_host, const double* ylb_host,
                               const double* yub_host);
/* Targets with pinned outputs (H non-empty: H C xs = H (ysp - Cd dhat)) or an integrating plant (I - A singular),
 * where xs cannot be eliminated through (I - A)^-1.  With s = [ysp; dhat] (ny + nd) and an orthonormal basis Z of
 * null(tA), tA = [I-A, -B; HC, 0] of full row rank, the targets are [xs; us] = K s + Z v, K = tA^+ tb, for the nw =
 * nu - nz remaining variables v, which solve
 *     min 1/2 v'(Z'PZ) v + (Fy ysp + Fd dhat + f0)'v   s.t.  lo0 - R s <= Abar v <= hi0 - R s   (mb rows).
 * Host arrays, row-major:  Hinv = (Z'PZ)^-1 (nw x nw), Abar (mb x nw), AH = Abar Hinv (mb x nw), Mbar = Abar Hinv Abar'
 * (mb x mb), Fy (nw x ny), Fd (nw x nd), f0 (nw), R (mb x (ny + nd)), lo0, hi0 (mb), Kx (nx x (ny + nd)),
 * Ku (nu x (ny + nd)), Zx (nx x nw), Zu (nu x nw), ulb, uub (nu).  The last nu rows are the input box in input order
 * (Abar = Zu, R = Ku, lo0 = ulb, hi0 = uub); the first mb - nu rows are free to use, e.g. output bounds
 * (Abar = C Zx, R = C Kx + [0 Cd], lo0 = ylb, hi0 = yub).  nu <= 32, 0 <= nw <= nu, nu <= mb <= 160.
 * nw = 0 is valid: the target is K s, and a sample whose K s violates a row is infeasible; the arrays of size zero
 * (Hinv, Abar, AH, Fy, Fd, f0, Zx, Zu) may then be NULL.  Solved by the dual active-set method of
 * nnmpc_ts_set_output_bounds; nnmpc_ts_solve*, nnmpc_sim_* and nnmpc_online_* take the handle unchanged, and an
 * infeasible sample raises NNMPC_WARN_TARGET and carries a negative iteration count. */
int nnmpc_ts_create_reduced(nnmpc_ts_t** out, int nx, int nu, int ny, int nd, int nw, int mb, const double* Hinv_host,
                            const double* Abar_host, const double* AH_host, const double* Mbar_host,
                            const double* Fy_host, const double* Fd_host, const double* f0_host, const double* R_host,
                            const double* lo0_host, const double* hi0_host, const double* Kx_host,
                            const double* Ku_host, const double* Zx_host, const double* Zu_host,
                            const double* ulb_host, const double* uub_host, int device);
int nnmpc_ts_destroy(nnmpc_ts_t* h);
/* ysp: dev B rows of ny doubles, row stride ysp_stride (doubles); d likewise. */
/* iters (nullable): active-set steps per sample; a sample whose solve stalled at the step cap or went
 * non-finite gets the NEGATED count -(steps+1) (and the host entry point returns NNMPC_WARN_TARGET). */
int nnmpc_ts_solve(nnmpc_ts_t* h, int B, const double* ysp, long long ysp_stride, const double* d,
                   long long d_stride, double* xs, double* us, int* iters, void* stream);
int nnmpc_ts_solve_host(nnmpc_ts_t* h, int B, const double* ysp, const double* d, double* xs,
                        double* us, int* iters);

/* ---- closed-loop offline data generation: simulate_offline (lib/linearMPC.py:827-880) ---------
 * B independent trajectories (the reference's processes, :786-825) advanced T steps together:
 * target selector -> regulator QP (warm started) -> u = useq[0:nu] -> x+ = Ax + Bu + Bd d.
 *   ABd    host nx x (nx+nu+nd): [A | B | Bd]
 * Inputs  setpoints dev [B][T][ny], disturbances dev [B][T][nd]  (chunk-major, as _split_scenarios)
 * Outputs x,xs dev [B][T][nx]; uprev,us,u dev [B][T][nu]  (row t = state BEFORE step t, :868-872)
 *         iters dev [B][T] int, kkt dev [B][T] (nullable)
 *   x_io, uprev_io dev B x nx / B x nu: in = initial state (:837-838), out = state after T steps
 *   resume != 0: the call continues the SAME B trajectories as the previous call on this handle
 *   (long trajectories advanced in slabs); the solver then warm-starts step 0 from the state it
 *   kept.  It only changes iteration counts, never which optimum is returned. */
int nnmpc_sim_create(nnmpc_sim_t** out, nnmpc_qp_t* qp, nnmpc_ts_t* ts, int nx, int nu, int nd,
                     int ny, const double* ABd_host, int device);
int nnmpc_sim_destroy(nnmpc_sim_t* h);
/* Arithmetic of the regulator-QP iteration inside the closed loop ("FP64 DMMA, or FP32 with FP64
 * residual refinement" of the north star).  Either way every returned solution has passed a KKT check
 * evaluated with P in FP64 (lib/linearMPC.py:503 is replaced by a certified optimum, not an estimate).
 *   NNMPC_PRECISION_F64    every iteration is an FP64 tensor-core (DMMA) GEMM with Top
 *   NNMPC_PRECISION_MIXED  iterations run on the tcgen05 tensor cores: fp16 increments of the operand
 *                          against a two-term fp16 split of Top, fp32 accumulation in TMEM, all solver
 *                          state in FP64; an FP64-accurate "anchor" x = Top w - c starts every QP and an
 *                          FP64-accurate KKT check g = P z + q certifies it (both on the INT8 tensor cores by
 *                          error-free slicing, or on FP64 DMMA: nnmpc_sim_set_exact_gemm); a check that fails
 *                          re-anchors the iteration from its own gradient */
enum { NNMPC_PRECISION_F64 = 0, NNMPC_PRECISION_MIXED = 1 };
int nnmpc_sim_set_precision(nnmpc_sim_t* h, int mode);
/* At most `slots` trajectories advance concurrently (default 8192).  A call with B > slots queues the
 * remaining chunks: a slot that finishes its chunk immediately takes the next one (cold start from
 * that chunk's x_io/uprev_io row), so the batch stays full until the queue is empty - the continuous
 * batching that replaces the reference's one-OS-process-per-chunk fan-out (lib/linearMPC.py:817-825).
 * With B > slots `resume` is ignored (every chunk starts cold). */
int nnmpc_sim_set_slots(nnmpc_sim_t* h, int slots);
/* Mixed mode only: the FP64 phases (anchors, exact checks, plant step, next targets) run every
 * `cadence`-th engine loop over the rows that accumulated meanwhile (default 4; 1 = every loop). */
int nnmpc_sim_set_cadence(nnmpc_sim_t* h, int cadence);
/* Mixed mode only: once at most `rows` trajectories of a call are still running, the rest of the call
 * iterates with skinny FP64 GEMMs over just those rows instead of full tensor-core passes
 * (rows < 0: automatic, max(48, B/256); 0: never). */
int nnmpc_sim_set_tail_rows(nnmpc_sim_t* h, int rows);
/* Mixed mode only: which tensor pipe evaluates the FP64-exact operator applies (anchors x = Top w - c, KKT checks
 * g = P z + q): 1 (default) = INT8 tcgen05 with error-free slicing (FP64-accurate, see oz_gemm.cuh), 0 = FP64 DMMA. */
int nnmpc_sim_set_exact_gemm(nnmpc_sim_t* h, int mode);
/* Mixed mode only: a trajectory whose last Douglas-Rachford residual ||d||_inf is at most factor * tol is in the late
 * phase of its QP; 128-row operand tiles made of such rows only run the tensor-core pass with the first fp16 operator
 * term alone (half the MMA work; the 2^-11 relative error of the dropped term is relative to a vanishing increment and
 * every result is still certified by the exact KKT check).  Default 0 = always both terms: measured on B200, only
 * 0.4 - 6 % of the tiles qualify (trajectories restart inside late tiles between re-layouts) and a row's arithmetic would
 * depend on its neighbours; factors up to 1e4 left iterations and exact checks per QP unchanged. */
int nnmpc_sim_set_one_term_threshold(nnmpc_sim_t* h, double factor);
/* cumulative since create: out3 = {128x128 tensor-core tiles of the iteration passes run with one operator term, with
 * both terms, tiles of the second-term delivery passes} */
int nnmpc_sim_tile_stats(nnmpc_sim_t* h, long long* out3);
/* Mixed mode only: the tensor-core pass multiplies the first fp16 operator term alone, and the second term (a 2^-11
 * relative correction, linear in the increments) is delivered every `every`-th pass for all increments since the last
 * delivery at once, by a one-term GEMM over the pending sums (rounded up to a multiple of the cadence; default 8;
 * 0 = both terms in every pass, the round-1 form; a handle this is never called on defers only for n >= 1536, below
 * which the MMAs are a small part of the pass).  MMA work per iteration falls from 2 to 1 + 1/every products;
 * fixed points and the exact KKT certification of every returned point are unchanged. */
int nnmpc_sim_set_second_term_cadence(nnmpc_sim_t* h, int every);
/* Optional per-QP sinks for the following nnmpc_sim_run calls (device pointers, either may be NULL; NULL, NULL
 * switches the capture off): useq [B][T][n] = the whole optimal input sequence of every regulator QP with the
 * target added back per stage - what get_control_sequence returns (lib/linearMPC.py:689) and DenseQPRegulator
 * keeps in .useq (:511) - and cost [B][T] = the optimal value 1/2 u'Pu + q'u in deviation variables.  Meant for
 * parity tests and diagnostics at small B*T (n doubles per sample); nnmpc_sim_run_host ignores it. */
int nnmpc_sim_set_capture(nnmpc_sim_t* h, double* useq_dev, double* cost_dev);
/* cumulative since create: out4 = {row-iterations, exact anchors, exact KKT checks, QPs solved} */
int nnmpc_sim_stats(nnmpc_sim_t* h, long long* out4);
/* cumulative since create: out2 = {QPs whose optimum has at least one active bound, active bounds in total} -
 * how constrained the workload is (bench.py reports it next to the condition number of P) */
int nnmpc_sim_active_stats(nnmpc_sim_t* h, long long* out2);
int nnmpc_sim_run(nnmpc_sim_t* h, int B, int T, double* x_io, double* uprev_io,
                  const double* setpoints, const double* disturbances, double* x, double* uprev,
                  double* xs, double* us, double* u, int* iters, double* kkt, double tol,
                  int max_iter, int resume, void* stream);
/* Batched regulator QPs through the engine (the data-parallel form of DenseQPRegulator.solve, lib/linearMPC.py:495-512):
 * B independent QPs, each its own x0 (B x nxa) and stage bounds lb/ub (B x nu), solved cold with continuous batching
 * over the handle's slots - the arithmetic (nnmpc_sim_set_precision: tcgen05 fp16 increments + INT8-exact anchors and
 * KKT checks, or FP64) and the certification are those of nnmpc_sim_run.  u (B x n) minimisers in deviation
 * variables; cost, kkt, iters (B, nullable).  The handle may have been created with ts = NULL, ABd_host = NULL,
 * nx = nxa - nu, nd = ny = 0. */
int nnmpc_sim_solve_qps(nnmpc_sim_t* h, int B, const double* x0, const double* lb, const double* ub, double* u,
                        double* cost, double* kkt, int* iters, double tol, int max_iter, void* stream);
int nnmpc_sim_run_host(nnmpc_sim_t* h, int B, int T, double* x_io, double* uprev_io,
                       const double* setpoints, const double* disturbances, double* x, double* uprev,
                       double* xs, double* us, double* u, int* iters, double* kkt, double tol,
                       int max_iter, int resume);

/* ---- structured network: RegulatorLayerWithUprev / WithoutUprev (lib/LinearMPCLayers.py:15-115)
 * and its NumPy deployment form NeuralNetworkController (lib/controller_evaluation.py:863-892).
 *   u = us + f(x,[uprev],xs,us) - f(xs,[us],xs,us),  f = (Dense+ReLU) x (L-1), Dense(no bias)
 * weights: Keras get_weights() order [W1,b1,...,W_{L-1},b_{L-1},Wout], W_i (in_i x out_i) row-major;
 * dims[0..L] = layer widths with dims[0] = input width (2nx+2nu or 2nx+nu), dims[L] = nu. */
int nnmpc_mlp_create(nnmpc_mlp_t** out, int nx, int nu, int with_uprev, int num_layers,
                     const int* dims, const double* const* weights_host,
                     const double* const* biases_host, int device);
int nnmpc_mlp_destroy(nnmpc_mlp_t* h);
/* Arithmetic of the Dense layers: 1 (default) = INT8 tcgen05 tensor cores - activations and weights as 4 signed
 * base-128 digit planes, the 10 digit-plane products of levels 0..3 accumulated exactly in INT32, FP64 bias / ReLU /
 * output assembly: ~1e-7 of the float64 layer, steady-state identity u = us exact; 0 = FP64 DMMA GEMMs (~1e-13);
 * 2 = split-fp16 tcgen05 GEMMs with fp32 TMEM accumulation (~2e-5: outside the 1e-5 tolerance, comparison only). */
int nnmpc_mlp_set_precision(nnmpc_mlp_t* h, int mode);
/* One training step of the structured network as cdu_train.py:24-62 / cstrs_train.py:24-61 fit it with Keras
 * (optimizer='adam', loss='mean_squared_error'): FP64 forward, loss = mean over B x nu of (us + f(x,..) - f(xs,..) - u)^2,
 * backward through both network passes, Adam update (Keras: lr_t = lr sqrt(1-beta2^t)/(1-beta1^t),
 * w -= lr_t m / (sqrt(v) + eps); defaults lr 1e-3, beta 0.9 / 0.999, eps 1e-7) with t = step (1-based).  apply = 0:
 * forward and loss only (validation).  All pointers device memory, B <= 262144; loss_host (nullable) receives the loss
 * of THIS batch before the update.  The inference operators are rebuilt lazily before the next forward. */
int nnmpc_mlp_train_step(nnmpc_mlp_t* h, long long B, const double* x, const double* uprev, const double* xs,
                         const double* us, const double* u_target, double lr, double beta1, double beta2, double eps,
                         long long step, int apply, double* loss_host, void* stream);
/* current weights in Keras get_weights() layout: weights_host[l] (in_l x out_l), biases_host[l] (out_l; NULL for the last) */
int nnmpc_mlp_get_weights(nnmpc_mlp_t* h, double* const* weights_host, double* const* biases_host);
/* x,xs dev B x nx; uprev,us dev B x nu (uprev ignored when !with_uprev); out dev B x nu.
 * xscale dev nx or NULL (x/xscale, xs/xscale, :863-866); ulb/uub dev nu or NULL (clip, :888-892).
 * Non-finite inputs: samples are independent, so a NaN or an infinity in one sample leaves every other sample
 * bit-identical.  A sample with a NaN in x, uprev, xs or us comes back NaN in every component, in every mode and with
 * or without the clip: ReLU and the clip keep a NaN, as the reference's np.where forms do.  An infinity gives a
 * non-finite output wherever the float64 reference is non-finite; in modes 1 and 2 the whole sample may come back
 * NaN, because a row holding an infinity has no finite scale. */
int nnmpc_mlp_forward(nnmpc_mlp_t* h, long long B, const double* x, const double* uprev,
                      const double* xs, const double* us, const double* xscale, const double* ulb,
                      const double* uub, double* out, void* stream);
int nnmpc_mlp_forward_host(nnmpc_mlp_t* h, long long B, const double* x, const double* uprev,
                           const double* xs, const double* us, const double* xscale,
                           const double* ulb, const double* uub, double* out);

/* ---- batched online closed loop: LinearMPCController.control_law / online_simulation (lib/linearMPC.py:646-669,
 * :703-718) and the validation study of lib/controller_evaluation.py:322-523 for S scenarios in lock step ---------
 * Every step: Kalman filter (:133-176) -> target selector -> controller -> running average stage cost (:691-701)
 * -> plant step and next measurement (:87-131).  Host operators (row-major):
 *   Fkf  (nx+nd) x (nx+nd+nu+ny)   [(I - L Caug) Aaug | (I - L Caug) Baug | L]  acting on [xhat; dhat; uprev; y]
 *   Fpl  (nx+ny) x (nx+nu+np)      [A B Bp; CA CB CBp]                           acting on [x; u; p]
 *   Kaug nu x (nx+nu)              saturated-LQR gain (nullable), Qaug/Raug/Maug the augmented stage cost (:626-644)
 *   xscale nx (nullable)           state scaling of the network inputs (controller_evaluation.py:863-866)
 * qp / mlp may be NULL when the corresponding controller kind is not used; handles must live on `device`. */
enum { NNMPC_ONLINE_MPC = 0, NNMPC_ONLINE_NN = 1, NNMPC_ONLINE_SATDLQR = 2 };
int nnmpc_online_create(nnmpc_online_t** out, nnmpc_qp_t* qp, nnmpc_ts_t* ts, nnmpc_mlp_t* mlp, int nx, int nu, int ny,
                        int nd, int np, const double* Fkf_host, const double* Fpl_host, const double* Kaug_host,
                        const double* Qaug_host, const double* Raug_host, const double* Maug_host,
                        const double* ulb_host, const double* uub_host, const double* xscale_host, int device);
int nnmpc_online_destroy(nnmpc_online_t* h);
/* All pointers are device memory.  In/out per scenario: x_io S x nx (plant state), xhat_io S x (nx+nd) (filter state
 * [xhat; dhat]), uprev_io S x nu.  Inputs: setpoints [S][T][ny], disturbances [S][T][np], noise [S][T+1][ny]
 * (measurement noise added to C x, entry 0 unused; nullable), y [S][T+1][ny] with y[:,0] = the first measurement.
 * Outputs: y[:,1:], u [S][T][nu]; nullable: x [S][T+1][nx] (plant states), xhat, xs [S][T][nx], us [S][T][nu],
 * ell_avg [S][T] (running average stage cost after each step), iters / kkt [S][T] (kind = MPC only). */
int nnmpc_online_run(nnmpc_online_t* h, int kind, int S, int T, double* x_io, double* xhat_io, double* uprev_io,
                     const double* setpoints, const double* disturbances, const double* noise, double* y, double* u,
                     double* x, double* xhat, double* xs, double* us, double* ell_avg, int* iters, double* kkt,
                     double tol, int max_iter, void* stream);

/* ---- self tests (used by tests/) -----------------------------------------------------------------
 * nnmpc_lp_gemm_test: the tcgen05 split-operator GEMM, C[M x N] = fp16(A)[M x K] (T1 + T2)[N x K]^T / s with
 * (T1, T2, s) the two-term fp16 split of the square FP64 operator Bt (N == K, bt_max = max |Bt|);
 * A, Bt, C are dense row-major FP64 device matrices. */
int nnmpc_lp_gemm_test(int M, int N, int K, const double* A, const double* Bt, double bt_max, double* C, int pair,
                       void* stream);   /* pair: 0 = one-CTA kernel with 128 x 128 tiles, 1 = CTA-pair (cta_group::2) kernel, 2 = one-CTA kernel with 256 x 128 tiles */
/* nnmpc_oz_gemm_test: the FP64-accurate GEMM on the INT8 tcgen05 tensor cores (error-free base-128 slicing of both
 * operands, exact INT32 accumulation, 36 INT8 products), C[M x N] = A[M x K] Bt[N x K]^T; dense row-major FP64
 * device matrices, K <= 32768. */
int nnmpc_oz_gemm_test(int M, int N, int K, const double* A, const double* Bt, double* C, void* stream);
/* nnmpc_exact_apply_test: the exact operator applies of the closed-loop engine, called as the engine calls them.
 *   kind 0: anchor  X[r] = Op A[r] - C[r]
 *   kind 1: check   G[r] = Op A[r] + C[r];  kres[r] = max(kres[r], ||A[r] - clip(A[r] - G[r], lb[r, k], ub[r, k])||_inf),
 *                   k = col % nu, and +Inf for a row with a NaN or an infinite G;  G = X, which may be NULL
 *   kind 2: store   X[r] = Op A[r]
 * In every kind r = rows[p] for p < min(*count, max_rows) (rows NULL: r = p), and no other row is touched.  Op is n x n
 * (n even, the INT8 pipe takes n <= 32768); A, C, X are B x n with every listed r < B; lb, ub are B x nu; kres holds B
 * non-negative doubles as bit patterns; count is a device int.  All pointers are device memory.
 * pipe 0 = FP64 DMMA (kind 0: the anchor GEMM of the FP64 path, kind 1: its exact check, kind 2: the plain store),
 * pipe 1 = INT8 digit planes (kind 0: 6 levels, kinds 1 and 2: 8 levels).
 * variant (pipe 1): -1 = the process default (NNMPC_OZ_VARIANT), 0..3 = that kernel variant.  Synchronises the stream. */
int nnmpc_exact_apply_test(int kind, int pipe, int variant, int B, int n, int nu, const double* Op, const int* rows,
                           const int* count, int max_rows, const double* A, const double* C, const double* lb,
                           const double* ub, double* X, unsigned long long* kres, void* stream);
/* nnmpc_lp_step_test: one kernel of the mixed-precision iteration (the fp16 tensor-core pass and the FP64 kernels around
 * it), called as the closed-loop engine calls it, on caller-owned device state; synchronises the stream.
 *   op 0 split        T1 = fp16(s Top), T2 = fp16(s Top - T1), s = 2^(10 - e) for top_max = m 2^e (m in [0.5, 1)):
 *                     D_out / S_out receive T1 / T2 as n rows of ldh = 64 ceil(n / 64) halves, sc_out[0] = s
 *   op 1 anchor_prep  listed rows: W = 2 clip(V) - V, E = 0
 *   op 2 dr_first     listed rows: one FP64 step from X, first increment into D_out at row pos_r[r] (none if < 0)
 *   op 3 reanchor     listed rows in emit_state: X = Z, W = Z + W rinv (rinv per column)
 *   op 4 emit         listed rows in emit_state: first increment from (X, W = w_lp) into D_out at row pos_r[r]
 *   op 5 iterate      one tensor-core pass over operand rows [0, *len_r): reads D_in (and S_in), writes D_out and
 *                     S_out at row pos_w[r] for r = list_r[p] in iter_state, folds max |d| into dres
 *   op 6 correct      X += T2 S_in / (s sS) over the rows op 5 would take part with
 * Listed rows (ops 1-4) are rows[p] for p < *count.  list_r, pos_w, pos_r NULL = identity; need2 (per 128 operand rows)
 * and tile_stat[2] are nullable.  kernel (ops 5, 6): -1 = the process default (NNMPC_LP_KERNEL, NNMPC_LP_TILE,
 * NNMPC_LP1_TILE), else two-term passes (s_mode 0) 0 = 128 x 128 tiles, 1 = 256 x 128 tiles, 2 = CTA pair, one-term
 * passes (s_mode 1, 2) and op 6: 0 = 128 x 128, 1 = 256 x 128.  s_mode (ops 2, 4, 5): 0 = no pending sums (S_out, sS
 * untouched), 1 = add the increment to S_in, 2 = start a new pending sum.  Shapes: X, V, W, Z, D_*, S_* are B x n
 * (fp16 as bit patterns), E is B x n floats, sc_in, sc_out, sS, dres, state, it, dtrig are per row, lb, ub are B x nu,
 * rinv has n entries; count and len_r are device ints.  Refuses n odd or <= 0, nu <= 0, and s_mode != 0 (or op 6) with
 * kernel 2. */
int nnmpc_lp_step_test(int op, int kernel, int s_mode, double alpha, int n, int nu, int B, const double* Top,
                       double top_max, const int* rows, const int* count, const int* list_r, const int* len_r,
                       const int* pos_w, const int* pos_r, int* state, int iter_state, int emit_state,
                       unsigned char* need2, double* X, double* V, double* W, float* E, double* sc_in, double* sc_out,
                       double* sS, unsigned long long* dres, int* it, const double* dtrig, const double* rinv,
                       const double* Z, const double* lb, const double* ub, const unsigned short* D_in,
                       const unsigned short* S_in, unsigned short* D_out, unsigned short* S_out,
                       unsigned long long* tile_stat, void* stream);
/* nnmpc_lp_pass_probe (tools/probes/lp_pass_split.py): one tensor-core pass over B x n synthetic state with the production
 * epilogue (ms[0]), with an epilogue that only drains TMEM (ms[1]) and with the production epilogue but no TMA loads / MMAs
 * (ms[2]: the epilogue alone); then the deferred-second-term form: the one-term pass (ms[3]) and the second-term delivery
 * GEMM (ms[4]); each averaged over reps launches; ms has room for 5 floats. */
int nnmpc_lp_pass_probe(int B, int n, int reps, float* ms);
/* C = A * Bt^T through the FP64 GEMM kernel */
int nnmpc_gemm_tn(int M, int N, int K, const double* A, long long lda, const double* Bt,
                  long long ldb, double* C, long long ldc, const int* rows, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NNMPC_H */
