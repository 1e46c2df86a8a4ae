// Internal interface of the batched target selector (shared by ts.cu and sim.cu).
#pragma once
#include "nnmpc_common.cuh"

struct nnmpc_ts {
  int nx, nu, ny, nd, device;
  int nw = 0;                                        // variables of the QP k_ts_general solves (nu unless reduced)
  int* fail = nullptr;                               // device flag: some solve of the last call missed its optimum
  double *Ht = nullptr, *Fy = nullptr, *Fd = nullptr, *f0 = nullptr, *Gx = nullptr, *Gd = nullptr;   // device operators
  double *ulb = nullptr, *uub = nullptr;
  // k_ts_general (output-constrained or reduced targets): min 1/2 v'Hinv^-1 v + (Fy ysp + Fd d + f0)'v over nw variables
  // s.t. lo0_i - R_i s <= Abar_i v <= hi0_i - R_i s (mb rows, the last nu of them the inputs'), AH = Abar Hinv,
  // Mbar = Abar Hinv Abar'.  Rows i < nR carry the offset R_i s: row i of R (row stride rld) holds rny coefficients on
  // ysp (0 or ny) followed by nd on d.
  //   output bounds (nnmpc_ts_set_output_bounds): v = us, Abar = [C Gx; I], R = C Gd + Cd on the ny output rows only
  //   reduced (nnmpc_ts_create_reduced): [xs; us] = K s + Z v with s = [ysp; d]; the kernel also forms xs and us
  bool general = false, reduced = false;
  int mb = 0, nR = 0, rld = 0, rny = 0;
  double *Hinv = nullptr, *Abar = nullptr, *AH = nullptr, *Mbar = nullptr, *R = nullptr, *lo0 = nullptr, *hi0 = nullptr;
  double *Kx = nullptr, *Ku = nullptr, *Zx = nullptr, *Zu = nullptr;
  nnmpc::DevBuf<double> hysp, hd, hxs, hus;          // staging for the host entry point
  nnmpc::DevBuf<int> hiters;
};

namespace nnmpc {

// Optional fused outputs for the closed-loop generator: when `x` is non-null the kernel also
// forms the regulator inputs x0 = [x-xs; uprev-us], lb = ulb-us, ub = uub-us
// (LinearMPCController.get_control_sequence, linearMPC.py:685-688), the warm-start shift
// dus = us_prev - us, and copies (x, uprev) into the dataset row.
struct TsFused {
  const double* x;        // B x nx   current state
  const double* uprev;    // B x nu
  double* x0;             // B x nxa_ld
  int nxa_ld;
  double* lb;             // B x nu
  double* ub;             // B x nu
  double* us_prev;        // B x nu  (in: previous target, out: this target)
  double* dus;            // B x nu
  double* row_x;          // dataset rows, stride row_stride_x / row_stride_u doubles between samples
  double* row_uprev;
  long long row_stride_x, row_stride_u;
};

// Optional indirection for the closed-loop engine: logical sample b is trajectory slot rows[b]
// (b < *count), at its own time index tcur[slot]; the strided arrays (ysp, d, xs, us, iters and the
// dataset rows of TsFused) are then indexed by chunk[slot]*T + tcur[slot], the per-slot buffers of TsFused
// (x, uprev, x0, lb, ub, us_prev, dus) by slot.
struct TsIndex {
  const int* rows;
  const int* count;
  const int* tcur;
  int T;
  const int* chunk = nullptr;   // optional: slot -> trajectory chunk it currently works on (default: the slot itself)
};

int ts_solve_device(nnmpc_ts* h, int B, const double* ysp, long long ysp_stride, const double* d,
                    long long d_stride, double* xs, long long xs_stride, double* us, long long us_stride,
                    int* iters, long long iters_stride, const TsFused* fused, const TsIndex* index,
                    int* fail_flag, cudaStream_t st);

}  // namespace nnmpc
