// Structured-network layers on the tcgen05 tensor cores (sm_100a): every Dense layer of
// RegulatorLayerWithUprev / WithoutUprev (/root/reference/lib/LinearMPCLayers.py:40-61, :91-112) as one pass of the
// split-operand GEMM of lp_gemm.cuh, within the 1e-5 output tolerance of the north star.
//
// Arithmetic.  Activations a and weights w are each held as a two-term fp16 split (hi + lo, 22 significant bits)
// and the layer forms the three products that matter,
//     a w ~ a_hi w_hi + a_hi w_lo + a_lo w_hi                          (a_lo w_lo ~ 2^-22 |a w| is dropped)
// in one fp32 TMEM accumulator: the A operand is the row [a_hi | a_lo] stacked along K, the operator is read twice
// (LpShape::b_wrap) and its second term only multiplies the first half (LpShape::kb2).  fp16 has a 5-bit exponent,
// so every row carries a power-of-two scale: the row that layer l WRITES is scaled from an upper bound of its
// entries, |h_j| <= max|a| max_j sum_i |W_ij| + max|b| with max|a| the MEASURED maximum of the row it read - at most
// a factor ~||W||_1 loose, which costs exponent range, not mantissa bits.  All scaling, bias, ReLU and the final
// us + f(x,..) - f(xs,..) (+ clip) are FP64 in the epilogue.  Rows 2b / 2b+1 hold the two network passes of sample b,
// so the steady-state identity u = us for x = xs, uprev = us holds bit for bit: identical rows give identical
// accumulators.
#pragma once
#include "lp_gemm.cuh"
#include "lp.cuh"

namespace nnmpc {

using MlpTile = lp::LpTile<128, lp::EPI_WARPS == 16 ? 3 : 4>;

// power of two s with s * bound in [2^13, 2^14)  (fp16 max is 65504); bound = 0 -> 1.  A NaN or infinite bound gives a
// NaN scale: the row it belongs to holds a NaN or an infinity, and every output of it comes back NaN through the
// 1 / s of the epilogues, whatever the tensor cores make of the non-finite operand.
__device__ __forceinline__ double mlp_row_scale(double bound) {
  if (!(bound <= 1.7e308)) return __longlong_as_double(0x7ff8000000000000ll);
  if (!(bound > 0.0)) return 1.0;
  int ex;
  frexp(bound, &ex);
  int sh = 14 - ex;
  sh = sh > 100 ? 100 : (sh < -100 ? -100 : sh);
  return ldexp(1.0, sh);
}

// fmax that keeps a NaN in either operand (fmax drops it, and the row would get a finite scale)
__device__ __forceinline__ double max_keep_nan(double m, double b) { return (m != m || b != b) ? m + b : fmax(m, b); }

__device__ __forceinline__ void mlp_split(double t, __half& hi, __half& lo) {
  hi = __double2half(t);
  lo = __double2half(t - (double)__half2float(hi));
}

// rows 2b and 2b+1 of the first-layer operand: [x/s, (uprev), xs/s, us] and [xs/s, (us), xs/s, us]
// (controller_evaluation.py:863-866 scaling), one warp per sample, as [hi | lo] fp16 with a per-row scale
__global__ void __launch_bounds__(256)
k_mlp_pack_tc(const double* __restrict__ x, const double* __restrict__ uprev, const double* __restrict__ xs,
              const double* __restrict__ us, const double* __restrict__ xscale, __half* __restrict__ A, long long pitch,
              int kp, double* __restrict__ sc, float* __restrict__ amax, long long B, int nx, int nu, int with_uprev) {
  const int lane = threadIdx.x & 31;
  const long long b = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  const int o1 = nx, o2 = nx + (with_uprev ? nu : 0), o3 = o2 + nx, o4 = o3 + nu;
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
    m1 = max_keep_nan(m1, fabs(v1));
    m2 = max_keep_nan(m2, fabs(v2));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    m1 = max_keep_nan(m1, __shfl_xor_sync(0xffffffffu, m1, o));
    m2 = max_keep_nan(m2, __shfl_xor_sync(0xffffffffu, m2, o));
  }
  const double s1 = mlp_row_scale(m1), s2 = mlp_row_scale(m2);
  __half* r1 = A + (2 * b) * pitch;
  __half* r2 = r1 + pitch;
  for (int c = lane; c < kp; c += 32) {
    __half h1 = __float2half(0.f), l1 = h1, h2 = h1, l2 = h1;
    if (c < o4) {
      double v1, v2;
      value(c, v1, v2);
      mlp_split(v1 * s1, h1, l1);
      mlp_split(v2 * s2, h2, l2);
    }
    r1[c] = h1; r1[kp + c] = l1;
    r2[c] = h2; r2[kp + c] = l2;
  }
  if (lane == 0) {
    sc[2 * b] = s1; sc[2 * b + 1] = s2;
    amax[2 * b] = (float)m1 * 1.0000002f; amax[2 * b + 1] = (float)m2 * 1.0000002f;   // rounded up: it feeds a bound
  }
}

// hidden layer: h = relu(acc / (s_row s_w) + bias) -> next operand row [hi | lo] with the scale of its bound
struct EpiMlpHidden {
  struct Params {
    __half* Aout;          // next operand, row pitch `pitch` elements, lo half at +kp_out
    long long pitch;
    int kp_out;
    const double* bias;    // N
    const double* sc_in;   // per row: scale of the operand this pass read
    const float* amax_in;  // per row: max |entry| of that operand (unscaled)
    double* sc_out;        // per row: scale of the operand written here
    float* amax_out;       // per row: max entry written here (atomicMax on the bit pattern; entries are >= 0 or +NaN)
    double inv_sw;         // 1 / weight scale
    double w1norm, bmax;   // max_j sum_i |W_ij|, max_j |b_j|
  };
  Params p;
  int row;
  bool ok;
  double inv_in, s_out;
  float hmax;
  __device__ EpiMlpHidden(const Params& p_, lp::EpiWarpSmem*, int) : p(p_), row(0), ok(false), inv_in(0), s_out(1), hmax(0) {}
  __device__ void begin_tile(int pos0, int M) {
    row = pos0 + (int)(threadIdx.x & 31);
    ok = row < M;
    hmax = 0.f;
    if (ok) {
      inv_in = p.inv_sw / p.sc_in[row];
      s_out = mlp_row_scale((double)p.amax_in[row] * p.w1norm + p.bmax);
    }
  }
  __device__ void chunk(int col0, const uint32_t (&acc)[lp::CW], int N) {
    if (!ok || col0 >= p.kp_out) return;
    __align__(16) __half hi[lp::CW];
    __align__(16) __half lo[lp::CW];
#pragma unroll
    for (int j = 0; j < lp::CW; ++j) {
      const int col = col0 + j;
      double h = 0.0;
      if (col < N) {
        h = (double)__uint_as_float(acc[j]) * inv_in + __ldg(p.bias + col);
        h = relu_keep_nan(h);                                   // keras relu; a NaN goes on to the output
        hmax = row_max_keep_nan(hmax, (float)h * 1.0000002f);
      }
      mlp_split(h * s_out, hi[j], lo[j]);
    }
    __half* dst = p.Aout + (long long)row * p.pitch + col0;
#pragma unroll
    for (int v = 0; v < lp::CW / 8; ++v) {
      reinterpret_cast<uint4*>(dst)[v] = reinterpret_cast<const uint4*>(hi)[v];
      reinterpret_cast<uint4*>(dst + p.kp_out)[v] = reinterpret_cast<const uint4*>(lo)[v];
    }
  }
  __device__ void end_tile() {
    if (!ok) return;
    p.sc_out[row] = s_out;                                      // every column tile writes the same value
    atomicMax(reinterpret_cast<unsigned int*>(p.amax_out + row), __float_as_uint(hmax));
  }
};

// last layer: out[b] = us[b] + (f(row 2b) - f(row 2b+1)), optional clip (controller_evaluation.py:888-892)
struct EpiMlpOut {
  struct Params {
    double* out;           // B x nu
    const double* us;      // B x nu
    const double* ulb;     // nu or null
    const double* uub;
    const double* sc_in;
    double inv_sw;
    int nu;
  };
  Params p;
  int row;
  bool ok;
  double inv_in;
  __device__ EpiMlpOut(const Params& p_, lp::EpiWarpSmem*, int) : p(p_), row(0), ok(false), inv_in(0) {}
  __device__ void begin_tile(int pos0, int M) {
    row = pos0 + (int)(threadIdx.x & 31);
    ok = row < M;
    inv_in = ok ? p.inv_sw / p.sc_in[row] : 0.0;
  }
  __device__ void chunk(int col0, const uint32_t (&acc)[lp::CW], int N) {
    const long long b = row >> 1;
#pragma unroll
    for (int j = 0; j < lp::CW; ++j) {
      const double f = (double)__uint_as_float(acc[j]) * inv_in;
      const double g = __shfl_xor_sync(0xffffffffu, f, 1);     // the partner pass sits in the neighbouring lane
      const int col = col0 + j;
      if (ok && !(row & 1) && col < N) {
        double v = p.us[b * p.nu + col] + (f - g);              // us + (out1 - out2), the reference order (:58-60)
        if (p.ulb) v = clip_keep_nan(v, p.ulb[col], p.uub[col]);
        p.out[b * p.nu + col] = v;
      }
    }
  }
  __device__ void end_tile() {}
};

// weights of one layer as the two-term fp16 operator (out x Kp, K-contiguous) with its scale and the norms the
// activation bound needs
struct MlpTcLayer {
  int in = 0, out = 0, kp = 0;
  double scale = 1.0, w1norm = 0.0, bmax = 0.0;
  DevBuf<__half> T1, T2;
  CUtensorMap tm1, tm2;
};

}  // namespace nnmpc
