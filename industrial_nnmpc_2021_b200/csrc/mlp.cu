// Batched forward of the structured regulator network.
//
// Replaces RegulatorLayerWithUprev.call / RegulatorLayerWithoutUprev.call
// (/root/reference/lib/LinearMPCLayers.py:40-61, :91-112; Keras, float64) and the NumPy
// deployment form NeuralNetworkController._get_control_input
// (/root/reference/lib/controller_evaluation.py:863-892):
//     u = us + f(x, [uprev], xs, us) - f(xs, [us], xs, us),   f = (Dense+ReLU)^(L-1), Dense(no bias)
// Both passes of a sample are interleaved as rows 2b / 2b+1 of one activation matrix, so every
// layer is a single FP64 tensor-core GEMM with bias+ReLU fused into the epilogue, and the last
// layer's epilogue forms us + out(2b) - out(2b+1) (+ clip) with one warp shuffle - the difference
// never goes through memory.
//
// Arithmetic modes (nnmpc_mlp_set_precision):
//   1 (default)  INT8 tcgen05 tensor cores: activations and weights as 4 signed base-128 digit planes, the 10
//                digit-plane products of levels 0..3 accumulated EXACTLY in INT32 (oz_gemm.cuh), bias / ReLU / output
//                assembly in FP64 - ~1e-7 of the float64 Keras layer, no accumulation error;
//   0            FP64 DMMA GEMMs (~1e-13);
//   2            split-fp16 tcgen05 GEMMs with fp32 TMEM accumulation (mlp_tc.cuh) - measured on B200: the fp32
//                accumulation of kind::f16 loses ~2^-22 of the running sum per MMA step (2e-6 rms, 1.4e-5 max per
//                832-wide layer, tools/probes/lp_accum_error.py), which leaves the 1e-5 tolerance in the tails, so
//                this mode is kept for comparison only.
#include "qp.cuh"
#include "mlp_tc.cuh"
#include "oz.cuh"

struct nnmpc_mlp {
  int nx, nu, with_uprev, L, device;
  int dims[17];
  int ld[17];          // even leading dimensions of the activations (ld[i] >= dims[i])
  double* Wt[16];      // device, transposed weights: dims[i+1] x ld[i]
  double* bias[16];    // device, dims[i+1] (null for the last layer)
  int maxw;            // widest hidden activation (ld)
  nnmpc::DevBuf<double> act0, act1;
  nnmpc::DevBuf<double> hx, hup, hxs, hus, hout, hscale, hlb, hub;
  // INT8 tcgen05 mode
  nnmpc::OzOperator ozW[16];        // weight digit planes per layer
  nnmpc::OzRows ozA[16];            // activation digit planes per layer (distinct contraction lengths)
  nnmpc::DevBuf<double> fout;       // last layer: f of both passes, 2 B x nu
  nnmpc::DevBuf<float> hf32;        // hidden activation between a layer's epilogue and the slicing of the next operand
  // training (nnmpc_mlp_train_step): Keras-layout kernels for the backward-data GEMM, Adam moments, caches
  double* Wk[16];                   // in x ldk (ldk = even(out)), kept in step with Wt
  double *mW[16], *vW[16], *mB[16], *vB[16];
  nnmpc::DevBuf<double> tr_act[17]; // activations a_0 .. a_{L-1}: 2B x ld[l]
  nnmpc::DevBuf<double> tr_f, tr_d0, tr_d1, tr_t1, tr_t2, tr_dW, tr_db;
  double* tr_loss;                  // device scalar
  int train_ready, dirty;           // dirty: the inference operators (digit planes, fp16 split) lag behind Wt
  // split-fp16 tcgen05 mode
  int tc_mode;                      // 1: INT8 tcgen05 layers, 2: split-fp16 tcgen05 layers, 0: FP64 DMMA
  nnmpc::MlpTcLayer tcl[16];
  int kp_max;
  long long tc_rows;                // operand rows the buffers / tensor maps below are sized for
  nnmpc::DevBuf<__half> tcA[2];     // ping-pong operands [rows][2 * kp_max]: [hi | lo]
  CUtensorMap tmA[16];              // layer l reads tcA[l & 1] as rows x 2 kp_l
  nnmpc::DevBuf<double> tcsc[2];    // per-row scales
  nnmpc::DevBuf<float> tcamax[2];   // per-row max |entry|
};

namespace nnmpc {

// rows 2b and 2b+1 of the first-layer input: [x/s, (uprev), xs/s, us] and [xs/s, (us), xs/s, us]
__global__ void k_pack_inputs(const double* __restrict__ x, const double* __restrict__ uprev,
                              const double* __restrict__ xs, const double* __restrict__ us,
                              const double* __restrict__ xscale, double* __restrict__ in, long long B, int nx,
                              int nu, int with_uprev, int ld) {
  const long long total = B * ld;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const int o1 = nx, o2 = nx + (with_uprev ? nu : 0), o3 = o2 + nx, o4 = o3 + nu;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const long long b = i / ld;
    const int c = (int)(i - b * ld);
    double v1, v2;
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
    } else if (c < o4) {
      v1 = us[b * nu + (c - o3)];
      v2 = v1;
    } else {
      v1 = v2 = 0.0;
    }
    in[(2 * b) * ld + c] = v1;
    in[(2 * b + 1) * ld + c] = v2;
  }
}

// last layer: out[b] = us[b] + acc(row 2b) - acc(row 2b+1), optional clip to [ulb, uub].
// Fragment rows g and g^1 sit in lanes 4 apart, tiles start at multiples of 8 rows, so a pair
// never straddles a fragment; every lane calls apply (ok flags predicate the store).
struct EpiStructOut {
  struct Params {
    double* out;        // B x nu
    const double* us;   // B x nu
    const double* ulb;  // nu or null
    const double* uub;
    int nu;
  };
  Params p;
  __device__ EpiStructOut(const Params& p_, int, int) : p(p_) {}
  __device__ void begin_row() {}
  __device__ void apply(int pr, int, int col, double a0, double a1, bool ok0, bool ok1) {
    const double b0 = __shfl_xor_sync(0xffffffffu, a0, 4);
    const double b1 = __shfl_xor_sync(0xffffffffu, a1, 4);
    if ((pr & 1) || !ok0) return;
    const long long b = pr >> 1;
    double v0 = p.us[b * p.nu + col] + (a0 - b0);   // us + (out1 - out2), the reference order (:58-60)
    if (p.ulb) v0 = clip_keep_nan(v0, p.ulb[col], p.uub[col]);
    p.out[b * p.nu + col] = v0;
    if (ok1) {
      double v1 = p.us[b * p.nu + col + 1] + (a1 - b1);
      if (p.ulb) v1 = clip_keep_nan(v1, p.ulb[col + 1], p.uub[col + 1]);
      p.out[b * p.nu + col + 1] = v1;
    }
  }
  __device__ void finish_row(int, int, int, bool) {}
};

static int mlp_forward_device(nnmpc_mlp* h, long long B, const double* x, const double* uprev, const double* xs,
                              const double* us, const double* xscale, const double* ulb, const double* uub,
                              double* out, cudaStream_t st) {
  if (B <= 0) return 0;
  // chunk the batch so the two activation buffers stay below ~2 GiB each
  long long chunk = (long long)(1ll << 28) / (2ll * h->maxw);
  chunk = chunk < 1024 ? 1024 : (chunk > (1 << 20) ? (1 << 20) : chunk);
  if (chunk > B) chunk = B;
  NNMPC_TRY(h->act0.ensure((size_t)2 * chunk * h->maxw));
  NNMPC_TRY(h->act1.ensure((size_t)2 * chunk * h->maxw));
  const int nx = h->nx, nu = h->nu, L = h->L;
  for (long long b0 = 0; b0 < B; b0 += chunk) {
    const long long nb = B - b0 < chunk ? B - b0 : chunk;
    k_pack_inputs<<<148 * 16, 256, 0, st>>>(x + b0 * nx, uprev ? uprev + b0 * nu : nullptr, xs + b0 * nx,
                                            us + b0 * nu, xscale, h->act0.p, nb, nx, nu, h->with_uprev, h->ld[0]);
    count_launch();
    double* cur = h->act0.p;
    double* nxt = h->act1.p;
    for (int l = 0; l < L; ++l) {
      GemmOperands g{cur, h->ld[l], h->Wt[l], h->ld[l], (int)(2 * nb), h->dims[l + 1], h->ld[l], nullptr, nullptr};
      if (l < L - 1) {
        // zero the padding column of an odd-width hidden layer once per chunk (it is read as K)
        if (h->ld[l + 1] != h->dims[l + 1])
          NNMPC_CUDA(cudaMemsetAsync(nxt, 0, (size_t)2 * nb * h->ld[l + 1] * 8, st));
        NNMPC_TRY(gemm_auto<EpiStore>(g, EpiStore::Params{nxt, h->ld[l + 1], h->bias[l], 1}, st));
        double* t = cur; cur = nxt; nxt = t;
      } else {
        EpiStructOut::Params ep{out + b0 * nu, us + b0 * nu, ulb, uub, nu};
        NNMPC_TRY(gemm_auto<EpiStructOut>(g, ep, st));
      }
    }
  }
  NNMPC_CUDA(cudaGetLastError());
  return 0;
}

// out[b] = us[b] + (f[2b] - f[2b+1]), optional clip (LinearMPCLayers.py:58-60, controller_evaluation.py:888-892)
__global__ void k_struct_out(const double* __restrict__ f, const double* __restrict__ us, const double* __restrict__ ulb,
                             const double* __restrict__ uub, double* __restrict__ out, long long B, int nu) {
  const long long total = B * nu;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / nu;
    const int c = (int)(i - b * nu);
    double v = us[i] + (f[(2 * b) * nu + c] - f[(2 * b + 1) * nu + c]);
    if (ulb) v = clip_keep_nan(v, ulb[c], uub[c]);
    out[i] = v;
  }
}

// INT8 tensor-core forward: the first-layer operand is cut into digit planes straight from the inputs, every hidden
// layer's epilogue writes relu(. + bias) as fp32 with the exact row maximum and one slicing pass cuts the planes the next
// layer reads, the last layer hands f of both passes to the output assembly.  No FP64 activations in memory.
static int mlp_forward_i8(nnmpc_mlp* h, long long B, const double* x, const double* uprev, const double* xs,
                          const double* us, const double* xscale, const double* ulb, const double* uub, double* out,
                          cudaStream_t st) {
  if (B <= 0) return 0;
  const int nx = h->nx, nu = h->nu, L = h->L;
  long long chunk = (long long)(1ll << 28) / (2ll * h->maxw);
  chunk = chunk < 1024 ? 1024 : (chunk > (1 << 18) ? (1 << 18) : chunk);
  if (chunk > B) chunk = B;
  for (int l = 0; l < L; ++l) NNMPC_TRY(oz_rows_ensure(&h->ozA[l], 2 * chunk, h->dims[l], st, 4));
  NNMPC_TRY(h->fout.ensure((size_t)2 * chunk * nu));
  for (int b = 0; b < 2; ++b) NNMPC_TRY(h->tcamax[b].ensure((size_t)2 * chunk));
  const long long ldh = ((long long)h->maxw + 63) / 64 * 64;      // fp32 scratch of one hidden activation
  NNMPC_TRY(h->hf32.ensure((size_t)2 * chunk * ldh));
  for (long long b0 = 0; b0 < B; b0 += chunk) {
    const long long nb = B - b0 < chunk ? B - b0 : chunk;
    const int M = (int)(2 * nb);
    NNMPC_TRY(oz_pack_network_input(&h->ozA[0], nb, x + b0 * nx, uprev ? uprev + b0 * nu : nullptr, xs + b0 * nx, us + b0 * nu,
                                    xscale, nx, nu, h->with_uprev, h->tcamax[0].p, st));
    for (int l = 0; l < L; ++l) {
      const bool last = l == L - 1;
      if (!last) NNMPC_CUDA(cudaMemsetAsync(h->tcamax[1].p, 0, (size_t)M * sizeof(float), st));
      NNMPC_TRY(oz_dense_planes(&h->ozW[l], &h->ozA[l], M, last ? nullptr : h->bias[l], last ? nullptr : &h->ozA[l + 1],
                                h->hf32.p, ldh, h->tcamax[1].p, last ? h->fout.p : nullptr, nu, h->device, st));
    }
    k_struct_out<<<148 * 4, 256, 0, st>>>(h->fout.p, us + b0 * nu, ulb, uub, out + b0 * nu, nb, nu);
    count_launch();
  }
  NNMPC_CUDA(cudaGetLastError());
  return 0;
}

// (out x ld) FP64 transposed weights -> two fp16 terms (rows padded with zeros, kp columns)
__global__ void k_split_weights(const double* __restrict__ Wt, int rows, int cols, int ld, int kp, double s,
                                __half* __restrict__ T1, __half* __restrict__ T2) {
  const long long total = (long long)rows * kp;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const long long r = i / kp;
    const int c = (int)(i - r * kp);
    const double t = c < cols ? Wt[r * ld + c] * s : 0.0;
    __half h1, h2;
    mlp_split(t, h1, h2);
    T1[i] = h1;
    T2[i] = h2;
  }
}

static int mlp_tc_ensure(nnmpc_mlp* h, long long rows, cudaStream_t st) {
  if (rows <= h->tc_rows) return 0;
  const long long rows_pad = (rows + 2 * lp::BM - 1) / (2 * lp::BM) * (2 * lp::BM);
  const long long pitch = 2ll * h->kp_max;
  for (int b = 0; b < 2; ++b) {
    NNMPC_TRY(h->tcA[b].ensure((size_t)rows_pad * pitch));
    NNMPC_CUDA(cudaMemsetAsync(h->tcA[b].p, 0, (size_t)rows_pad * pitch * sizeof(__half), st));
    NNMPC_TRY(h->tcsc[b].ensure((size_t)rows_pad));
    NNMPC_TRY(h->tcamax[b].ensure((size_t)rows_pad));
  }
  for (int l = 0; l < h->L; ++l)
    if (!lp::make_tmap_f16(&h->tmA[l], h->tcA[l & 1].p, rows_pad, 2ll * h->tcl[l].kp, pitch, lp::BM))
      return set_error(NNMPC_ERR_CUDA, "cuTensorMapEncodeTiled failed for the structured-network operands");
  h->tc_rows = rows_pad;
  return 0;
}

static int mlp_forward_tc(nnmpc_mlp* h, long long B, const double* x, const double* uprev, const double* xs,
                          const double* us, const double* xscale, const double* ulb, const double* uub, double* out,
                          cudaStream_t st) {
  if (B <= 0) return 0;
  const int nx = h->nx, nu = h->nu, L = h->L;
  long long chunk = B < 131072 ? B : 131072;            // samples per pass: 2 x chunk operand rows
  NNMPC_TRY(mlp_tc_ensure(h, 2 * chunk, st));
  const long long pitch = 2ll * h->kp_max;
  const int sms = device_sm_count(h->device);
  for (long long b0 = 0; b0 < B; b0 += chunk) {
    const long long nb = B - b0 < chunk ? B - b0 : chunk;
    const int M = (int)(2 * nb);
    k_mlp_pack_tc<<<(unsigned)((nb + 7) / 8), 256, 0, st>>>(x + b0 * nx, uprev ? uprev + b0 * nu : nullptr, xs + b0 * nx,
                                                           us + b0 * nu, xscale, h->tcA[0].p, pitch, h->tcl[0].kp,
                                                           h->tcsc[0].p, h->tcamax[0].p, nb, nx, nu, h->with_uprev);
    count_launch();
    for (int l = 0; l < L; ++l) {
      const MlpTcLayer& W = h->tcl[l];
      const int in = l & 1, on = in ^ 1;
      lp::LpShape g{M, W.out, 2 * W.kp, nullptr, 0, nullptr, nullptr, W.kp / lp::BK, W.kp / lp::BK};
      cudaError_t e;
      if (l < L - 1) {
        NNMPC_CUDA(cudaMemsetAsync(h->tcamax[on].p, 0, (size_t)M * sizeof(float), st));
        EpiMlpHidden::Params ep{h->tcA[on].p, pitch, h->tcl[l + 1].kp, h->bias[l], h->tcsc[in].p, h->tcamax[in].p,
                                h->tcsc[on].p, h->tcamax[on].p, 1.0 / W.scale, W.w1norm, W.bmax};
        e = lp::launch_lp_gemm<MlpTile, EpiMlpHidden>(h->tmA[l], W.tm1, W.tm2, g, ep, sms, st);
      } else {
        EpiMlpOut::Params ep{out + b0 * nu, us + b0 * nu, ulb, uub, h->tcsc[in].p, 1.0 / W.scale, nu};
        e = lp::launch_lp_gemm<MlpTile, EpiMlpOut>(h->tmA[l], W.tm1, W.tm2, g, ep, sms, st);
      }
      count_launch();
      if (e != cudaSuccess) return set_error(NNMPC_ERR_CUDA, "structured-network tcgen05 launch failed: %s", cudaGetErrorString(e));
    }
  }
  NNMPC_CUDA(cudaGetLastError());
  return 0;
}

// ---- training step: MSE + Adam on the structured network (cdu_train.py:24-62, cstrs_train.py:24-61) -----------------
// Keras compiles the model with optimizer='adam', loss='mean_squared_error' and fits u = us + f(x,..) - f(xs,..)
// to the MPC inputs.  One step here = forward in FP64 with every activation kept, loss, backward through both
// network passes (rows 2b / 2b+1 carry +/- the output gradient), Adam on every kernel and bias.  All contractions are
// the FP64 tensor-core GEMM of gemm_f64.cuh (C = A Bt^T, both operands K-contiguous):
//     forward      a_{l+1} = relu(a_l Wt_l^T + b_l)                     A = a_l (2B x in),        Bt = Wt_l (out x in)
//     backward     delta_l = (delta_{l+1} Wk_l^T) . [a_l > 0]           A = delta_{l+1} (2B x out), Bt = Wk_l (in x out)
//     gradient     dWt_l   = delta_{l+1}^T a_l                          A = delta_{l+1}^T (out x 2B), Bt = a_l^T (in x 2B)
struct EpiMaskStore {      // C = acc * [mask > 0]
  struct Params {
    double* C;
    long long ldc;
    const double* mask;
    long long ldm;
  };
  Params p;
  __device__ EpiMaskStore(const Params& p_, int, int) : p(p_) {}
  __device__ void begin_row() {}
  __device__ void apply(int pr, int, int col, double v0, double v1, bool ok0, bool ok1) {
    if (ok0) p.C[(long long)pr * p.ldc + col] = p.mask[(long long)pr * p.ldm + col] > 0.0 ? v0 : 0.0;
    if (ok1) p.C[(long long)pr * p.ldc + col + 1] = p.mask[(long long)pr * p.ldm + col + 1] > 0.0 ? v1 : 0.0;
  }
  __device__ void finish_row(int, int, int, bool) {}
};

// dst (C x ldd) = src (R x lds, first C columns)^T
__global__ void k_transpose(const double* __restrict__ src, long long lds, int R, int C, double* __restrict__ dst, long long ldd) {
  __shared__ double tile[32][33];
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < R && c < C) ? src[(long long)r * lds + c] : 0.0;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < C && r < R) dst[(long long)c * ldd + r] = tile[threadIdx.x][i];
  }
}

// out = us + f(2b) - f(2b+1); loss += sum (out - u)^2 / (B nu); delta rows 2b / 2b+1 = +/- 2 (out - u) / (B nu)
__global__ void __launch_bounds__(256)
k_train_out(const double* __restrict__ f, long long ldf, const double* __restrict__ us, const double* __restrict__ u,
            double* __restrict__ delta, long long ldd, double* __restrict__ loss, long long B, int nu) {
  __shared__ double red[8];
  const double scale = 1.0 / ((double)B * (double)nu);
  double acc = 0.0;
  const long long total = B * ldd;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / ldd;
    const int c = (int)(i - b * ldd);
    double g = 0.0;
    if (c < nu) {
      const double e = us[b * nu + c] + (f[(2 * b) * ldf + c] - f[(2 * b + 1) * ldf + c]) - u[b * nu + c];
      acc += e * e;
      g = 2.0 * e * scale;
    }
    delta[(2 * b) * ldd + c] = g;
    delta[(2 * b + 1) * ldd + c] = -g;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += red[w];
    atomicAdd(loss, t * scale);
  }
}

// row sums of an (R x K) matrix: db_o = sum over the batch of delta^T[o][.]
__global__ void k_rowsum(const double* __restrict__ src, long long lds, int R, int K, double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  for (int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < R; r += gridDim.x * (blockDim.x >> 5)) {
    double a = 0.0;
    for (int k = lane; k < K; k += 32) a += src[(long long)r * lds + k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) out[r] = a;
  }
}

// Adam as Keras applies it (optimizer_v2/adam.py, non-amsgrad): lr_t = lr sqrt(1 - b2^t) / (1 - b1^t),
// m = b1 m + (1 - b1) g, v = b2 v + (1 - b2) g^2, w -= lr_t m / (sqrt(v) + eps).  W2 (nullable) is the second layout of
// the same kernel: element (r, c) of W (R x ldw) lives at W2[c * ld2 + r].
__global__ void k_adam(double* __restrict__ W, long long ldw, int R, int C, double* __restrict__ W2, long long ld2,
                       double* __restrict__ m, double* __restrict__ v, const double* __restrict__ g, long long ldg,
                       double lr_t, double b1, double b2, double eps) {
  const long long total = (long long)R * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / C;
    const int c = (int)(i - r * C);
    const double gr = g[r * ldg + c];
    const double mn = b1 * m[i] + (1.0 - b1) * gr;
    const double vn = b2 * v[i] + (1.0 - b2) * gr * gr;
    m[i] = mn;
    v[i] = vn;
    const double w = W[r * ldw + c] - lr_t * mn / (sqrt(vn) + eps);
    W[r * ldw + c] = w;
    if (W2) W2[(long long)c * ld2 + r] = w;
  }
}

static int mlp_train_ensure(nnmpc_mlp* h, long long B) {
  const int L = h->L;
  if (!h->train_ready) {
    for (int l = 0; l < L; ++l) {
      const int in = h->dims[l], outw = h->dims[l + 1], ld = h->ld[l], ldk = (outw + 1) & ~1;
      NNMPC_CUDA(cudaMalloc((void**)&h->Wk[l], (size_t)in * ldk * sizeof(double)));
      NNMPC_CUDA(cudaMemset(h->Wk[l], 0, (size_t)in * ldk * sizeof(double)));
      dim3 grid((in + 31) / 32, (outw + 31) / 32), blk(32, 8);
      k_transpose<<<grid, blk>>>(h->Wt[l], ld, outw, in, h->Wk[l], ldk);
      count_launch();
      for (double** q : {&h->mW[l], &h->vW[l]}) {
        NNMPC_CUDA(cudaMalloc((void**)q, (size_t)outw * in * sizeof(double)));
        NNMPC_CUDA(cudaMemset(*q, 0, (size_t)outw * in * sizeof(double)));
      }
      if (l < L - 1)
        for (double** q : {&h->mB[l], &h->vB[l]}) {
          NNMPC_CUDA(cudaMalloc((void**)q, (size_t)outw * sizeof(double)));
          NNMPC_CUDA(cudaMemset(*q, 0, (size_t)outw * sizeof(double)));
        }
    }
    NNMPC_CUDA(cudaMalloc((void**)&h->tr_loss, sizeof(double)));
    h->train_ready = 1;
  }
  const size_t rows = (size_t)2 * B;
  size_t wmax = 0, gmax = 0;
  for (int l = 0; l < L; ++l) {
    NNMPC_TRY(h->tr_act[l].ensure(rows * h->ld[l]));
    const size_t w = (size_t)((h->dims[l + 1] + 1) & ~1);
    if (w > wmax) wmax = w;
    if ((size_t)h->ld[l] > wmax) wmax = h->ld[l];
    const size_t gsz = (size_t)h->dims[l + 1] * h->ld[l];
    if (gsz > gmax) gmax = gsz;
  }
  NNMPC_TRY(h->tr_f.ensure(rows * ((h->nu + 1) & ~1)));
  NNMPC_TRY(h->tr_d0.ensure(rows * wmax));
  NNMPC_TRY(h->tr_d1.ensure(rows * wmax));
  NNMPC_TRY(h->tr_t1.ensure(rows * wmax));
  NNMPC_TRY(h->tr_t2.ensure(rows * wmax));
  NNMPC_TRY(h->tr_dW.ensure(gmax));
  NNMPC_TRY(h->tr_db.ensure(wmax));
  return 0;
}

// forward in FP64 keeping the activations; returns f (2B x ldf) in h->tr_f
static int mlp_train_forward(nnmpc_mlp* h, long long B, const double* x, const double* uprev, const double* xs,
                             const double* us, cudaStream_t st) {
  const int L = h->L, nx = h->nx, nu = h->nu;
  k_pack_inputs<<<148 * 8, 256, 0, st>>>(x, uprev, xs, us, nullptr, h->tr_act[0].p, B, nx, nu, h->with_uprev, h->ld[0]);
  count_launch();
  for (int l = 0; l < L; ++l) {
    GemmOperands g{h->tr_act[l].p, h->ld[l], h->Wt[l], h->ld[l], (int)(2 * B), h->dims[l + 1], h->ld[l], nullptr, nullptr};
    if (l < L - 1) {
      if (h->ld[l + 1] != h->dims[l + 1])
        NNMPC_CUDA(cudaMemsetAsync(h->tr_act[l + 1].p, 0, (size_t)2 * B * h->ld[l + 1] * sizeof(double), st));
      NNMPC_TRY(gemm_auto<EpiStore>(g, EpiStore::Params{h->tr_act[l + 1].p, h->ld[l + 1], h->bias[l], 1}, st));
    } else {
      const int ldf = (nu + 1) & ~1;
      if (ldf != nu) NNMPC_CUDA(cudaMemsetAsync(h->tr_f.p, 0, (size_t)2 * B * ldf * sizeof(double), st));
      NNMPC_TRY(gemm_auto<EpiStore>(g, EpiStore::Params{h->tr_f.p, ldf, nullptr, 0}, st));
    }
  }
  return 0;
}

// device-pointer forward in the handle's arithmetic mode, for other translation units (online.cu)
static int mlp_refresh(nnmpc_mlp* h);
int mlp_forward_dispatch(nnmpc_mlp* h, long long B, const double* x, const double* uprev, const double* xs,
                         const double* us, const double* xscale, const double* ulb, const double* uub, double* out,
                         cudaStream_t st) {
  if (h->dirty) NNMPC_TRY(mlp_refresh(h));
  return (h->tc_mode == 1 ? mlp_forward_i8 : h->tc_mode == 2 ? mlp_forward_tc : mlp_forward_device)(
      h, B, x, uprev, xs, us, xscale, ulb, uub, out, st);
}
// (Re)build everything derived from one layer's weights: device copies of the transposed kernel (out x ld) and the
// bias, the INT8 digit planes, the two-term fp16 split with its tensor maps, and the norms the fp16 path bounds its
// activations with.  Called by create and, after training steps, before the next forward.
int mlp_install_layer(nnmpc_mlp* h, int l, const double* Wt_host, const double* bias_host) {
  const int in = h->dims[l], outw = h->dims[l + 1], ld = h->ld[l];
  double wmax = 0.0, w1 = 0.0;
  for (int o = 0; o < outw; ++o) {
    double a = 0.0;
    for (int i = 0; i < in; ++i) {
      const double w = fabs(Wt_host[(size_t)o * ld + i]);
      a += w;
      if (w > wmax) wmax = w;
    }
    if (a > w1) w1 = a;
  }
  if (!h->Wt[l]) NNMPC_CUDA(cudaMalloc((void**)&h->Wt[l], (size_t)outw * ld * sizeof(double)));
  NNMPC_CUDA(cudaMemcpy(h->Wt[l], Wt_host, (size_t)outw * ld * sizeof(double), cudaMemcpyHostToDevice));
  NNMPC_TRY(oz_slice_operator(h->Wt[l], outw, in, &h->ozW[l], 0, ld));       // INT8 digit planes of the weights
  MlpTcLayer& T = h->tcl[l];
  T.in = in; T.out = outw; T.kp = (in + lp::BK - 1) / lp::BK * lp::BK;
  if (T.kp > h->kp_max) h->kp_max = T.kp;
  T.w1norm = w1 * 1.0000001;
  T.bmax = 0.0;
  if (bias_host) {
    for (int o = 0; o < outw; ++o) T.bmax = fmax(T.bmax, fabs(bias_host[o]));
    if (!h->bias[l]) NNMPC_CUDA(cudaMalloc((void**)&h->bias[l], (size_t)outw * sizeof(double)));
    NNMPC_CUDA(cudaMemcpy(h->bias[l], bias_host, (size_t)outw * sizeof(double), cudaMemcpyHostToDevice));
  }
  // two-term fp16 operator: scale = the power of two that puts max |s W| in [512, 1024)
  int ex = 0;
  frexp(wmax > 0.0 ? wmax : 1.0, &ex);
  T.scale = ldexp(1.0, 10 - ex);
  const long long rows_pad = ((long long)outw + lp::BN2 - 1) / lp::BN2 * lp::BN2;
  NNMPC_TRY(T.T1.ensure((size_t)rows_pad * T.kp));
  NNMPC_TRY(T.T2.ensure((size_t)rows_pad * T.kp));
  NNMPC_CUDA(cudaMemset(T.T1.p, 0, (size_t)rows_pad * T.kp * sizeof(__half)));
  NNMPC_CUDA(cudaMemset(T.T2.p, 0, (size_t)rows_pad * T.kp * sizeof(__half)));
  k_split_weights<<<148 * 4, 256>>>(h->Wt[l], outw, in, ld, T.kp, T.scale, T.T1.p, T.T2.p);
  count_launch();
  NNMPC_CUDA(cudaDeviceSynchronize());
  if (!lp::make_tmap_f16(&T.tm1, T.T1.p, rows_pad, T.kp, T.kp, MlpTile::BN) ||
      !lp::make_tmap_f16(&T.tm2, T.T2.p, rows_pad, T.kp, T.kp, MlpTile::BN))
    return set_error(NNMPC_ERR_CUDA, "cuTensorMapEncodeTiled failed for the structured-network weights");
  return 0;
}

// after training steps: rebuild the inference operators (digit planes, fp16 split, norms) from the trained kernels
static int mlp_refresh(nnmpc_mlp* h) {
  NNMPC_CUDA(cudaDeviceSynchronize());
  for (int l = 0; l < h->L; ++l) {
    const int outw = h->dims[l + 1], ld = h->ld[l];
    double* w = new (std::nothrow) double[(size_t)outw * ld];
    double* b = (l < h->L - 1) ? new (std::nothrow) double[(size_t)outw] : nullptr;
    int rc = (!w || (l < h->L - 1 && !b)) ? set_error(NNMPC_ERR_NOMEM, "out of host memory") : 0;
    if (rc == 0 && cudaMemcpy(w, h->Wt[l], (size_t)outw * ld * sizeof(double), cudaMemcpyDeviceToHost) != cudaSuccess)
      rc = set_error(NNMPC_ERR_CUDA, "weight download failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (rc == 0 && b && cudaMemcpy(b, h->bias[l], (size_t)outw * sizeof(double), cudaMemcpyDeviceToHost) != cudaSuccess)
      rc = set_error(NNMPC_ERR_CUDA, "bias download failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (rc == 0) rc = mlp_install_layer(h, l, w, b);
    delete[] w;
    delete[] b;
    if (rc < 0) return rc;
  }
  h->dirty = 0;
  return 0;
}

int mlp_dims(const nnmpc_mlp* h, int* nx, int* nu, int* with_uprev) {
  *nx = h->nx; *nu = h->nu; *with_uprev = h->with_uprev;
  return h->device;
}

}  // namespace nnmpc

using namespace nnmpc;

extern "C" {

int nnmpc_mlp_create(nnmpc_mlp_t** out, int nx, int nu, int with_uprev, int num_layers, const int* dims,
                     const double* const* weights_host, const double* const* biases_host, int device) {
  if (!out || !dims || !weights_host) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_create: null argument");
  if (num_layers < 1 || num_layers > 16) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_create: 1..16 layers");
  const int in_w = 2 * nx + (with_uprev ? 2 : 1) * nu;
  if (dims[0] != in_w) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_create: dims[0]=%d, expected %d", dims[0], in_w);
  if (dims[num_layers] != nu) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_create: last width must equal nu");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return set_error(NNMPC_ERR_CUDA, "nnmpc_mlp_create: no CUDA device (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_create: bad device %d", device);
  DeviceGuard dg(device);
  nnmpc_mlp* h = new (std::nothrow) nnmpc_mlp();
  if (!h) return set_error(NNMPC_ERR_NOMEM, "out of host memory");
  h->nx = nx; h->nu = nu; h->with_uprev = with_uprev; h->L = num_layers; h->device = device;
  h->maxw = 0;
  for (int i = 0; i <= num_layers; ++i) {
    if (dims[i] < 1) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_create: bad width");
    h->dims[i] = dims[i];
    h->ld[i] = (dims[i] + 1) & ~1;
    if (i < num_layers && h->ld[i] > h->maxw) h->maxw = h->ld[i];
  }
  h->tc_mode = 1;
  h->tc_rows = 0;
  h->kp_max = 0;
  for (int l = 0; l < 16; ++l) h->Wt[l] = h->bias[l] = h->Wk[l] = h->mW[l] = h->vW[l] = h->mB[l] = h->vB[l] = nullptr;
  h->tr_loss = nullptr;
  h->train_ready = h->dirty = 0;
  int rc = 0;
  for (int l = 0; l < num_layers && rc == 0; ++l) {
    const int in = dims[l], outw = dims[l + 1], ld = h->ld[l];
    double* tmp = new (std::nothrow) double[(size_t)outw * ld];
    if (!tmp) { rc = set_error(NNMPC_ERR_NOMEM, "out of host memory"); break; }
    const double* W = weights_host[l];  // in x out, row-major (Keras kernel layout)
    for (int o = 0; o < outw; ++o) {
      for (int i = 0; i < in; ++i) tmp[(size_t)o * ld + i] = W[(size_t)i * outw + o];
      for (int i = in; i < ld; ++i) tmp[(size_t)o * ld + i] = 0.0;
    }
    if (l < num_layers - 1 && (!biases_host || !biases_host[l]))
      rc = set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_create: missing bias %d", l);
    else
      rc = mlp_install_layer(h, l, tmp, l < num_layers - 1 ? biases_host[l] : nullptr);
    delete[] tmp;
  }
  if (rc < 0) {          // a half-built handle is released, not leaked
    nnmpc_mlp_destroy(h);
    return rc;
  }
  *out = h;
  return 0;
}

int nnmpc_mlp_set_precision(nnmpc_mlp_t* h, int mode) {
  if (!h) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_set_precision: null handle");
  if (mode < 0 || mode > 2)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_set_precision: mode must be 0 (FP64 DMMA), 1 (INT8 tcgen05) or 2 (split-fp16 tcgen05)");
  h->tc_mode = mode;
  return 0;
}

int nnmpc_mlp_destroy(nnmpc_mlp_t* h) {
  if (!h) return 0;
  DeviceGuard dg(h->device);
  for (int l = 0; l < h->L; ++l) {
    if (h->Wt[l]) cudaFree(h->Wt[l]);
    if (h->bias[l]) cudaFree(h->bias[l]);
    h->tcl[l].T1.release();
    h->tcl[l].T2.release();
    h->ozW[l].release();
    h->ozA[l].release();
    for (double* q : {h->Wk[l], h->mW[l], h->vW[l], h->mB[l], h->vB[l]})
      if (q) cudaFree(q);
    h->tr_act[l].release();
  }
  if (h->tr_loss) cudaFree(h->tr_loss);
  for (nnmpc::DevBuf<double>* q : {&h->tr_f, &h->tr_d0, &h->tr_d1, &h->tr_t1, &h->tr_t2, &h->tr_dW, &h->tr_db}) q->release();
  h->fout.release();
  h->hf32.release();
  for (int b = 0; b < 2; ++b) { h->tcA[b].release(); h->tcsc[b].release(); h->tcamax[b].release(); }
  h->act0.release(); h->act1.release();
  h->hx.release(); h->hup.release(); h->hxs.release(); h->hus.release(); h->hout.release();
  h->hscale.release(); h->hlb.release(); h->hub.release();
  delete h;
  return 0;
}

int nnmpc_mlp_train_step(nnmpc_mlp_t* h, long long B, const double* x, const double* uprev, const double* xs,
                         const double* us, const double* u_target, double lr, double beta1, double beta2, double eps,
                         long long step, int apply, double* loss_host, void* stream) {
  if (!h || !x || !xs || !us || !u_target) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_train_step: null argument");
  if (h->with_uprev && !uprev) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_train_step: uprev required");
  if (B <= 0 || B > (1ll << 18) || step < 1)
    return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_train_step: batch size must be in 1..262144 and step >= 1");
  DeviceGuard dg(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  NNMPC_TRY(mlp_train_ensure(h, B));
  const int L = h->L, nu = h->nu, M2 = (int)(2 * B);
  NNMPC_TRY(mlp_train_forward(h, B, x, uprev, xs, us, st));
  const int ldf = (nu + 1) & ~1;
  double* dcur = h->tr_d0.p;          // delta_{l+1}: 2B x even(dims[l+1])
  double* dnxt = h->tr_d1.p;
  NNMPC_CUDA(cudaMemsetAsync(h->tr_loss, 0, sizeof(double), st));
  k_train_out<<<148 * 2, 256, 0, st>>>(h->tr_f.p, ldf, us, u_target, dcur, ldf, h->tr_loss, B, nu);
  count_launch();
  if (apply) {
    const double lr_t = lr * sqrt(1.0 - pow(beta2, (double)step)) / (1.0 - pow(beta1, (double)step));
    for (int l = L - 1; l >= 0; --l) {
      const int in = h->dims[l], outw = h->dims[l + 1], ld = h->ld[l], ldo = (outw + 1) & ~1, ldk = ldo;
      // delta_{l+1}^T (out x 2B) and a_l^T (ld x 2B)
      dim3 blk(32, 8);
      k_transpose<<<dim3((outw + 31) / 32, (M2 + 31) / 32), blk, 0, st>>>(dcur, ldo, M2, outw, h->tr_t1.p, M2);
      k_transpose<<<dim3((ld + 31) / 32, (M2 + 31) / 32), blk, 0, st>>>(h->tr_act[l].p, ld, M2, ld, h->tr_t2.p, M2);
      count_launch(2);
      GemmOperands gw{h->tr_t1.p, M2, h->tr_t2.p, M2, outw, ld, M2, nullptr, nullptr};
      NNMPC_TRY(gemm_auto<EpiStore>(gw, EpiStore::Params{h->tr_dW.p, ld, nullptr, 0}, st));
      if (l < L - 1) {
        k_rowsum<<<(outw + 7) / 8, 256, 0, st>>>(h->tr_t1.p, M2, outw, M2, h->tr_db.p);
        count_launch();
      }
      if (l > 0) {   // delta_l = (delta_{l+1} Wk_l^T) . [a_l > 0]   (uses the kernel BEFORE this step's update)
        GemmOperands gd{dcur, ldo, h->Wk[l], ldk, M2, in, ldk, nullptr, nullptr};
        if (ld != in) NNMPC_CUDA(cudaMemsetAsync(dnxt, 0, (size_t)M2 * ld * sizeof(double), st));
        NNMPC_TRY(gemm_auto<EpiMaskStore>(gd, EpiMaskStore::Params{dnxt, ld, h->tr_act[l].p, ld}, st));
      }
      k_adam<<<148 * 4, 256, 0, st>>>(h->Wt[l], ld, outw, in, h->Wk[l], ldk, h->mW[l], h->vW[l], h->tr_dW.p, ld, lr_t, beta1,
                                      beta2, eps);
      count_launch();
      if (l < L - 1) {
        k_adam<<<8, 256, 0, st>>>(h->bias[l], 1, outw, 1, nullptr, 0, h->mB[l], h->vB[l], h->tr_db.p, 1, lr_t, beta1, beta2, eps);
        count_launch();
      }
      double* t = dcur; dcur = dnxt; dnxt = t;
    }
    h->dirty = 1;
  }
  if (loss_host) NNMPC_CUDA(cudaMemcpyAsync(loss_host, h->tr_loss, sizeof(double), cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaStreamSynchronize(st));
  NNMPC_CUDA(cudaGetLastError());
  return 0;
}

int nnmpc_mlp_get_weights(nnmpc_mlp_t* h, double* const* weights_host, double* const* biases_host) {
  if (!h || !weights_host) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_get_weights: null argument");
  DeviceGuard dg(h->device);
  NNMPC_CUDA(cudaDeviceSynchronize());
  for (int l = 0; l < h->L; ++l) {
    const int in = h->dims[l], outw = h->dims[l + 1], ld = h->ld[l];
    double* w = new (std::nothrow) double[(size_t)outw * ld];
    if (!w) return set_error(NNMPC_ERR_NOMEM, "out of host memory");
    cudaError_t e = cudaMemcpy(w, h->Wt[l], (size_t)outw * ld * sizeof(double), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess)
      for (int i = 0; i < in; ++i)
        for (int o = 0; o < outw; ++o) weights_host[l][(size_t)i * outw + o] = w[(size_t)o * ld + i];   // Keras layout (in, out)
    delete[] w;
    if (e == cudaSuccess && l < h->L - 1 && biases_host && biases_host[l])
      e = cudaMemcpy(biases_host[l], h->bias[l], (size_t)outw * sizeof(double), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return set_error(NNMPC_ERR_CUDA, "nnmpc_mlp_get_weights: %s", cudaGetErrorString(e));
  }
  return 0;
}

int nnmpc_mlp_forward(nnmpc_mlp_t* h, long long B, const double* x, const double* uprev, const double* xs,
                      const double* us, const double* xscale, const double* ulb, const double* uub, double* out,
                      void* stream) {
  if (B == 0 && h) return 0;
  if (!h || !x || !xs || !us || !out) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_forward: null argument");
  if (h->with_uprev && !uprev) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_forward: uprev required");
  if ((ulb == nullptr) != (uub == nullptr)) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_forward: ulb/uub both or none");
  if (B < 0) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_forward: negative batch");
  DeviceGuard dg(h->device);
  return mlp_forward_dispatch(h, B, x, uprev, xs, us, xscale, ulb, uub, out, (cudaStream_t)stream);
}

int nnmpc_mlp_forward_host(nnmpc_mlp_t* h, long long B, const double* x, const double* uprev, const double* xs,
                           const double* us, const double* xscale, const double* ulb, const double* uub, double* out) {
  if (B == 0 && h) return 0;
  if (!h || !x || !xs || !us || !out) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_forward_host: null argument");
  if (h->with_uprev && !uprev) return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_forward_host: uprev required");
  if ((ulb == nullptr) != (uub == nullptr))
    return set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_forward_host: ulb/uub both or none");
  if (B <= 0) return B == 0 ? 0 : set_error(NNMPC_ERR_BADARG, "nnmpc_mlp_forward_host: negative batch");
  DeviceGuard dg(h->device);
  const size_t b = (size_t)B;
  const int nx = h->nx, nu = h->nu;
  NNMPC_TRY(h->hx.ensure(b * nx));
  NNMPC_TRY(h->hxs.ensure(b * nx));
  NNMPC_TRY(h->hus.ensure(b * nu));
  NNMPC_TRY(h->hup.ensure(b * nu));
  NNMPC_TRY(h->hout.ensure(b * nu));
  NNMPC_TRY(h->hscale.ensure(nx));
  NNMPC_TRY(h->hlb.ensure(nu));
  NNMPC_TRY(h->hub.ensure(nu));
  cudaStream_t st = 0;
  NNMPC_CUDA(cudaMemcpyAsync(h->hx.p, x, b * nx * 8, cudaMemcpyHostToDevice, st));
  NNMPC_CUDA(cudaMemcpyAsync(h->hxs.p, xs, b * nx * 8, cudaMemcpyHostToDevice, st));
  NNMPC_CUDA(cudaMemcpyAsync(h->hus.p, us, b * nu * 8, cudaMemcpyHostToDevice, st));
  if (h->with_uprev) NNMPC_CUDA(cudaMemcpyAsync(h->hup.p, uprev, b * nu * 8, cudaMemcpyHostToDevice, st));
  if (xscale) NNMPC_CUDA(cudaMemcpyAsync(h->hscale.p, xscale, (size_t)nx * 8, cudaMemcpyHostToDevice, st));
  if (ulb) {
    NNMPC_CUDA(cudaMemcpyAsync(h->hlb.p, ulb, (size_t)nu * 8, cudaMemcpyHostToDevice, st));
    NNMPC_CUDA(cudaMemcpyAsync(h->hub.p, uub, (size_t)nu * 8, cudaMemcpyHostToDevice, st));
  }
  NNMPC_TRY(mlp_forward_dispatch(h, B, h->hx.p, h->with_uprev ? h->hup.p : nullptr, h->hxs.p, h->hus.p,
                                 xscale ? h->hscale.p : nullptr, ulb ? h->hlb.p : nullptr, ulb ? h->hub.p : nullptr,
                                 h->hout.p, st));
  NNMPC_CUDA(cudaMemcpyAsync(out, h->hout.p, b * nu * 8, cudaMemcpyDeviceToHost, st));
  NNMPC_CUDA(cudaStreamSynchronize(st));
  return 0;
}

}  // extern "C"
