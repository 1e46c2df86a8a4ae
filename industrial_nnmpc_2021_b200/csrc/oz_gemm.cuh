// FP64-accurate GEMM on the INT8 tcgen05 tensor cores (error-free "Ozaki" slicing), sm_100a.
//
//   C[M x N] = A[M x K] * Bt[N x K]^T          A: per-sample FP64 rows, Bt: a shared FP64 operator
//
// The mixed-precision regulator-QP engine needs two FP64-exact operator applies per QP - the anchor
// x = Top w - c that starts it and the KKT check g = P z + q that certifies it
// (/root/reference/lib/linearMPC.py:503-504 is the cvxopt solve both replace) - and on B200 the FP64
// tensor pipe (DMMA, 36 TFLOP/s) made them half of the closed-loop step.  Here every row of A and of Bt is
// scaled by a power of two into [-1/2, 1/2] and cut into signed base-128 digits
//     a = 2^f sum_i a_i 128^-(i+1),   b = 2^e sum_j b_j 128^-(j+1),   a_i, b_j in [-64, 64]  (int8, exact)
// so that  a . b = 2^(f+e) sum_L 128^-(L+2) sum_{i+j=L} sum_k a_i[k] b_j[k].  The inner sums are INT8 GEMMs
// with INT32 accumulation, which is EXACT (|sum| <= 8 pairs x K x 2^12 <= 2^30 < 2^31 for K <= 32768, the
// longest contraction oz_slice_operator accepts), so the only error is the truncation at level LMAX: at most (LMAX+1) K 2^(-7 (LMAX+1) - 2) relative to 2^(f+e)
// (LMAX = 7, K = 4480: 1.2e-13 - below the rounding error of an FP64 dot product of that length), plus the
// final FP64 summation of the levels.  36 INT8 products replace one FP64 product at 1/125 of its cost each.
//
// Kernel structure (persistent, one CTA per SM, warp specialised):
//   warp 0     TMA producer.  Per 128-byte k-block: the NS operator-slice tiles (64 rows x 128 B each) into a
//              double-buffered set, then the NS sample-slice tiles (128 rows x 128 B) through a 4-slot ring,
//              highest slice first (it has the fewest products, so the ring drains slowly at first and the next
//              k-block's operator set is in flight long before it is needed)
//   warp 1     one thread issues tcgen05.mma.kind::i8 (M = 128, N = 64, K = 32): product (i, j) accumulates into
//              TMEM level i + j (LMAX + 1 accumulators of 64 columns = all 512 TMEM columns at LMAX = 7)
//   warps 2-5  epilogue: tcgen05.ld the int32 levels of the warp's 32 rows, fold them in FP64 from the
//              smallest level up, scale by 2^(f+e), hand 16-column row chunks to the fused epilogue functor
#pragma once
#include "lp_gemm.cuh"   // PTX wrappers shared with the fp16 kernel (mbarrier, TMA, TMEM, descriptors)

namespace nnmpc {
namespace oz {

constexpr int BM = 128;            // sample rows per tile = TMEM lanes
constexpr int BN = 64;             // operator rows (output columns) per tile
constexpr int BKB = 128;           // bytes (= int8 elements) per k-block = one 128-byte swizzle span
constexpr int UMMA_KB = 32;        // int8 elements per tcgen05.mma
constexpr int NS_MAX = 8;          // slices kept per number (56 bits)
constexpr int A_SLOTS = 4;
constexpr int B_STAGES = 2;
constexpr int A_TILE = BM * BKB;   // 16 KB
constexpr int B_TILE = BN * BKB;   // 8 KB
constexpr int THREADS = 192;
constexpr int TMEM_COLS = 512;
constexpr int CH = 16;             // columns per epilogue chunk
constexpr int SMEM_BYTES = A_SLOTS * A_TILE + B_STAGES * NS_MAX * B_TILE + 1024 + 256;
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory");

__host__ __device__ constexpr uint32_t make_idesc_i8(int M, int N) {
  // c_format S32 (2) | a_format signed 8 bit (1) | b_format signed 8 bit (1) | both K-major | N >> 3 | M >> 4
  return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

struct OzShape {
  int M;               // rows of A (upper bound when m_dev is given)
  int N;               // rows of Bt = output columns
  int KB;              // k-blocks of 128 bytes (the slice buffers are zero padded to whole blocks)
  const int* m_dev;    // optional device-side row count
  long long a_rows_pad;   // rows per slice in the stacked sample-slice matrix
  long long b_rows_pad;   // rows per slice in the stacked operator-slice matrix
  const double* fscale;   // per position: 2^f of the sample row
  const double* escale;   // per output column: 2^e of the operator row
  int group_rows;      // row tiles per L2 group (<= 0: all)
};

// tile order: super-groups of group_rows row tiles; inside one, column tile major / row tile minor, so the CTAs in
// flight share a few operator column tiles and one group of sample rows (both stay in L2)
__device__ __forceinline__ void oz_tile_coords(int t, int ntm, int ntn, int group_rows, int& bm, int& bn) {
  if (group_rows <= 0 || group_rows >= ntm) {
    bn = t / ntm;
    bm = t - bn * ntm;
    return;
  }
  const int per_group = group_rows * ntn;
  const int gi = t / per_group;
  const int rem = t - gi * per_group;
  const int r0 = gi * group_rows;
  const int gr = (ntm - r0 < group_rows) ? ntm - r0 : group_rows;
  bn = rem / gr;
  bm = r0 + (rem - bn * gr);
}

// Epilogue concept (one lane owns one output row of the tile):
//   struct Epi { struct Params {...};
//     __device__ Epi(const Params&);
//     __device__ void begin_row(int pos, bool row_ok);          // pos = position in the row list
//     __device__ void chunk(int col0, const double (&v)[CH], int N);   // CH consecutive columns of this row
//     __device__ void end_row();
//   };
template <int LMAX, class Epi>
__global__ void __launch_bounds__(THREADS, 1)
oz_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, OzShape g,
               typename Epi::Params ep) {
  constexpr int NS = LMAX + 1;
  static_assert(NS <= NS_MAX && NS * BN <= TMEM_COLS, "levels");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* a_ring = base;                                   // A_SLOTS x 16 KB
  uint8_t* b_sets = base + A_SLOTS * A_TILE;                // B_STAGES x NS_MAX x 8 KB
  uint64_t* bars = reinterpret_cast<uint64_t*>(b_sets + B_STAGES * NS_MAX * B_TILE);
  uint64_t* a_full = bars;                    // [A_SLOTS]
  uint64_t* a_empty = a_full + A_SLOTS;       // [A_SLOTS]
  uint64_t* b_full = a_empty + A_SLOTS;       // [B_STAGES]
  uint64_t* b_empty = b_full + B_STAGES;      // [B_STAGES]
  uint64_t* acc_full = b_empty + B_STAGES;    // [1]
  uint64_t* acc_empty = acc_full + 1;         // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int M = g.m_dev ? min(*g.m_dev, g.M) : g.M;
  const int ntn = (g.N + BN - 1) / BN;
  const int ntm = (M + BM - 1) / BM;
  const int tiles = ntn * ntm;

  if (warp == 0 && lane == 0) {
    lp::tma_prefetch_desc(&tmA);
    lp::tma_prefetch_desc(&tmB);
    for (int s = 0; s < A_SLOTS; ++s) {
      lp::mbar_init(a_full + s, 1);
      lp::mbar_init(a_empty + s, 1);
    }
    for (int s = 0; s < B_STAGES; ++s) {
      lp::mbar_init(b_full + s, 1);
      lp::mbar_init(b_empty + s, 1);
    }
    lp::mbar_init(acc_full, 1);
    lp::mbar_init(acc_empty, 4);     // one arrival per epilogue warp
    lp::fence_barrier_init();
  }
  if (warp == 1) lp::tmem_alloc(tmem_slot, TMEM_COLS);
  lp::tc_fence_before();
  __syncthreads();
  lp::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      int as = 0, bs = 0;
      uint32_t aph = 0, bph = 0;
      for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
        int bm, bn;
        oz_tile_coords(t, ntm, ntn, g.group_rows, bm, bn);
        for (int kb = 0; kb < g.KB; ++kb) {
          lp::mbar_wait(b_empty + bs, bph ^ 1);
          lp::mbar_expect_tx(b_full + bs, NS * B_TILE);
          for (int j = 0; j < NS; ++j)
            lp::tma_load_2d_hint(b_sets + (bs * NS_MAX + j) * B_TILE, &tmB, b_full + bs, kb * BKB,
                                 (int)(j * g.b_rows_pad) + bn * BN, lp::L2_EVICT_LAST);
          if (++bs == B_STAGES) { bs = 0; bph ^= 1; }
          for (int i = LMAX; i >= 0; --i) {
            lp::mbar_wait(a_empty + as, aph ^ 1);
            lp::mbar_expect_tx(a_full + as, A_TILE);
            lp::tma_load_2d(a_ring + as * A_TILE, &tmA, a_full + as, kb * BKB, (int)(i * g.a_rows_pad) + bm * BM);
            if (++as == A_SLOTS) { as = 0; aph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_i8(BM, BN);
      int as = 0, bs = 0;
      uint32_t aph = 0, bph = 0;
      uint32_t tph = 0;
      for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
        lp::mbar_wait(acc_empty, tph ^ 1);        // the epilogue has drained the accumulators
        lp::tc_fence_after();
        for (int kb = 0; kb < g.KB; ++kb) {
          lp::mbar_wait(b_full + bs, bph);
          lp::tc_fence_after();
          const uint32_t sb = lp::smem_u32(b_sets + bs * NS_MAX * B_TILE);
          for (int i = LMAX; i >= 0; --i) {
            lp::mbar_wait(a_full + as, aph);
            lp::tc_fence_after();
            const uint64_t da = lp::make_sw128_kmajor_desc(lp::smem_u32(a_ring + as * A_TILE));
            for (int j = 0; j <= LMAX - i; ++j) {
              const uint64_t db = lp::make_sw128_kmajor_desc(sb + j * B_TILE);
              const uint32_t tacc = tmem_base + (uint32_t)((i + j) * BN);
#pragma unroll
              for (int k = 0; k < BKB / UMMA_KB; ++k)   // level i + j is first written by (i, j = 0) in this order
                umma_i8(tacc, da + 2 * k, db + 2 * k, idesc, (kb | j | k) ? 1u : 0u);
            }
            lp::umma_commit(a_empty + as);
            if (++as == A_SLOTS) { as = 0; aph ^= 1; }
          }
          lp::umma_commit(b_empty + bs);
          if (++bs == B_STAGES) { bs = 0; bph ^= 1; }
        }
        lp::umma_commit(acc_full);
        tph ^= 1;
      }
    }
  } else {
    // ===== epilogue warps: TMEM lane quarter = warp % 4 =====
    const int q = warp & 3;
    Epi epi(ep);
    uint32_t tph = 0;
    for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
      int bm, bn;
      oz_tile_coords(t, ntm, ntn, g.group_rows, bm, bn);
      const int pos = bm * BM + q * 32 + lane;
      const bool rok = pos < M;
      const double fs = rok ? g.fscale[pos] : 0.0;
      epi.begin_row(pos, rok);
      lp::mbar_wait(acc_full, tph);
      lp::tc_fence_after();
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
      for (int c = 0; c < BN / CH; ++c) {
        double v[CH];
#pragma unroll
        for (int k = 0; k < CH; ++k) v[k] = 0.0;
        // smallest level first: v = (v + acc_L) / 128 folds the levels exactly like a Horner scheme
#pragma unroll
        for (int L = LMAX; L >= 0; --L) {
          uint32_t acc[CH];
          lp::tmem_ld_32x16(trow + (uint32_t)(L * BN + c * CH), acc);
          lp::tmem_ld_wait();
#pragma unroll
          for (int k = 0; k < CH; ++k) v[k] = (v[k] + (double)(int)acc[k]) * 0.0078125;
        }
        const int col0 = bn * BN + c * CH;
#pragma unroll
        for (int k = 0; k < CH; ++k) {
          const int col = col0 + k;
          const double es = col < g.N ? g.escale[col] : 0.0;
          v[k] = v[k] * 0.0078125 * fs * es;      // 128^-(L+2) 2^(f+e)
        }
        if (rok) epi.chunk(col0, v, g.N);
      }
      epi.end_row();
      lp::tc_fence_before();
      __syncwarp();
      if (lane == 0) lp::mbar_arrive(acc_empty);
      tph ^= 1;
    }
  }

  lp::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    lp::tc_fence_after();
    lp::tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ---- second-generation kernel: level windows, 128-column tiles, just-in-time operator slices -----------
// A tcgen05.mma with both operands in shared memory reads A (128 x 32 B) and B (N x 32 B) for every
// instruction, so an N = 64 tile moves 6 KB per 262k MACs and is bound by the 128 B/clk shared-memory port, not
// by the INT8 pipe; N = 128 moves 8 KB per 524k MACs.  128 columns x 8 levels do not fit TMEM (512 columns), so
// the levels are computed in two launches of 4 accumulators each: levels 4..7 first (raw partial sums to a
// scratch matrix), then levels 0..3, whose epilogue adds the partial sums and runs the fused functor.
// Operator slices are not double buffered as a set in the high window: with the products ordered i ascending /
// j descending, slice B_j is last used by sample slice i = LHI - j and first used (next k-block) by
// i = max(0, LLO - j), so each B_j has its own slot and is refilled just in time, in exactly the order the slots
// are released.  The low window (slices 0..3) fits twice and double buffers them.  Eight epilogue warps (two per
// TMEM lane quarter) fold the levels, because with TMEM full the epilogue is exposed time.
// Measured on B200 (tools/probes/oz_rates.py, profiles/r01ao_oz_rates.txt): 72 TFLOP/s FP64-equivalent
// (2.6 POP/s INT8) from 1024 rows up, 2.0x cuBLAS DGEMM, errors <= 3e-12 on N(0,1) operands of length 4480.
constexpr int EPI_WARPS2 = 8;                   // two warps per TMEM lane quarter, each folds half of the tile's columns
constexpr int THREADS2 = 64 + 32 * EPI_WARPS2;  // the accumulators are not double buffered (TMEM is full), so the
                                                // epilogue is exposed time: 8 warps halve it

template <int BN2_>
struct OzTile2 {
  static constexpr int BN = BN2_;
  static constexpr int B_TILE = BN * BKB;
  static constexpr int A_SLOTS = (BN == 128) ? 5 : 8;
  static constexpr int SMEM_BYTES = A_SLOTS * A_TILE + NS_MAX * B_TILE + 1024 + 512;
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory");
};

struct OzShape2 {
  OzShape s;
  const double* partial_in;   // nullable: per (position, column) partial sum of the lower levels, added before scaling
  long long ldp;
  int raw_out;                // 1: hand the unscaled level sum to the functor (partial-sum store)
};

template <int LLO, int LHI, int BN_, class Epi>
__global__ void __launch_bounds__(THREADS2, 1)
oz_gemm2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, OzShape2 g2,
                typename Epi::Params ep) {
  using T = OzTile2<BN_>;
  constexpr int BN = T::BN;
  constexpr int NL = LHI - LLO + 1;
  static_assert(LHI < NS_MAX && LLO >= 0 && NL >= 1 && NL * BN <= TMEM_COLS, "level window");
  // A window that uses at most half of the operator-slice slots (levels 0..3: slices 0..3) double buffers them:
  // there every slice is needed again within a few products of its release, too soon for a just-in-time refill
  // (measured: 29 % tensor-pipe activity for window 0..3 against 54 % for window 4..7).
  constexpr int NSB = LHI + 1;                          // operator slices this window uses
  constexpr bool DB = 2 * NSB <= NS_MAX;
  // A window that fits TMEM twice (e.g. levels 0..3 at 64 columns: 256 of 512) double buffers the accumulators, so
  // the level-folding epilogue of a tile overlaps the products of the next one - what matters when the contraction
  // is short (structured-network layers: K = 568 .. 1024, 5 - 8 k-blocks per tile).
  constexpr int ACC = (2 * NL * BN <= TMEM_COLS) ? 2 : 1;
  auto b_slot = [](int j, uint32_t kbc) -> int { return DB ? (int)(kbc & 1u) * NSB + j : j; };
  auto b_par = [](uint32_t kbc) -> uint32_t { return DB ? (kbc >> 1) & 1u : kbc & 1u; };
  const OzShape& g = g2.s;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* a_ring = base;                                   // A_SLOTS x 16 KB
  uint8_t* b_slots = base + T::A_SLOTS * A_TILE;            // NS_MAX x B_TILE (slot j holds operator slice j)
  uint64_t* bars = reinterpret_cast<uint64_t*>(b_slots + NS_MAX * T::B_TILE);
  uint64_t* a_full = bars;                      // [A_SLOTS]
  uint64_t* a_empty = a_full + T::A_SLOTS;      // [A_SLOTS]
  uint64_t* b_full = a_empty + T::A_SLOTS;      // [NS_MAX]
  uint64_t* b_empty = b_full + NS_MAX;          // [NS_MAX]
  uint64_t* acc_full = b_empty + NS_MAX;        // [ACC]
  uint64_t* acc_empty = acc_full + 2;           // [ACC]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int M = g.m_dev ? min(*g.m_dev, g.M) : g.M;
  const int ntn = (g.N + BN - 1) / BN;
  const int ntm = (M + BM - 1) / BM;
  const int tiles = ntn * ntm;

  if (warp == 0 && lane == 0) {
    lp::tma_prefetch_desc(&tmA);
    lp::tma_prefetch_desc(&tmB);
    for (int s = 0; s < T::A_SLOTS; ++s) {
      lp::mbar_init(a_full + s, 1);
      lp::mbar_init(a_empty + s, 1);
    }
    for (int s = 0; s < NS_MAX; ++s) {
      lp::mbar_init(b_full + s, 1);
      lp::mbar_init(b_empty + s, 1);
    }
    for (int s = 0; s < ACC; ++s) {
      lp::mbar_init(acc_full + s, 1);
      lp::mbar_init(acc_empty + s, EPI_WARPS2);
    }
    lp::fence_barrier_init();
  }
  if (warp == 1) lp::tmem_alloc(tmem_slot, TMEM_COLS);
  lp::tc_fence_before();
  __syncthreads();
  lp::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer: per k-block  A_0, B_LHI..B_LLO, A_1, B_(LLO-1), A_2, B_(LLO-2), ...  (order of first use) =====
    if (lane == 0) {
      int as = 0;
      uint32_t aph = 0, kbc = 0;       // kbc: running k-block count (a B slot turns over once per k-block, or per two when double buffered)
      for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
        int bm, bn;
        oz_tile_coords(t, ntm, ntn, g.group_rows, bm, bn);
        for (int kb = 0; kb < g.KB; ++kb, ++kbc) {
          const uint32_t bph = b_par(kbc);
          for (int i = 0; i <= LHI; ++i) {
            lp::mbar_wait(a_empty + as, aph ^ 1);
            lp::mbar_expect_tx(a_full + as, A_TILE);
            lp::tma_load_2d(a_ring + as * A_TILE, &tmA, a_full + as, kb * BKB, (int)(i * g.a_rows_pad) + bm * BM);
            if (++as == T::A_SLOTS) { as = 0; aph ^= 1; }
            const int jhi = (i == 0) ? LHI : LLO - i;      // slices first used by sample slice i
            const int jlo = (i == 0) ? LLO : LLO - i;
            for (int j = jhi; j >= jlo && j >= 0; --j) {
              const int sl = b_slot(j, kbc);
              lp::mbar_wait(b_empty + sl, bph ^ 1);
              lp::mbar_expect_tx(b_full + sl, T::B_TILE);
              lp::tma_load_2d_hint(b_slots + sl * T::B_TILE, &tmB, b_full + sl, kb * BKB, (int)(j * g.b_rows_pad) + bn * BN,
                                   lp::L2_EVICT_LAST);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    // The whole warp runs this loop with uniform control flow and lane 0 issues: the product schedule is fully
    // unrolled (LLO, LHI are compile-time), so every descriptor is a warp-uniform value plus a constant and an
    // instruction costs a few issue slots.  (With a divergent single-thread loop the issuing thread spent ~16
    // instructions per tcgen05.mma and was the bottleneck of the first-generation kernel: 75 clk per
    // 128 x 64 x 32 product against 48 clk of shared-memory time.)
    constexpr uint32_t idesc = make_idesc_i8(BM, BN);
    const bool issue = lane == 0;
    int as = 0;
    uint32_t aph = 0, kbc = 0, ti = 0;
    const uint64_t da_base = lp::make_sw128_kmajor_desc(lp::smem_u32(a_ring));
    const uint64_t db_base = lp::make_sw128_kmajor_desc(lp::smem_u32(b_slots));
    for (int t = blockIdx.x; t < tiles; t += gridDim.x, ++ti) {
      const uint32_t acs = ACC == 2 ? (ti & 1u) : 0u;                       // accumulator stage of this tile
      const uint32_t tph = ACC == 2 ? (ti >> 1) & 1u : ti & 1u;             // its phase
      lp::mbar_wait(acc_empty + acs, tph ^ 1);
      lp::tc_fence_after();
      for (int kb = 0; kb < g.KB; ++kb, ++kbc) {
        const uint32_t first = kb ? 1u : 0u;
        const uint32_t bph = b_par(kbc);
        const int sbase = DB ? (int)(kbc & 1u) * NSB : 0;      // first operator-slice slot of this k-block
#pragma unroll
        for (int i = 0; i <= LHI; ++i) {
          lp::mbar_wait(a_full + as, aph);
          lp::tc_fence_after();
          const uint64_t da = da_base + (uint64_t)(as * (A_TILE >> 4));
#pragma unroll
          for (int j = LHI - i; j >= (LLO - i > 0 ? LLO - i : 0); --j) {
            if (i == (LLO - j > 0 ? LLO - j : 0)) {          // first use of slice j in this k-block (compile-time)
              lp::mbar_wait(b_full + sbase + j, bph);
              lp::tc_fence_after();
            }
            const uint64_t db = db_base + (uint64_t)((sbase + j) * (T::B_TILE >> 4));
            const uint32_t tacc = tmem_base + (uint32_t)((acs * NL + (i + j - LLO)) * BN);
            if (issue) {
              // every level of the window is first written by sample slice 0, step 0 of the tile's first k-block
              umma_i8(tacc, da, db, idesc, i == 0 ? first : 1u);
              umma_i8(tacc, da + 2, db + 2, idesc, 1u);
              umma_i8(tacc, da + 4, db + 4, idesc, 1u);
              umma_i8(tacc, da + 6, db + 6, idesc, 1u);
            }
          }
          if (issue) {
            lp::umma_commit(a_empty + as);
            lp::umma_commit(b_empty + sbase + (LHI - i));     // slice LHI - i was last used by sample slice i
          }
          __syncwarp();
          if (++as == T::A_SLOTS) { as = 0; aph ^= 1; }
        }
      }
      if (issue) lp::umma_commit(acc_full + acs);
      __syncwarp();
    }
  } else {
    // ===== epilogue warps =====
    const int q = warp & 3;                       // TMEM lane quarter this warp may read
    const int hsel = (warp - 2) >> 2;             // which half of the tile's column chunks it folds
    constexpr int CHUNKS = BN / CH / 2;
    Epi epi(ep);
    uint32_t ti = 0;
    // 128^-(LLO+1) as a compile-time power of two
    const double lev0 = __longlong_as_double((long long)(1023 - 7 * (LLO + 1)) << 52);
    for (int t = blockIdx.x; t < tiles; t += gridDim.x, ++ti) {
      const uint32_t acs = ACC == 2 ? (ti & 1u) : 0u;
      const uint32_t tph = ACC == 2 ? (ti >> 1) & 1u : ti & 1u;
      int bm, bn;
      oz_tile_coords(t, ntm, ntn, g.group_rows, bm, bn);
      const int pos = bm * BM + q * 32 + lane;
      const bool rok = pos < M;
      const double fs = rok ? g.fscale[pos] : 0.0;
      epi.begin_row(pos, rok);
      lp::mbar_wait(acc_full + acs, tph);
      lp::tc_fence_after();
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acs * NL * BN);
#pragma unroll 1
      for (int c = hsel * CHUNKS; c < (hsel + 1) * CHUNKS; ++c) {
        double v[CH];
        // what the chunk adds and scales with is requested BEFORE the TMEM loads and the level fold, so that its
        // latency (the partial sums of the other window come from HBM) is covered by them: with single-buffered
        // accumulators the epilogue of the low window is as long as its products (round-1 profile: half of the
        // tile time), and these loads used to be issued at their first use
        const int colc = bn * BN + c * CH;
        double pin[CH], es[CH];
        {
          // whole chunk inside and an even row pitch of the partial sums: 16-byte loads (colc is a multiple of 16)
          const bool vec_ok = colc + CH <= g.N && (!g2.partial_in || (g2.ldp & 1) == 0);
          const bool has_p = g2.partial_in && rok;
          const double* pp = g2.partial_in + (has_p ? (long long)pos * g2.ldp + colc : 0);
#pragma unroll
          for (int k = 0; k < CH; k += 2) {
            double2 t = make_double2(0.0, 0.0), e2 = make_double2(0.0, 0.0);
            if (vec_ok) {
              if (has_p) t = *reinterpret_cast<const double2*>(pp + k);
              if (!g2.raw_out) e2 = *reinterpret_cast<const double2*>(g.escale + colc + k);
            } else {
              if (has_p && colc + k < g.N) t.x = pp[k];
              if (has_p && colc + k + 1 < g.N) t.y = pp[k + 1];
              if (!g2.raw_out && colc + k < g.N) e2.x = g.escale[colc + k];
              if (!g2.raw_out && colc + k + 1 < g.N) e2.y = g.escale[colc + k + 1];
            }
            pin[k] = t.x; pin[k + 1] = t.y;
            es[k] = e2.x; es[k + 1] = e2.y;
          }
        }
        if constexpr (NL <= 4) {
          // Fold the levels in 64-bit INTEGER arithmetic (exact: |acc_L| < 2^31, three shifts by 7 bits stay below
          // 2^53) and convert once: one I2F + one multiply per element on the FP64 pipe instead of a convert, an add
          // and a multiply per LEVEL.  The FP64 ALU (64 FMA/clk/SM on B200) is what the epilogue of a short
          // contraction is bound by.
          long long sacc[CH];
#pragma unroll
          for (int k = 0; k < CH; ++k) sacc[k] = 0;
#pragma unroll
          for (int L = 0; L < NL; ++L) {
            uint32_t acc[CH];
            lp::tmem_ld_32x16(trow + (uint32_t)(L * BN + c * CH), acc);
            lp::tmem_ld_wait();
#pragma unroll
            for (int k = 0; k < CH; ++k) sacc[k] = sacc[k] * 128 + (long long)(int)acc[k];
          }
          // sum_L acc_L 128^(NL-1-L) x 128^-NL x 128^-(LLO+1) = sum_L acc_L 128^-(L+LLO+2)
          const double wnl = __longlong_as_double((long long)(1023 - 7 * (NL + LLO + 1)) << 52);
#pragma unroll
          for (int k = 0; k < CH; ++k) v[k] = (double)sacc[k] * wnl;
        } else {
#pragma unroll
          for (int k = 0; k < CH; ++k) v[k] = 0.0;
#pragma unroll
          for (int L = NL - 1; L >= 0; --L) {
            uint32_t acc[CH];
            lp::tmem_ld_32x16(trow + (uint32_t)(L * BN + c * CH), acc);
            lp::tmem_ld_wait();
#pragma unroll
            for (int k = 0; k < CH; ++k) v[k] = (v[k] + (double)(int)acc[k]) * 0.0078125;
          }
#pragma unroll
          for (int k = 0; k < CH; ++k) v[k] *= lev0;                 // sum_L acc_L 128^-(L+2)
        }
        const int col0 = colc;
#pragma unroll
        for (int k = 0; k < CH; ++k) {
          v[k] += pin[k];                              // 0 where there is no partial sum (or the column is outside)
          if (!g2.raw_out) v[k] *= fs * es[k];         // es = 0 outside N
        }
        if (rok) epi.chunk(col0, v, g.N);
      }
      epi.end_row();
      lp::tc_fence_before();
      __syncwarp();
      if (lane == 0) lp::mbar_arrive(acc_empty + acs);
    }
  }

  lp::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    lp::tc_fence_after();
    lp::tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

template <int LLO, int LHI, int BN_, class Epi>
inline cudaError_t launch_oz_gemm2(const CUtensorMap& tmA, const CUtensorMap& tmB, const OzShape2& g,
                                   const typename Epi::Params& ep, int num_sms, cudaStream_t st) {
  using T = OzTile2<BN_>;
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!configured[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(oz_gemm2_kernel<LLO, LHI, BN_, Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         T::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    configured[dev & 63] = true;
  }
  if (g.s.M <= 0 || g.s.N <= 0 || g.s.KB <= 0) return cudaSuccess;
  const long long tiles = (long long)((g.s.N + T::BN - 1) / T::BN) * ((g.s.M + BM - 1) / BM);
  const unsigned grid = (unsigned)(tiles < num_sms ? tiles : num_sms);
  oz_gemm2_kernel<LLO, LHI, BN_, Epi><<<grid, THREADS2, T::SMEM_BYTES, st>>>(tmA, tmB, g, ep);
  return cudaGetLastError();
}

// max of |row| entries that keeps a NaN wherever it meets one ((b <= m) ? m : b alone drops an m that is NaN)
__device__ __forceinline__ double nan_max(double m, double b) { return (b <= m || m != m) ? m : b; }

// ---- slicing: one CTA per row; rows[] (optional) gathers the source rows, position p is the destination row -----
//   src row -> 2^f (max |a| <= 2^(f-1)) and NS signed base-128 digit planes dst[(s * rows_pad + p) * ldb + k]
template <int NS>
__global__ void __launch_bounds__(256)
k_oz_slice(const int* __restrict__ rows, const int* __restrict__ count, const double* __restrict__ src, long long ld_src,
           int ncols, int8_t* __restrict__ dst, long long rows_pad, long long ldb, double* __restrict__ scale_out,
           int max_rows) {
  // grid-stride over the listed rows (the grid is capped by the launcher; the list length lives on the device, or
  // every one of max_rows rows is taken)
  const long long total = count ? (*count < max_rows ? *count : max_rows) : (long long)max_rows;
  __shared__ double red[8];
  for (long long p = blockIdx.x; p < total; p += gridDim.x) {
    const long long r = rows ? rows[p] : p;
    const double* a = src + r * ld_src;
    double m = 0.0;
    for (int k = threadIdx.x; k < ncols; k += blockDim.x) {
      const double b = fabs(a[k]);
      m = nan_max(m, b);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double b = __shfl_xor_sync(0xffffffffu, m, o);
      m = nan_max(m, b);
    }
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    m = red[0];
    for (int w = 1; w < 8; ++w) m = nan_max(m, red[w]);
    __syncthreads();                                        // red[] is reused by the next row
    const bool bad = !(m <= 1.7e308);                       // NaN / Inf row: the result must not look finite
    int ex = 0;
    if (!bad && m > 0.0) frexp(m, &ex);                     // m = mant 2^ex, mant in [0.5, 1)  =>  m <= 2^ex = 2^(f-1)
    const double inv = bad ? 0.0 : ldexp(1.0, -(ex + 1));
    for (int k = threadIdx.x; k < ncols; k += blockDim.x) {
      double t = bad ? 0.0 : a[k] * inv;                    // |t| <= 1/2, exact
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        t *= 128.0;
        const double d = rint(t);                           // |d| <= 64
        t -= d;                                             // exact, |t| <= 1/2
        dst[((long long)s * rows_pad + p) * ldb + k] = (int8_t)(int)d;
      }
    }
    if (threadIdx.x == 0)
      scale_out[p] = bad ? __longlong_as_double(0x7ff8000000000000ll) : ldexp(1.0, ex + 1);
  }
}

// Same for SHORT rows (structured-network activations, K ~ 10^3): one warp per row, 8 rows per CTA, no block-wide
// synchronisation; every lane cuts 4 consecutive numbers per step and stores a char4 per digit plane.
template <int NS>
__global__ void __launch_bounds__(256)
k_oz_slice_warp(const double* __restrict__ src, long long ld_src, int ncols, int8_t* __restrict__ dst, long long rows_pad,
                long long ldb, double* __restrict__ scale_out, long long nrows) {
  const int lane = threadIdx.x & 31;
  const long long wpg = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long p = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); p < nrows; p += wpg) {
    const double* a = src + p * ld_src;
    double m = 0.0;
    for (int k = lane; k < ncols; k += 32) {
      const double b = fabs(a[k]);
      m = nan_max(m, b);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double b = __shfl_xor_sync(0xffffffffu, m, o);
      m = nan_max(m, b);
    }
    const bool bad = !(m <= 1.7e308);
    int ex = 0;
    if (!bad && m > 0.0) frexp(m, &ex);
    const double inv = bad ? 0.0 : ldexp(1.0, -(ex + 1));
    const int n4 = ncols & ~3;
    for (int k = 4 * lane; k < n4; k += 128) {
      double t[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) t[e] = bad ? 0.0 : a[k + e] * inv;
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        char4 d;
        int8_t* dd = reinterpret_cast<int8_t*>(&d);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          t[e] *= 128.0;
          const double r = rint(t[e]);
          t[e] -= r;
          dd[e] = (int8_t)(int)r;
        }
        *reinterpret_cast<char4*>(dst + ((long long)s * rows_pad + p) * ldb + k) = d;
      }
    }
    for (int k = n4 + lane; k < ncols; k += 32) {
      double t = bad ? 0.0 : a[k] * inv;
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        t *= 128.0;
        const double r = rint(t);
        t -= r;
        dst[((long long)s * rows_pad + p) * ldb + k] = (int8_t)(int)r;
      }
    }
    if (lane == 0) scale_out[p] = bad ? __longlong_as_double(0x7ff8000000000000ll) : ldexp(1.0, ex + 1);
  }
}

// uint8 row-major matrix [rows][cols bytes], leading dimension ld bytes -> tensor map with boxes of box_rows x 128 B
inline bool make_tmap_u8(CUtensorMap* tm, const void* base, long long rows, long long cols, long long ld, int box_rows) {
  lp::EncodeTiledFn fn = lp::encode_tiled_fn();
  if (!fn) return false;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld};
  cuuint32_t box[2] = {(cuuint32_t)BKB, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

template <int LMAX, class Epi>
inline cudaError_t launch_oz_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, const OzShape& g,
                                  const typename Epi::Params& ep, int num_sms, cudaStream_t st) {
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!configured[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(oz_gemm_kernel<LMAX, Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e != cudaSuccess) return e;
    configured[dev & 63] = true;
  }
  if (g.M <= 0 || g.N <= 0 || g.KB <= 0) return cudaSuccess;
  const long long tiles = (long long)((g.N + BN - 1) / BN) * ((g.M + BM - 1) / BM);
  const unsigned grid = (unsigned)(tiles < num_sms ? tiles : num_sms);
  oz_gemm_kernel<LMAX, Epi><<<grid, THREADS, SMEM_BYTES, st>>>(tmA, tmB, g, ep);
  return cudaGetLastError();
}

}  // namespace oz
}  // namespace nnmpc
