// b200ot — gaussian kernel convolution on the 5th-gen tensor cores, for dimensions where -2 x.y^T is a
// real dense contraction (8 < D <= 64):
//     out_i = sum_j w_j exp(-|x_i - y_j|^2 / (2 blur^2)) = sum_j w_j 2^( X_i.Y_j - |X_i|^2/2 - |Y_j|^2/2 )
// Reference semantics: gaussian_kernel + the matvecs of kernel_loss
// (src/geomloss/_legacy/kernel_samples.py:62-68, :116-137).
//
// The whole exponent is produced by tcgen05.mma into TMEM:
//   * each operand is split into TWO fp16 terms X = h + l (22 significant bits) and stored ONCE as [h | l] along
//     K; the three cross products that matter (hh, hl, lh: error ~2^-22 |X||Y|, measured <= 3e-6 relative on the
//     kernel value down to blur = .3 at D = 64) are formed by pointing the A and B operand addresses at the
//     matching segments — no duplicated data in shared memory or L2, 3*Dk/16 MMA instructions per tile, fp32
//     accumulation.  (First version: three bf16 terms and six products — twice the tensor work for accuracy the
//     fp32 accumulation cannot use; fp16's narrow range is harmless for centred, scaled coordinates.)
//   * one extra 16-wide K chunk, issued as a BF16 instruction (fp32 range: potentials / eps reach 1e5), carries
//     the rank-one terms:  A: [1,1,1, r_h,r_m,r_l, 0..],  B: [c_h,c_m,c_l, 1,1,1, 0..] with r = -|X|^2/2,
//     c = -|Y|^2/2 split in three bf16 terms,
//   so the epilogue is  tcgen05.ld -> MUFU.EX2 -> FFMA with the column weight  and nothing else.
//
// Operand tiles are pre-packed in global memory by tc_pack_kernel in the exact image the UMMA descriptors
// expect (K-major, no swizzle: for every 8-element K chunk the 16-byte pieces of all rows are
// contiguous), so a column tile is ONE 1-D bulk-TMA copy; the column weights ride at the end of the image.
// The ROW operand of a CTA is staged once into TMEM (tcgen05.st, lane = row, two bf16 per 32-bit column) and
// the MMAs run in TS mode: at M = 128 an SS-mode MMA needs 128 B/clk of shared-memory reads — the whole
// shared-memory bandwidth of the SM — and measured 1.34e12 pairs/s at D = 64; TS mode halves that and
// reached 1.58e12 with the six-product bf16 operands (1.27 PFLOP/s of MMA work, profiles/r01_conv_bench.jsonl).
// CTA = TMA warp + MMA warp (one elected thread issues) + NEPI epilogue warps; smem ring of column tiles
// with full/empty mbarriers; two accumulator buffers in TMEM so that the MMAs of tile t+1 overlap the
// exponentials of tile t.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "tc.cuh"

namespace b200ot {

constexpr int kTcM = 128;  // rows per CTA tile = M of the MMA

__host__ __device__ inline int tc_dk(int D) { return ((D + 15) / 16) * 16; }
constexpr int kTcTerms = 2;  // fp16 split terms per coordinate
// K extent of an operand image: the split terms + one 16-wide chunk of rank-one terms
__host__ __device__ inline int tc_kp(int D) { return kTcTerms * tc_dk(D) + 16; }
__host__ __device__ inline int tc_dk_of_kp(int kp) { return (kp - 16) / kTcTerms; }
__host__ __device__ inline int64_t tc_a_img_bytes(int kp) { return (int64_t)kTcM * kp * 2; }
// column image: bf16 operand data | fp32 weights
__host__ __device__ inline int64_t tc_b_img_bytes(int kp, int bn) { return (int64_t)bn * kp * 2 + (int64_t)bn * 4; }

// Laplacian / energy kernels: the coordinate scale s = max |x - c| over both clouds, computed on the device into the
// plan's misc block.  1/s as the pack kernel and the finalize both see it (bit-identical X in the two places).
__device__ inline float tc_coord_scale(const float* s_ptr) {
  const float s = *s_ptr;
  return (s > 0.f && s <= 3.0e38f) ? s : 1.f;  // all points on the centre (or a non-finite input): unit scale
}
__device__ inline float tc_coord_inv(const float* s_ptr) { return 1.f / tc_coord_scale(s_ptr); }

// ---------------------------------------------------------------------------------------------------
// pack: one thread per (padded) point; writes its 16-byte piece of every K chunk of its tile image
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 pack8_f16(const __half* src) {
  uint4 v;
  v.x = (uint32_t)__half_as_ushort(src[0]) | ((uint32_t)__half_as_ushort(src[1]) << 16);
  v.y = (uint32_t)__half_as_ushort(src[2]) | ((uint32_t)__half_as_ushort(src[3]) << 16);
  v.z = (uint32_t)__half_as_ushort(src[4]) | ((uint32_t)__half_as_ushort(src[5]) << 16);
  v.w = (uint32_t)__half_as_ushort(src[6]) | ((uint32_t)__half_as_ushort(src[7]) << 16);
  return v;
}

// Column images carry, besides the split coordinates, the per-column additive exponent term
//   c_j = h_scale * (h_a[j] + h_scale_b * h_b[j]) - |Y_j|^2 / 2      (h_a null: just the fold)
// in the rank-one chunk, and the fp32 weight w_j (kernel conv) behind the bf16 data.  Padding columns get
// c = -1e38 when h_a is given (softmin: they must vanish from the log-sum-exp) and w = 0 otherwise.
//
// coord_absmax (laplacian / energy): the device-side extent s of both clouds (coord_absmax_kernel); coordinates are
// then X = scale / s * (x - c), i.e. |X| <= scale, and the epilogues / finalize undo the 1/s.
static __global__ void tc_pack_kernel(const float* __restrict__ pts, const float* __restrict__ w,
                                      const float* __restrict__ h_a, const float* __restrict__ h_b,
                                      float h_scale_b, float h_scale, const float* __restrict__ center,
                                      float scale, int64_t n, int D, int kp, int tile, int is_cols,
                                      unsigned char* __restrict__ out,
                                      const float* __restrict__ row_extra = nullptr,
                                      const float* __restrict__ w_absmax = nullptr, int pad_tiles = 1,
                                      const float* __restrict__ coord_absmax = nullptr) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (coord_absmax != nullptr) scale *= tc_coord_inv(coord_absmax);
  const int64_t group = (int64_t)tile * pad_tiles;  // images are written for a multiple of pad_tiles tiles
  const int64_t npad = ((n + group - 1) / group) * group;
  if (p >= npad) return;
  const int64_t t = p / tile;
  const int pt = (int)(p % tile);
  const int dk = tc_dk(D);
  const int64_t img_bytes = (int64_t)tile * kp * 2 + (is_cols ? (int64_t)tile * 4 : 0);
  unsigned char* img = out + t * img_bytes;
  const bool live = p < n;
  float sq = 0.f;
  for (int kc = 0; kc < dk / 8; ++kc) {
    __half term[kTcTerms][8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int d = kc * 8 + k;
      float X = 0.f;
      if (live && d < D) X = scale * (pts[p * D + d] - (center ? center[d] : 0.f));
      X = fminf(fmaxf(X, -60000.f), 60000.f);  // fp16 range (only reached when every exponent underflows anyway)
      const __half h = __float2half_rn(X);
      const __half l = __float2half_rn(X - __half2float(h));
      // sqrt kernels: |X|^2 of the value the MMAs multiply (h + l, 22 bits) — with the fp32 X the expansion would
      // carry a 2^-22 |X|^2 bias in d^2, which sqrt turns into a relative error of r at near-coincident pairs
      const float Xq = (coord_absmax != nullptr) ? __half2float(h) + __half2float(l) : X;
      sq = fmaf(Xq, Xq, sq);
      term[0][k] = h;
      term[1][k] = l;
    }
#pragma unroll
    for (int s = 0; s < kTcTerms; ++s)
      *reinterpret_cast<uint4*>(img + ((int64_t)(s * (dk / 8) + kc) * tile + pt) * 16) = pack8_f16(term[s]);
  }
  // rank-one chunk (16 wide): rows [1,1,1, r_h,r_m,r_l, 0..]   columns [c_h,c_m,c_l, 1,1,1, 0..]
  {
    float r = live ? -0.5f * sq : 0.f;
    if (!is_cols && row_extra != nullptr && live) r -= row_extra[p];  // softmin backward: exponent - lse2_i
    if (is_cols && h_a != nullptr) {
      if (live) {
        float h = h_a[p];
        if (h_b != nullptr) h = fmaf(h_scale_b, h_b[p], h);
        r = fmaf(h_scale, h, r);
      } else {
        r = -1.0e38f;
      }
    }
    const __nv_bfloat16 rh = __float2bfloat16_rn(r);
    const float q1 = r - __bfloat162float(rh);
    const __nv_bfloat16 rm = __float2bfloat16_rn(q1);
    const __nv_bfloat16 rl = __float2bfloat16_rn(q1 - __bfloat162float(rm));
    const uint32_t one = 0x3F80u;  // bf16 1.0
    const uint32_t a = __bfloat16_as_ushort(rh), b = __bfloat16_as_ushort(rm), c = __bfloat16_as_ushort(rl);
    uint4 v;
    if (is_cols) {
      v.x = a | (b << 16);
      v.y = c | (one << 16);
      v.z = one | (one << 16);
    } else {
      v.x = one | (one << 16);
      v.y = one | (a << 16);
      v.z = b | (c << 16);
    }
    v.w = 0u;
    const int chunk = kTcTerms * (dk / 8);
    *reinterpret_cast<uint4*>(img + ((int64_t)chunk * tile + pt) * 16) = v;
    *reinterpret_cast<uint4*>(img + ((int64_t)(chunk + 1) * tile + pt) * 16) = make_uint4(0u, 0u, 0u, 0u);
  }
  if (is_cols) {
    // (row-gradient kernels feed P = w e to an fp16 GEMM: weights are normalised to |w| <= 1, undone in the finalize)
    float wv = (live && w) ? w[p] : 0.f;
    if (w_absmax != nullptr && *w_absmax > 0.f) wv /= *w_absmax;
    reinterpret_cast<float*>(img + (int64_t)tile * kp * 2)[pt] = wv;
  }
}

// ---------------------------------------------------------------------------------------------------
// the reduction kernel
// ---------------------------------------------------------------------------------------------------
constexpr int kTcMaxStage = 4;
constexpr int kTcRT = 2;  // row tiles per CTA in the forward kernels (each column tile is used twice from shared memory)

template <int BN_, int NEPI_>
struct TcCfg {
  static constexpr int BN = BN_;          // columns per tile = N of the MMA
  static constexpr int NEPI = NEPI_;      // epilogue warps (4, 8 or 16)
  static constexpr int THREADS = 64 + 32 * NEPI;
  static constexpr int A_COL0 = kTcRT * BN;  // the row operands live in TMEM behind the accumulators
  static constexpr int A_COLS = 80;          // per row tile: kp/2 <= 72 columns (D <= 64: kp = 144 halves)
  static constexpr int TMEM_COLS = 512;
  static_assert(A_COL0 + kTcRT * A_COLS <= 512, "TMEM budget");
  static_assert(NEPI == 4 || NEPI == 8 || NEPI == 16, "epilogue warps come in groups of four (one per TMEM lane quarter)");
  static_assert(BN % 64 == 0 && BN <= 128, "unsupported column tile");
};

// MODE 0: gaussian kernel conv  part[(split*NH + half)*N + row]   = sum_j w_j 2^S_ij
// MODE 1: softmin               part2[(split*NH + half)*N + row]  = (m, s) with sum_j 2^S_ij = s 2^m  (lazy max,
//         sum-guarded exactly like softmin.cuh; same partial format as softmin_partial_kernel)
// MODE 4: laplacian kernel conv  part[...] = sum_j w_j 2^(-kc s r_ij)      r = sqrt(max(-2 S_ij, clampq / s^2))
// MODE 5: energy kernel conv     part[...] = s sum_j w_j r_ij              (the caller negates: k = -|x - y|)
//         S is accumulated on coordinates X = (x - c) / s (|X| <= 1: tc_pack_kernel's coord_absmax), so r is the
//         distance in units of s; kc = log2(e) / blur; clampq = the clamp on |x - y|^2 in the units of x.
// (row gradients — modes 2 and 3, 4 and 5 — are a two-GEMM kernel of their own: tcbwd.cuh)
//
// A CTA owns kTcRT = 2 row tiles (2 x 128 rows) and ping-pongs between them: step (k, r) multiplies row tile r by
// column tile k into accumulator r, so (i) every column tile fetched from L2 feeds 2 x 128 rows — at one row tile
// per CTA the kernel was L2 -> shared-memory bound (5.8 TB/s at D = 64) — and (ii) the MMAs of step (k, 1) overlap
// the exponentials of step (k, 0), those of (k+1, 0) the exponentials of (k, 1): the two accumulators double as
// the double buffer.
template <class C, int MODE>
__global__ void __launch_bounds__(C::THREADS, 1)
    tc_reduce_kernel(const unsigned char* __restrict__ a_imgs, const unsigned char* __restrict__ b_imgs,
                     float* __restrict__ part, int64_t N, int kp, int ntiles_b, int tiles_per_split, int NSTAGE,
                     int D, int self_mode, float kc = 0.f, float clampq = 0.f,
                     const float* __restrict__ coord_absmax = nullptr) {
  constexpr int BN = C::BN, NEPI = C::NEPI, RT = kTcRT;
  static_assert(MODE == 0 || MODE == 1 || MODE == 4 || MODE == 5, "row gradients live in tcbwd.cuh");
  constexpr bool SQRT = MODE >= 4;
  extern __shared__ __align__(1024) unsigned char smem[];
  const int a_bytes = kTcM * kp * 2;
  const int b_bytes = BN * kp * 2 + BN * 4;
  unsigned char* sb = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NSTAGE * b_bytes);
  uint64_t* bar_a = bars;
  uint64_t* full_b = bars + 1;
  uint64_t* empty_b = full_b + kTcMaxStage;
  uint64_t* tmem_full = empty_b + kTcMaxStage;
  uint64_t* tmem_empty = tmem_full + RT;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + RT);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row_tile0 = blockIdx.x * RT;  // (the row images are padded to a multiple of RT tiles)
  const int split = blockIdx.y;
  const int t0 = split * tiles_per_split;
  const int t1 = min(ntiles_b, t0 + tiles_per_split);
  const int nt = t1 - t0;

  if (threadIdx.x == 0) {
    mbar_init(bar_a, 4);  // the four lane quarters of the row operands
    for (int s = 0; s < NSTAGE; ++s) {
      mbar_init(&full_b[s], 1);
      mbar_init(&empty_b[s], 1 + NEPI);  // MMA completion + every epilogue warp (it reads the weights)
    }
    for (int a = 0; a < RT; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], NEPI);
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, C::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      for (int k = 0; k < nt; ++k) {
        const int st = k % NSTAGE;
        if (k >= NSTAGE) mbar_wait(&empty_b[st], ((k / NSTAGE) + 1) & 1);
        mbar_arrive_expect_tx(&full_b[st], b_bytes);
        tma_load_1d(sb + st * b_bytes, b_imgs + (int64_t)(t0 + k) * b_bytes, b_bytes, &full_b[st]);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one thread) =====
    if (lane == 0) {
      const uint32_t idesc = make_idesc_f16(kTcM, BN), idesc_r1 = make_idesc_bf16(kTcM, BN);
      const int seg = tc_dk_of_kp(kp) / 8;  // 8-element chunks per split term
      mbar_wait(bar_a, 0);
      tc_fence_after();
      for (int k = 0; k < nt; ++k) {
        const int st = k % NSTAGE;
        mbar_wait(&full_b[st], (k / NSTAGE) & 1);
        const uint32_t b_addr = smem_u32(sb + st * b_bytes);
#pragma unroll
        for (int r = 0; r < RT; ++r) {
          if (k >= 1) mbar_wait(&tmem_empty[r], (k + 1) & 1);
          tc_fence_after();
          const uint32_t a_tmem = tmem_base + C::A_COL0 + r * C::A_COLS;
          const uint32_t d_addr = tmem_base + r * BN;
          // rank-one chunk first (bf16; overwrites the accumulator), then the three fp16 cross products
          {
            const uint64_t db = make_smem_desc(b_addr + kTcTerms * seg * (BN * 16), BN * 16, 128);
            umma_bf16_ts(d_addr, a_tmem + kTcTerms * seg * 4, db, idesc_r1, false);  // 4 TMEM columns per 8 elements
          }
#pragma unroll
          for (int prod = 0; prod < 3; ++prod) {
            // (A term, B term): hh, hl, lh
            const int ta = (prod == 2) ? 1 : 0, tb = (prod == 1) ? 1 : 0;
            for (int kk = 0; kk < seg / 2; ++kk) {
              const uint64_t db = make_smem_desc(b_addr + (tb * seg + 2 * kk) * (BN * 16), BN * 16, 128);
              umma_bf16_ts(d_addr, a_tmem + (ta * seg + 2 * kk) * 4, db, idesc, true);
            }
          }
          umma_commit(&tmem_full[r]);  // accumulator r ready for the epilogue
        }
        umma_commit(&empty_b[st]);  // operand slot consumed by both row tiles
      }
    }
  } else {
    // ===== epilogue: TMEM -> exp2 -> weighted row sums =====
    const int ew = warp - 2;
    const int quarter = warp & 3;              // TMEM lanes this warp may touch: 32*quarter .. +31
    const int half = ew / 4;                   // column share when several warps cover one lane quarter
    constexpr int NH = NEPI / 4;
    constexpr int CW = BN / NH;                // columns per warp per tile
    const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
    if (ew < 4) {
      // stage this CTA's row operands into TMEM once: thread = row (TMEM lane), 16 halves (8 columns) at a time
      for (int r = 0; r < RT; ++r) {
        const unsigned char* src = a_imgs + (int64_t)(row_tile0 + r) * a_bytes + (quarter * 32 + lane) * 16;
        for (int c2 = 0; c2 < kp / 16; ++c2) {
          const uint4 lo = *reinterpret_cast<const uint4*>(src + (int64_t)(2 * c2) * kTcM * 16);
          const uint4 hi = *reinterpret_cast<const uint4*>(src + (int64_t)(2 * c2 + 1) * kTcM * 16);
          const uint32_t v8[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
          tmem_st8(lane_base + C::A_COL0 + r * C::A_COLS + c2 * 8, v8);
        }
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_a);
    }
    float cs = 1.f, cq = 0.f, c2 = 0.f;  // sqrt kernels: extent s, clamp on the scaled d^2, exponent per unit of r
    if constexpr (SQRT) {
      cs = tc_coord_scale(coord_absmax);
      cq = clampq / cs / cs;
      c2 = -kc * cs;
    }
    float acc[RT];                 // MODE 0, 4, 5: weighted sums
    float m[RT], srun[RT];         // MODE 1: running (m, s)
#pragma unroll
    for (int r = 0; r < RT; ++r) {
      acc[r] = 0.f;
      m[r] = kNegBig;
      srun[r] = 0.f;
    }
    for (int k = 0; k < nt; ++k) {
      const int st = k % NSTAGE;
      const float* wts = reinterpret_cast<const float*>(sb + st * b_bytes + BN * kp * 2);
#pragma unroll
      for (int r = 0; r < RT; ++r) {
        mbar_wait(&tmem_full[r], k & 1);
        tc_fence_after();
        float ts0 = 0.f, ts1 = 0.f;
#pragma unroll
        for (int c0 = 0; c0 < CW; c0 += 32) {
          float v[32];
          tmem_ld32(lane_base + r * BN + half * CW + c0, v);
          if constexpr (MODE != 1) {
            if (self_mode) {
              // rows and columns are the SAME cloud (the K_xx / K_yy terms of an MMD): the exponent of the pair
              // (i, i) is -|X_i - X_i|^2/2 = 0 exactly, but the expansion X.X - |X|^2/2 - |X|^2/2 cancels three
              // O(|x/blur|^2) numbers in fp32 (5e-3 at blur = .05, D = 64 — BASELINE configs[2], where the diagonal
              // IS the loss; for the sqrt kernels, r_ii = sqrt(fp32 noise) instead of sqrt(clamp)).  Warp-uniform
              // test, taken on one column tile in N/128.
              const int64_t col0 = (int64_t)(t0 + k) * BN + half * CW + c0;
              const int64_t row_lo = (int64_t)(row_tile0 + r) * kTcM + quarter * 32;
              if (col0 < row_lo + 32 && row_lo < col0 + 32) {
                const int diag = (int)(row_lo + lane - col0);
#pragma unroll
                for (int c = 0; c < 32; ++c)
                  if (c == diag) v[c] = 0.f;
              }
            }
            if constexpr (SQRT) {
#pragma unroll
              for (int c = 0; c < 32; ++c) {
                // d^2 >= cq >= 0; r = d^2 rsqrt(d^2) is 0, not NaN, at d^2 = 0 (unclamped, or the diagonal)
                const float d2 = fmaxf(-2.f * v[c], cq);
                const float r = d2 * rsqrt_approx(fmaxf(d2, 1e-30f));
                v[c] = (MODE == 4) ? ex2_approx(c2 * r) : r;
              }
            } else {
#pragma unroll
              for (int c = 0; c < 32; ++c) v[c] = ex2_approx(v[c]);
            }
            const float4* w4 = reinterpret_cast<const float4*>(wts + half * CW + c0);
#pragma unroll
            for (int c = 0; c < 32; c += 4) {
              const float4 w = w4[c / 4];
              ts0 = fmaf(v[c + 0], w.x, ts0);
              ts1 = fmaf(v[c + 1], w.y, ts1);
              ts0 = fmaf(v[c + 2], w.z, ts0);
              ts1 = fmaf(v[c + 3], w.w, ts1);
            }
          } else {
            float cs0 = 0.f, cs1 = 0.f;
#pragma unroll
            for (int c = 0; c < 32; c += 2) {
              cs0 += ex2_approx(v[c] - m[r]);
              cs1 += ex2_approx(v[c + 1] - m[r]);
            }
            if (!(cs0 + cs1 <= 1.8446744e19f)) {
              // outdated max (a term above 2^64 or an overflow): rebase on this chunk's max and redo it
              float cm = v[0];
#pragma unroll
              for (int c = 1; c < 32; ++c) cm = fmaxf(cm, v[c]);
              const float sc = ex2_approx(m[r] - cm);
              srun[r] *= sc;
              ts0 *= sc;
              ts1 *= sc;
              m[r] = cm;
              cs0 = 0.f;
              cs1 = 0.f;
#pragma unroll
              for (int c = 0; c < 32; c += 2) {
                cs0 += ex2_approx(v[c] - m[r]);
                cs1 += ex2_approx(v[c + 1] - m[r]);
              }
            }
            ts0 += cs0;
            ts1 += cs1;
          }
        }
        if constexpr (MODE != 1) {
          acc[r] += ts0 + ts1;
        } else {
          srun[r] += ts0 + ts1;
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&tmem_empty[r]);
          if (r == RT - 1) mbar_arrive(&empty_b[st]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < RT; ++r) {
      const int64_t row = (int64_t)(row_tile0 + r) * kTcM + quarter * 32 + lane;
      if (row < N) {
        if constexpr (MODE != 1) {
          part[((int64_t)split * NH + half) * N + row] = (MODE == 5) ? cs * acc[r] : acc[r];
        } else {
          reinterpret_cast<float2*>(part)[((int64_t)split * NH + half) * N + row] = make_float2(m[r], srun[r]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, C::TMEM_COLS);
}

}  // namespace b200ot
