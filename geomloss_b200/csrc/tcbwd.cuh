// b200ot — row gradients on the tensor cores, 8 < D <= 64: TWO chained GEMMs per column tile, FlashAttention
// style, both on tcgen05 with every intermediate in TMEM.
//
//   S_ij = X_i.Y_j - |X_i|^2/2 - |Y_j|^2/2 (+ H_j - lse2_i)          GEMM 1 (as in tcconv.cuh: fp16x2 split
//                                                                    operands, three cross products, rank-one chunk)
//   P_ij = 2^S_ij (* w_j)                                            epilogue warps: tcgen05.ld -> MUFU.EX2
//   G_ik = sum_j P_ij Y_jk                                           GEMM 2: A = P (TMEM), B = the SAME column
//                                                                    image read MN-major (K = column index)
//
// Reference semantics: the autograd of gaussian_kernel's matvec (src/geomloss/_legacy/kernel_samples.py:62-68,
// :116-137) and of the softmin (sinkhorn_samples.py:32-71) w.r.t. the row cloud:
//   gaussian:  d/dx_i = go_i * sum_j k_ij w_j (y_j - x_i) / blur^2 ;  softmin: d/dx_i = go_i * (x_i - sum_j p_ij y_j)
// i.e. per row the D+1 sums {sum_j P_ij, sum_j P_ij Y_jk}; the finalize kernels turn them into gradients.
//
// * P is written back IN PLACE over the S accumulator it was computed from (fp32 S -> fp16 hi | fp16 lo of P:
//   a 32-column chunk of S becomes 16 columns of hi and 16 columns of lo), so TMEM holds: two S/P buffers
//   (2 x 128 columns), the row operand X (<= 72), and G (dk <= 64 columns, lives for the whole CTA).
// * P = hi + lo (2 fp16 terms; |P| <= 1: softmax weights, or kernel values times weights normalised to
//   max|w| = 1 by the pack kernel), Y = h + l (the image's two terms): G = hi.h + hi.l + lo.h, error
//   ~2^-22 |P||Y| (+ 6e-8 absolute where P falls into fp16's subnormal range).
// * The column image of tcconv.cuh ([kgroup][column][8 bf16], K-major for GEMM 1) is, read with k = column,
//   exactly the canonical MN-major no-swizzle layout (core matrix = 8 columns x 16 B of one 8-dim group), so
//   GEMM 2 needs no second copy of Y: only a descriptor with b_major = MN, LBO = 128 B (next 8 columns),
//   SBO = BN*16 B (next 8 dims).
// * MMA issue order S(0) S(1) G(0) S(2) G(1) ...: the tensor pipe always has the next tile's S to chew on while
//   the epilogue warps turn S(k) into P(k); the in-order pipe makes "S(k+2) overwrites buffer k%2 after G(k)
//   has read it" free of extra barriers.
#pragma once
#include "tcconv.cuh"

namespace b200ot {

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
      "%15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// (lo, hi) fp32 -> packed f16x2, round to nearest even; element `lo` in bits 0..15
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float2 unpack_f16x2(uint32_t v) {
  return __half22float2(*reinterpret_cast<const __half2*>(&v));
}

// fp16 x fp16 -> fp32, A K-major (TMEM), B MN-major
__host__ __device__ constexpr uint32_t make_idesc_f16_bmn(int M, int N) { return make_idesc_f16(M, N) | (1u << 16); }

// MODE 2: gaussian row gradient (P = w_j 2^S), MODE 3: softmin row gradient (P = 2^(S - lse2_i): lse2 rides in the
// row operand's rank-one chunk).  part[(split*N + row)*(D+1) + {0, 1+k}] = sum_j P_ij {1, Y_jk}
//
// PT = fp16 terms of P fed to GEMM 2.  PT = 2: P = hi + lo, products hi.h, hi.l, lo.h (error ~2^-22 |P||Y|).
// PT = 1: P = hi only, products hi.h, hi.l — a third less GEMM-2 work and no lo split / second tcgen05.st in the
// epilogue.  Every weight is then perturbed by <= 2^-12 relative (round to nearest, unbiased); the row sum of P is
// taken over the SAME rounded values, so the gradient (sum_j P_ij Y_j) - X_i (sum_j P_ij) = sum_j hi_ij (Y_j - X_i)
// stays a combination of exact differences — the perturbation never meets the cancellation between the two sums.
//
// MERGE: GEMM 2's hi.h and hi.l products are one N = 2 dk instruction per K step (G occupies 2 dk <= 128 columns,
// 384..511), the halves are added at read-back: 16 instead of 24 instructions and TMEM reads of P per tile.
//
// LDALL (8 epilogue warps: a warp owns 64 columns of a tile): the two 32-column chunks come from one
// tcgen05.ld.x64 instead of two x32 round trips.
//
// MODE 4 / 5: laplacian / energy row gradient.  d/dx_i sum_j w_j k(r_ij) = sum_j w_j k'(r_ij)/r_ij (x_i - y_j), so
// P_ij = w_j k'(r)/r makes the same (N, D+1) sums as MODE 2.  With X = (x - c)/s (|X| <= 1, tc_pack_kernel's
// coord_absmax) and r in units of s, the kernel feeds GEMM 2 with
//   P_ij = w_j min(1/r_ij, 1/rho) (* 2^(-kc s r_ij), laplacian)      rho = kTcSqrtRho
// and the negative factor -1 (energy) or -1/blur (laplacian) goes into the finalize's coefficient; the 1/s of 1/r
// and the s of (x_i - y_j) cancel.  P <= 1/rho = 2^14 (fp16 range) and the typical pair (r ~ 1) is in fp16's normal
// range.  Pairs with r < rho (2^-14 of the extent of the clouds: far below the ~1e-3 to which the fp32 expansion
// resolves r near 0) count with weight 1/rho instead of 1/r.  Pairs inside the clamp (-2 S <= clampq / s^2: the
// reference's clamp_min, pykeops' zero gradient at r = 0) contribute exactly zero.
//
// self_mode: rows and columns are the same cloud (the K_xx term): the exponent of pair (i, i) is exactly 0, as in
// tc_reduce_kernel — matters when sum_j P_ij is used as the forward VALUE (b200ot_kernel_conv_fwd_bwd_x).
constexpr float kTcSqrtRho = 1.0f / 16384.0f;

template <class C, int MODE, int PT, bool LDALL, bool MERGE>
__global__ void __launch_bounds__(C::THREADS, 1)
    tc_bwd_kernel(const unsigned char* __restrict__ a_imgs, const unsigned char* __restrict__ b_imgs,
                  float* __restrict__ part, int64_t N, int kp, int ntiles_b, int tiles_per_split, int NSTAGE, int D,
                  int self_mode, float kc = 0.f, float clampq = 0.f,
                  const float* __restrict__ coord_absmax = nullptr) {
  static_assert(PT == 1 || PT == 2, "P is fed to GEMM 2 as one or two fp16 terms");
  static_assert(MODE >= 2 && MODE <= 5, "forward reductions live in tcconv.cuh");
  constexpr bool SQRT = MODE >= 4;
  constexpr int BN = C::BN, NEPI = C::NEPI, NACC = 2;
  static_assert(BN == 128 && (NEPI == 8 || NEPI == 16), "layout below assumes 128-column tiles, 8 or 16 epilogue warps");
  constexpr int NH = NEPI / 4;   // warps per TMEM lane quarter = column shares of a tile
  constexpr int CW = BN / NH;    // columns per warp per tile (64 or 32)
  constexpr int A_COL0 = NACC * BN;   // row operand X behind the two S/P buffers
  constexpr int G_COL0 = 384;         // gradient accumulator (dk <= 64 columns; MERGE: 2 dk <= 128)
  extern __shared__ __align__(1024) unsigned char smem[];
  const int a_bytes = kTcM * kp * 2;
  const int dk = tc_dk_of_kp(kp);
  const int b_bytes = BN * kp * 2 + BN * 4;
  unsigned char* sb = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NSTAGE * b_bytes);
  uint64_t* bar_a = bars;
  uint64_t* full_b = bars + 1;
  uint64_t* empty_b = full_b + kTcMaxStage;
  uint64_t* s_full = empty_b + kTcMaxStage;   // S(k) accumulated
  uint64_t* p_ready = s_full + NACC;          // P(k) written by all epilogue warps
  uint64_t* g_done = p_ready + NACC;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(g_done + 1);
  float* sp_x = reinterpret_cast<float*>(tmem_slot + 2);  // [NH-1][128] sum_j P of the other column shares

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row_tile = blockIdx.x;
  const int split = blockIdx.y;
  const int t0 = split * tiles_per_split;
  const int t1 = min(ntiles_b, t0 + tiles_per_split);
  const int nt = t1 - t0;

  if (threadIdx.x == 0) {
    mbar_init(bar_a, 4);
    for (int s = 0; s < NSTAGE; ++s) {
      mbar_init(&full_b[s], 1);
      mbar_init(&empty_b[s], 1);  // released by the commit behind GEMM 2 of the tile
    }
    for (int a = 0; a < NACC; ++a) {
      mbar_init(&s_full[a], 1);
      mbar_init(&p_ready[a], NEPI);
    }
    mbar_init(g_done, 1);
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
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
      const uint32_t idesc_s = make_idesc_f16(kTcM, BN), idesc_r1 = make_idesc_bf16(kTcM, BN);
      const uint32_t idesc_g = make_idesc_f16_bmn(kTcM, dk);
      const uint32_t idesc_g2 = make_idesc_f16_bmn(kTcM, 2 * dk);  // MERGE: hi x [Y_h | Y_l]
      const int seg = dk / 8;  // 8-element chunks per split term
      const uint32_t a_tmem = tmem_base + A_COL0, g_tmem = tmem_base + G_COL0;
      mbar_wait(bar_a, 0);
      tc_fence_after();
      for (int k = 0; k <= nt; ++k) {
        if (k < nt) {
          // ---- GEMM 1: S(k) -> buffer k%2 ----
          const int st = k % NSTAGE, acc = k % NACC;
          mbar_wait(&full_b[st], (k / NSTAGE) & 1);
          tc_fence_after();
          const uint32_t b_addr = smem_u32(sb + st * b_bytes);
          const uint32_t d_addr = tmem_base + acc * BN;
          {
            const uint64_t db = make_smem_desc(b_addr + kTcTerms * seg * (BN * 16), BN * 16, 128);
            umma_bf16_ts(d_addr, a_tmem + kTcTerms * seg * 4, db, idesc_r1, false);
          }
#pragma unroll
          for (int prod = 0; prod < 3; ++prod) {
            const int ta = (prod == 2) ? 1 : 0, tb = (prod == 1) ? 1 : 0;  // hh, hl, lh
            for (int kk = 0; kk < seg / 2; ++kk) {
              const uint64_t db = make_smem_desc(b_addr + (tb * seg + 2 * kk) * (BN * 16), BN * 16, 128);
              umma_bf16_ts(d_addr, a_tmem + (ta * seg + 2 * kk) * 4, db, idesc_s, true);
            }
          }
          umma_commit(&s_full[acc]);
        }
        if (k >= 1) {
          // ---- GEMM 2: G += P(k-1) . Y(k-1), K = the 128 columns of the tile, 16 per instruction ----
          const int j = k - 1, st = j % NSTAGE, acc = j % NACC;
          mbar_wait(&p_ready[acc], (j / NACC) & 1);
          tc_fence_after();
          const uint32_t b_addr = smem_u32(sb + st * b_bytes);
          const uint32_t p_tmem = tmem_base + acc * BN;
          if constexpr (MERGE) {
            // the l term of Y follows its h term in the image (8-dim groups 0..seg-1 = h, seg..2 seg-1 = l, one
            // stride): ONE instruction with N = 2 dk multiplies hi by [Y_h | Y_l] into [G_a | G_b] — the same tensor
            // work as two N = dk instructions, but P is read from TMEM once instead of twice
#pragma unroll
            for (int kk = 0; kk < BN / 16; ++kk) {
              const uint32_t pa = p_tmem + 32 * (kk >> 1) + 8 * (kk & 1);
              const uint64_t db = make_smem_desc(b_addr + (2 * kk) * 128, 128, BN * 16);
              umma_bf16_ts(g_tmem, pa, db, idesc_g2, !(j == 0 && kk == 0));
            }
            if constexpr (PT == 2) {
#pragma unroll
              for (int kk = 0; kk < BN / 16; ++kk) {  // lo . Y_h -> G_a
                const uint32_t pa = p_tmem + 32 * (kk >> 1) + 8 * (kk & 1) + 16;
                const uint64_t db = make_smem_desc(b_addr + (2 * kk) * 128, 128, BN * 16);
                umma_bf16_ts(g_tmem, pa, db, idesc_g, true);
              }
            }
          } else {
#pragma unroll
            for (int prod = 0; prod < PT + 1; ++prod) {
              // (P term, Y term): hi.h, hi.l, lo.h (the last one only when P carries its lo term)
              const int tp = (prod == 2) ? 1 : 0, ty = (prod == 1) ? 1 : 0;
#pragma unroll
              for (int kk = 0; kk < BN / 16; ++kk) {
                // columns 16kk..16kk+15 of the tile: 32-column chunk kk/2, half kk%2; hi at +0, lo at +16
                const uint32_t pa = p_tmem + 32 * (kk >> 1) + 8 * (kk & 1) + 16 * tp;
                const uint64_t db = make_smem_desc(b_addr + ty * seg * (BN * 16) + (2 * kk) * 128, 128, BN * 16);
                umma_bf16_ts(g_tmem, pa, db, idesc_g, !(j == 0 && prod == 0 && kk == 0));
              }
            }
          }
          umma_commit(&empty_b[st]);  // the column tile may be overwritten once GEMM 2 has read it
        }
      }
      umma_commit(g_done);
    }
  } else {
    // ===== epilogue warps: S -> P (in place), row sums of P =====
    const int ew = warp - 2;
    const int quarter = warp & 3;  // TMEM lanes 32*quarter .. +31
    const int half = ew / 4;       // column share: columns CW*half .. +CW-1 of every tile
    const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const int64_t row = (int64_t)row_tile * kTcM + quarter * 32 + lane;
    if (ew < 4) {
      const unsigned char* src = a_imgs + (int64_t)row_tile * a_bytes + (quarter * 32 + lane) * 16;
      for (int c2 = 0; c2 < kp / 16; ++c2) {
        const uint4 lo = *reinterpret_cast<const uint4*>(src + (int64_t)(2 * c2) * kTcM * 16);
        const uint4 hi = *reinterpret_cast<const uint4*>(src + (int64_t)(2 * c2 + 1) * kTcM * 16);
        const uint32_t r[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
        tmem_st8(lane_base + A_COL0 + c2 * 8, r);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_a);
    }
    float cq = 0.f, c2 = 0.f;  // sqrt kernels: clamp on the scaled d^2, exponent per unit of r
    if constexpr (SQRT) {
      const float cs = tc_coord_scale(coord_absmax);
      cq = clampq / cs / cs;
      c2 = -kc * cs;
    }
    float sum0 = 0.f, sum1 = 0.f;
    for (int k = 0; k < nt; ++k) {
      const int st = k % NSTAGE, acc = k % NACC;
      mbar_wait(&s_full[acc], (k / NACC) & 1);
      tc_fence_after();
      const float* wts = reinterpret_cast<const float*>(sb + st * b_bytes + BN * kp * 2);
      // one 32-column chunk of S -> P, in place; v = the chunk's exponents (registers)
      auto chunk = [&](float* v, const int col0) {
        if constexpr (MODE != 3) {
          if (self_mode) {
            // warp-uniform: does this 32-column chunk meet the diagonal of this warp's 32 rows?
            const int64_t gcol0 = (int64_t)(t0 + k) * BN + col0;
            const int64_t row_lo = (int64_t)row_tile * kTcM + quarter * 32;
            if (gcol0 < row_lo + 32 && row_lo < gcol0 + 32) {
              const int diag = (int)(row_lo + lane - gcol0);
#pragma unroll
              for (int c = 0; c < 32; ++c)
                if (c == diag) v[c] = 0.f;
            }
          }
        }
        uint32_t ph[16], pl[16];
        float cs0 = 0.f, cs1 = 0.f;  // per-chunk sums (two-level accumulation, like the forward kernel's per-tile sums)
#pragma unroll
        for (int c = 0; c < 32; c += 2) {
          float p0, p1;
          if constexpr (SQRT) {
            const float d0 = -2.f * v[c], d1 = -2.f * v[c + 1];
            const float q0 = rsqrt_approx(fmaxf(d0, kTcSqrtRho * kTcSqrtRho));  // min(1/r, 1/rho)
            const float q1 = rsqrt_approx(fmaxf(d1, kTcSqrtRho * kTcSqrtRho));
            p0 = q0;
            p1 = q1;
            if constexpr (MODE == 4) {
              p0 *= ex2_approx(c2 * (d0 * q0));  // r = d^2 min(1/r, 1/rho): exact for r >= rho
              p1 *= ex2_approx(c2 * (d1 * q1));
            }
            // (selected after the exponential: at d^2 < 0 (rounding) it may overflow)
            p0 = d0 > cq ? p0 : 0.f;
            p1 = d1 > cq ? p1 : 0.f;
          } else {
            p0 = ex2_approx(v[c]);
            p1 = ex2_approx(v[c + 1]);
          }
          if constexpr (MODE != 3) {
            const float2 w = *reinterpret_cast<const float2*>(wts + col0 + c);
            p0 *= w.x;
            p1 *= w.y;
          }
          const uint32_t h = pack_f16x2(p0, p1);
          ph[c / 2] = h;
          if constexpr (PT == 2) {
            cs0 += p0;
            cs1 += p1;
            const float2 hf = unpack_f16x2(h);
            pl[c / 2] = pack_f16x2(p0 - hf.x, p1 - hf.y);
          } else {
            const float2 hf = unpack_f16x2(h);  // the sums see exactly what GEMM 2 sees
            cs0 += hf.x;
            cs1 += hf.y;
          }
        }
        sum0 += cs0;
        sum1 += cs1;
        tmem_st16(lane_base + acc * BN + col0, ph);
        if constexpr (PT == 2) tmem_st16(lane_base + acc * BN + col0 + 16, pl);
      };
      if constexpr (LDALL && CW == 64) {
        // both chunks of this warp's 64 columns in ONE tcgen05.ld: one TMEM round trip per tile instead of two
        float vv[64];
        tmem_ld64(lane_base + acc * BN + half * CW, vv);
        chunk(&vv[0], half * CW);
        chunk(&vv[32], half * CW + 32);
      } else {
#pragma unroll
        for (int c0 = 0; c0 < CW; c0 += 32) {
          float v[32];
          tmem_ld32(lane_base + acc * BN + half * CW + c0, v);
          chunk(v, half * CW + c0);
        }
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_ready[acc]);
    }
    // ---- G is complete once every MMA has retired: read it back, add the row sums of the two halves ----
    if (half >= 1) sp_x[(half - 1) * 128 + quarter * 32 + lane] = sum0 + sum1;
    asm volatile("bar.sync 1, %0;" ::"r"(32 * NEPI) : "memory");
    mbar_wait(g_done, 0);
    tc_fence_after();
    if (half * 32 < dk) {
      float g[32];
      tmem_ld32(lane_base + G_COL0 + half * 32, g);
      if constexpr (MERGE) {
        float gb[32];  // G_b = hi . Y_l lives dk columns further
        tmem_ld32(lane_base + G_COL0 + dk + half * 32, gb);
#pragma unroll
        for (int c = 0; c < 32; ++c) g[c] += gb[c];
      }
      if (row < N) {
        float* dst = part + ((int64_t)split * N + row) * (D + 1);
        if (half == 0) {
          float tot = sum0 + sum1;
#pragma unroll
          for (int h2 = 1; h2 < NH; ++h2) tot += sp_x[(h2 - 1) * 128 + quarter * 32 + lane];
          dst[0] = tot;
        }
#pragma unroll
        for (int c = 0; c < 32; ++c)
          if (half * 32 + c < D) dst[1 + half * 32 + c] = g[c];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

}  // namespace b200ot
