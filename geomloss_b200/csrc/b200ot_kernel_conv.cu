// b200ot — kernel convolutions  out_i = sum_j k(x_i, y_j) w_j  and their row gradients.
// Reference semantics: the matvecs of kernel_loss (src/geomloss/_legacy/kernel_samples.py:116-137) with
//   gaussian  k = exp(-|x/s - y/s|^2 / 2)                    (kernel_samples.py:62-68)
//   laplacian k = exp(-sqrt(max(|x/s - y/s|^2, 1e-8)))       (kernel_samples.py:71-77, utils.py:56-61)
//   energy    k = -sqrt(max(|x - y|^2, 1e-8))                (kernel_samples.py:80-82)
// evaluated on the fly (never as an N x M matrix) by rowsum_partial_kernel.
#include "b200ot.h"
#include "host_util.cuh"
#include "pack.cuh"
#include "plan.cuh"
#include "rowsum.cuh"
#include "rowsum_launch.cuh"
#include "tcbwd.cuh"
#include "tcconv.cuh"

#include <stdio.h>
#include <stdlib.h>

#include <type_traits>

namespace b200ot {

struct ConvScales {
  float scale;   // coordinate scale
  float clampq;  // clamp on the scaled squared distance
  int direct;
  int extra;
};

// `kind` may carry B200OT_KERNEL_UNCLAMPED (laplacian / energy with pykeops' unclamped sqrt)
static int kind_base(int kind) { return kind & 0xff; }
static bool valid_kind(int kind) {
  return kind_base(kind) >= 0 && kind_base(kind) <= 2 && (kind & ~(0xff | B200OT_KERNEL_UNCLAMPED)) == 0;
}

static ConvScales conv_scales(int kind_flags, float blur) {
  ConvScales c;
  const int kind = kind_base(kind_flags);
  const float clamp = cost_clamp(kind_flags);  // B200OT_KERNEL_UNCLAMPED == B200OT_P_UNCLAMPED
  if (kind == B200OT_KERNEL_GAUSSIAN) {
    c.scale = sqrtf(kLog2e) / blur;  // 2^(-|X-Y|^2/2) = exp(-|x-y|^2 / (2 blur^2))
    c.clampq = 0.f;
    c.direct = 0;
    c.extra = 2;
  } else if (kind == B200OT_KERNEL_LAPLACIAN) {
    c.scale = kLog2e / blur;  // 2^(-|X-Y|) = exp(-|x-y| / blur)
    c.clampq = kLog2e * kLog2e * clamp;
    c.direct = 1;
    c.extra = 1;
  } else {
    c.scale = 1.f;
    c.clampq = clamp;
    c.direct = 1;
    c.extra = 1;
  }
  return c;
}

__global__ void conv_fwd_finalize_kernel(const float* __restrict__ part, int n_split, float sign,
                                         float* __restrict__ out, int64_t N) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  float a = 0.f;
  for (int s = 0; s < n_split; ++s) a += part[(int64_t)s * N + i];
  out[i] = sign * a;
}

// gaussian: part (n_split, N, D+1): [0] = sum W e, [1+k] = sum W e Y_k   -> go (accY - X acc0) / (scale blur^2)
// laplacian / energy: part (n_split, N, D): sum W e u_k                    -> -go acc / blur   (energy: -go acc)
// laplacian / energy on the tensor cores (coord_absmax != null): part (n_split, N, D+1) as for the gaussian, with
//   X = (x - c) / s and P = w k'(r)/r up to the factor -coef (tcbwd.cuh, MODE 4 / 5)     -> go coef (accY - X acc0)
__global__ void conv_bwd_finalize_kernel(const float* __restrict__ part, int n_split, const float* __restrict__ x,
                                         const float* __restrict__ center, const float* __restrict__ grad_out,
                                         float* __restrict__ grad_x, int64_t N, int D, int kind, float scale,
                                         float coef, const float* __restrict__ w_absmax,
                                         float* __restrict__ value_out = nullptr,
                                         const float* __restrict__ coord_absmax = nullptr) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  if (coord_absmax != nullptr) scale = tc_coord_inv(coord_absmax);
  float go = grad_out ? grad_out[i] : 1.f;  // no upstream gradient: the unit row gradient (value + gradient pass)
  float wmax = 1.f;
  if (w_absmax != nullptr && *w_absmax > 0.f) wmax = *w_absmax;  // tensor-core path: weights were normalised
  go *= wmax;
  if (kind == B200OT_KERNEL_GAUSSIAN || coord_absmax != nullptr) {
    const int na = D + 1;
    float a0 = 0.f;
    for (int s = 0; s < n_split; ++s) a0 += part[((int64_t)s * N + i) * na];
    if (value_out) value_out[i] = wmax * a0;  // sum_j w_j k_ij: the forward value comes with the gradient sums
    for (int k = 0; k < D; ++k) {
      float a = 0.f;
      for (int s = 0; s < n_split; ++s) a += part[((int64_t)s * N + i) * na + 1 + k];
      const float c = center ? center[k] : 0.f;
      const float X = scale * (x[i * D + k] - c);
      grad_x[i * D + k] = go * coef * (a - X * a0);
    }
  } else {
    for (int k = 0; k < D; ++k) {
      float a = 0.f;
      for (int s = 0; s < n_split; ++s) a += part[((int64_t)s * N + i) * D + k];
      grad_x[i * D + k] = go * coef * a;
    }
  }
}

// max_j |w_j| into *out (zero-initialised by the caller); bit order of non-negative floats = integer order
__global__ void absmax_kernel(const float* __restrict__ w, int64_t n, float* __restrict__ out) {
  float m = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(w[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f && !(m != m)) atomicMax(reinterpret_cast<unsigned int*>(out), __float_as_uint(m));
}

// max_k |x_ik - c_k| over the rows of x:(n, D) and y:(m, D) into *out (zero-initialised by the caller): the coordinate
// scale s of the tensor-core laplacian / energy kernels (tcconv.cuh: tc_coord_scale)
__global__ void coord_absmax_kernel(const float* __restrict__ x, int64_t n, const float* __restrict__ y, int64_t m,
                                    int D, const float* __restrict__ center, float* __restrict__ out) {
  float v = 0.f;
  const int64_t nx = n * D, total = nx + m * D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const float p = i < nx ? x[i] : y[i - nx];
    v = fmaxf(v, fabsf(p - (center ? center[i % D] : 0.f)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  if ((threadIdx.x & 31) == 0 && v > 0.f) atomicMax(reinterpret_cast<unsigned int*>(out), __float_as_uint(v));
}

template <int MODE, int D>
static int launch_rowsum(const ReducePlan& pl, cudaStream_t st, const float* x, const float* center, float scale,
                         float clampq, const float* cols, float* part, int64_t N, const int4* seg = nullptr,
                         const int2* pieces = nullptr) {
  if (pl.small) {
    using C = RowSumCfg<MODE, D, kSmallR, kSmallNT, kSmallTJ, 3, 4>;
    return launch_rowsum_kernel<C>(pl, st, x, center, scale, clampq, cols,
                            (const float*)nullptr, part, N, pl.ntiles, pl.tiles_per_split, seg, pieces);
  }
  // D >= 5: one row per thread (same 512 rows per CTA) keeps the 2 x (D+1) accumulator pairs in registers
  using C = std::conditional_t<(D <= 4), RowSumCfg<MODE, D, kBigR, kBigNT, kBigTJ, 3, 2>,
                               RowSumCfg<MODE, D, 1, kBigR * kBigNT, kBigTJ, 3, 1>>;
  return launch_rowsum_kernel<C>(pl, st, x, center, scale, clampq, cols, (const float*)nullptr,
                          part, N, pl.ntiles, pl.tiles_per_split, seg, pieces);
}

template <int MODE>
static int launch_rowsum_d(int D, const ReducePlan& pl, cudaStream_t st, const float* x, const float* center,
                           float scale, float clampq, const float* cols, float* part, int64_t N,
                           const int4* seg = nullptr, const int2* pieces = nullptr) {
  switch (D) {
    case 1: return launch_rowsum<MODE, 1>(pl, st, x, center, scale, clampq, cols, part, N, seg, pieces);
    case 2: return launch_rowsum<MODE, 2>(pl, st, x, center, scale, clampq, cols, part, N, seg, pieces);
    case 3: return launch_rowsum<MODE, 3>(pl, st, x, center, scale, clampq, cols, part, N, seg, pieces);
    case 4: return launch_rowsum<MODE, 4>(pl, st, x, center, scale, clampq, cols, part, N, seg, pieces);
    case 5: return launch_rowsum<MODE, 5>(pl, st, x, center, scale, clampq, cols, part, N, seg, pieces);
    case 6: return launch_rowsum<MODE, 6>(pl, st, x, center, scale, clampq, cols, part, N, seg, pieces);
    case 7: return launch_rowsum<MODE, 7>(pl, st, x, center, scale, clampq, cols, part, N, seg, pieces);
    case 8: return launch_rowsum<MODE, 8>(pl, st, x, center, scale, clampq, cols, part, N, seg, pieces);
    default: return B200OT_EINVAL;
  }
}

static int conv_pack(const float* y, const float* w, const float* center, int64_t M, int D, const ConvScales& cs,
                     float* cols, cudaStream_t st, const int* src = nullptr) {
  const int nf2 = colfmt_nf2(D, cs.extra);
  const int64_t mpad = round_up64(M, kPackPad);
  const int threads = 256;
  pack_cols_kernel<<<(unsigned)ceil_div64(mpad, threads), threads, 0, st>>>(
      y, nullptr, nullptr, 0.f, 0.f, w, center, cs.scale, cs.direct, D, nf2, M, mpad, cols, src);
  B200OT_CUDA_TRY(cudaGetLastError());
  return B200OT_OK;
}

// the N x M launch of a CUDA-core kernel convolution (dense plan, or ranges when seg != null)
static int conv_partial(int kind_flags, bool bwd, const ReducePlan& pl, cudaStream_t st, const float* x,
                        const float* center, const ConvScales& cs, const float* cols, float* part, int64_t N, int D,
                        const int4* seg = nullptr, const int2* pieces = nullptr) {
  const int kind = kind_base(kind_flags);
  if (kind == B200OT_KERNEL_GAUSSIAN)
    return bwd ? launch_rowsum_d<kGaussBwd>(D, pl, st, x, center, cs.scale, cs.clampq, cols, part, N, seg, pieces)
               : launch_rowsum_d<kGaussFwd>(D, pl, st, x, center, cs.scale, cs.clampq, cols, part, N, seg, pieces);
  if (kind == B200OT_KERNEL_LAPLACIAN)
    return bwd ? launch_rowsum_d<kLaplaceBwd>(D, pl, st, x, center, cs.scale, cs.clampq, cols, part, N, seg, pieces)
               : launch_rowsum_d<kLaplaceFwd>(D, pl, st, x, center, cs.scale, cs.clampq, cols, part, N, seg, pieces);
  return bwd ? launch_rowsum_d<kEnergyBwd>(D, pl, st, x, center, cs.scale, cs.clampq, cols, part, N, seg, pieces)
             : launch_rowsum_d<kEnergyFwd>(D, pl, st, x, center, cs.scale, cs.clampq, cols, part, N, seg, pieces);
}

static float conv_bwd_coef(int kind_flags, const ConvScales& cs, float blur) {
  const int kind = kind_base(kind_flags);
  if (kind == B200OT_KERNEL_GAUSSIAN) return 1.0f / (cs.scale * blur * blur);
  if (kind == B200OT_KERNEL_LAPLACIAN) return -1.0f / blur;
  return -1.0f;
}

// ---------------------------------------------------------------------------------------------------
// tensor-core path (gaussian; laplacian / energy above B200OT_MAX_D), 8 < D <= 64: see tcconv.cuh
// ---------------------------------------------------------------------------------------------------
constexpr int kTcBN = 128;    // columns per MMA tile
constexpr int kTcEpi = 16;    // epilogue warps of the forward kernels: 4 per TMEM lane quarter hide the tcgen05.ld latency
using TcConvCfg = TcCfg<kTcBN, kTcEpi>;
using TcBwdCfg = TcCfg<kTcBN, 8>;  // (16 epilogue warps measured no faster with PT = 2: 0.453 s vs 0.441 s on the D=64 MMD)
using TcBwdCfg16 = TcCfg<kTcBN, 16>;

struct TcPlan {
  int kp, nstage, n_split, tiles_per_split;
  int64_t a_tiles, a_tiles_pad, b_tiles, a_bytes, b_bytes, smem;
  int64_t off_b, off_part, off_misc, total;
};

// Which path serves an operator.  Above B200OT_MAX_D the tensor-core kernels are the only ones.  At or below it both
// exist: the CUDA-core kernels are FMA-pipe bound from D = 5 up while the tensor-core kernels run the zero-padded
// dk = 16 problem at the same rate whatever D.  Measured on B200 at N = M = 4e5 (tools/ab_tc_route.py,
// profiles/r02_ab_tc_route.jsonl; CUDA-core -> tensor-core, 1e12 pairs/s):
//   softmin forward   D = 5: 3.36 -> 3.38   D = 6: 2.99 -> 3.32   D = 7: 2.69 -> 3.29   D = 8: 2.13 -> 3.26
//   gaussian forward  D = 4: 3.93 -> 3.58   D = 5: 2.58 -> 3.58   D = 6: 2.27 -> 3.58   D = 8: 1.82 -> 3.58
//   row gradients     D = 7: 1.60 / 1.48 -> 1.54 / 1.46 (softmin / gaussian); D = 8: 1.33 / 1.36 -> 1.54 / 1.46
// (the same ratios at N = M = 1e5 and 3e4).  The forward operators switch at D = 6 (softmin) and D = 5 (gaussian).  The
// row gradients stay on the CUDA cores for every D <= 8: the gain is 8-16 % at D = 8 only, and the fp16 image of P that
// GEMM 2 consumes costs accuracy at small blur in low dimension (relative difference between the two paths' gradients at
// blur = .05: 3e-3 at D = 4, 5e-4 at D = 6, 6e-5 at D = 8).  Problems below 8e8 pairs keep the CUDA-core kernels (the
// cross-over was measured down to N = M = 3e4).  $B200OT_TC_MIN_D ("d" or "softmin_fwd,softmin_bwd,conv_fwd,conv_bwd")
// and $B200OT_TC_MIN_PAIRS override the defaults for A/B timing and for the parity tests of both routes — read on every
// call, never set by the bench.
static const int kTcMinDimDefault[4] = {6, 9, 5, 9};
static const double kTcMinPairsDefault = 8.0e8;

bool tc_routed(int op, int D, int64_t N, int64_t M) {
  if (!tc_capable_dim(D)) return false;
  if (D > B200OT_MAX_D) return true;
  int min_dim[4] = {kTcMinDimDefault[0], kTcMinDimDefault[1], kTcMinDimDefault[2], kTcMinDimDefault[3]};
  double min_pairs = kTcMinPairsDefault;
  if (const char* e = getenv("B200OT_TC_MIN_D")) {
    int v[4];
    const int n = sscanf(e, "%d,%d,%d,%d", &v[0], &v[1], &v[2], &v[3]);
    if (n == 1) {
      for (int k = 0; k < 4; ++k) min_dim[k] = v[0];
    } else if (n == 4) {
      for (int k = 0; k < 4; ++k) min_dim[k] = v[k];
    }
  }
  if (const char* e = getenv("B200OT_TC_MIN_PAIRS")) {
    const double v = atof(e);
    if (v >= 0.0) min_pairs = v;
  }
  return D >= min_dim[op] && (double)N * (double)M >= min_pairs;
}

bool tc_any_routed(int D, int64_t N, int64_t M) {
  for (int op = 0; op < 4; ++op)
    if (tc_routed(op, D, N, M)) return true;
  return false;
}

// Tuning of the row-gradient kernels (tcbwd.cuh): fp16 terms of P in GEMM 2 (PT), epilogue warps, one tcgen05.ld.x64
// per tile (LDALL), hi.[Y_h | Y_l] as one N = 2 dk instruction (MERGE).  Measured on B200, gaussian row gradients at
// N = M = 4e5, D = 64 / D = 16, ms per reduction (tools/ab_tc_route.py, profiles/r02_ab_tc_route.jsonl):
//   "2,8,0,0" 130.2 / 109.5   "2,8,0,1" 118.0 / 91.0 (shipped)   "2,8,1,0" 130.7 / 110.0   "2,16,0,0" 137.1 / 116.3
//   "2,16,0,1" 120.8 / 97.9   "1,8,0,0" 110.8 / 89.6             "1,8,0,1" 101.9 / 75.2    "1,16,0,1" 105.7 / 82.7
// MERGE is accuracy-neutral (same products, same fp32 accumulation) and ships.  PT = 1 is another 14-17 % but feeds GEMM 2
// an 11-bit image of P whose subnormal flush also reaches the row sums — kept as a knob, not the default.
// $B200OT_TC_BWD ("p_terms,epi,ldall,merge") overrides the default for A/B timing and the variants' parity tests.
struct TcBwdTuning {
  int p_terms, epi, ldall, merge;
};
static const TcBwdTuning kTcBwdDefault = {2, 8, 0, 1};
static TcBwdTuning tc_bwd_tuning() {
  TcBwdTuning t = kTcBwdDefault;
  if (const char* e = getenv("B200OT_TC_BWD")) {
    int a, b, c, d;
    if (sscanf(e, "%d,%d,%d,%d", &a, &b, &c, &d) == 4 && (a == 1 || a == 2) && (b == 8 || b == 16) &&
        (c == 0 || c == 1) && (d == 0 || d == 1)) {
      t.p_terms = a;
      t.epi = b;
      t.ldall = c;
      t.merge = d;
    }
  }
  return t;
}

static TcPlan make_tc_plan(int64_t N, int64_t M, int D, bool bwd = false) {
  TcPlan p;
  p.kp = tc_kp(D);
  p.a_tiles = ceil_div64(N, kTcM);
  p.a_tiles_pad = ceil_div64(p.a_tiles, kTcRT) * kTcRT;  // forward CTAs own kTcRT row tiles
  p.b_tiles = ceil_div64(M, kTcBN);
  p.a_bytes = tc_a_img_bytes(p.kp);
  p.b_bytes = tc_b_img_bytes(p.kp, kTcBN);
  const int64_t bar_bytes = 2048;  // mbarriers, the TMEM slot, (backward) 3 x 128 floats of row-sum exchange
  const int64_t avail = 227 * 1024 - bar_bytes - 1024;  // the row operand lives in TMEM, not in shared memory
  int64_t ns = avail / p.b_bytes;
  p.nstage = (int)(ns > kTcMaxStage ? kTcMaxStage : ns);
  p.smem = p.nstage * p.b_bytes + bar_bytes;
  int64_t want = ceil_div64((int64_t)num_sms() * 4, bwd ? p.a_tiles : p.a_tiles_pad / kTcRT);
  if (want < 1) want = 1;
  if (want > 64) want = 64;
  if (want > p.b_tiles) want = p.b_tiles;
  p.tiles_per_split = (int)ceil_div64(p.b_tiles, want);
  p.n_split = (int)ceil_div64(p.b_tiles, p.tiles_per_split);
  p.off_b = round_up64(p.a_tiles_pad * p.a_bytes, 256);
  p.off_part = p.off_b + round_up64(p.b_tiles * p.b_bytes, 256);
  // partials: (m, s) pairs forward, D+1 sums per row backward
  p.off_misc = p.off_part + round_up64((int64_t)p.n_split * (kTcEpi / 4) * N * 4 * (bwd ? D + 1 : 2), 256);
  p.total = p.off_misc + 256;  // [0]: max|w| of the row-gradient pass
  return p;
}

int64_t tc_scratch_bytes(int64_t N, int64_t M, int D) {
  // forward and row-gradient launches split the columns differently: size for the larger of the two
  return std::max(make_tc_plan(N, M, D, false).total, make_tc_plan(N, M, D, true).total);
}

// Laplacian / energy on the tensor cores (tcconv.cuh / tcbwd.cuh, MODE 4 / 5): the exponent factor per unit of
// distance and the clamp on |x - y|^2 in the units of x.  The pykeops convention (UNCLAMPED) clamps at exactly 0:
// r = 0 and a zero gradient at coincident points.
struct TcSqrtParams {
  float kc, clampq;
};
static TcSqrtParams tc_sqrt_params(int kind_flags, float blur) {
  const float clamp = (kind_flags & B200OT_KERNEL_UNCLAMPED) ? 0.f : cost_clamp(kind_flags);
  if (kind_base(kind_flags) == B200OT_KERNEL_LAPLACIAN) return {kLog2e / blur, clamp * blur * blur};
  return {0.f, clamp};
}

// The coordinate scale s of the sqrt kernels, max |x - c| over both clouds, into the plan's misc block (behind
// max|w|): energy has no exponent to bound |X| (the gaussian pack's +-60000 clamp would cut real coordinates), and
// with |X| <= 1 every fp16 operand term is in range whatever the units of the data.
static int tc_coord_absmax(const TcPlan& p, unsigned char* base, const float* x, int64_t N, const float* y, int64_t M,
                           int D, const float* center, cudaStream_t st, const float** out) {
  float* s = reinterpret_cast<float*>(base + p.off_misc) + 1;
  B200OT_CUDA_TRY(cudaMemsetAsync(s, 0, sizeof(float), st));
  coord_absmax_kernel<<<(unsigned)std::min<int64_t>(ceil_div64((N + M) * D, 256), 1024), 256, 0, st>>>(x, N, y, M, D,
                                                                                                      center, s);
  B200OT_CUDA_TRY(cudaGetLastError());
  *out = s;
  return B200OT_OK;
}

// Row gradients on the tensor-core path (kind 0: gaussian conv, 1: softmin p=2, 2 / 3: laplacian / energy conv with
// tc_sqrt_params (kc, clampq); their coordinate scale is returned in *coord_out for the finalize).  Leaves n_part sets
// of (N, D+1) partial sums in *part_out.
int bwd_partial_tc(int kind, const float* x, const float* y, const float* w, const float* h_a, const float* h_b,
                   float h_scale_b, const float* lse2, const float* center, float scale, int64_t N, int64_t M, int D,
                   void* scratch, float** part_out, int* n_part_out, cudaStream_t st, const float** w_absmax_out,
                   float kc, float clampq, const float** coord_out) {
  const TcPlan p = make_tc_plan(N, M, D, true);
  if (p.nstage < 1) return B200OT_EINVAL;
  unsigned char* base = reinterpret_cast<unsigned char*>(scratch);
  unsigned char* a_imgs = base;
  unsigned char* b_imgs = base + p.off_b;
  float* part = reinterpret_cast<float*>(base + p.off_part);
  const bool sqrt_kind = kind >= 2;
  const float* coord = nullptr;
  if (sqrt_kind) {
    const int rc = tc_coord_absmax(p, base, x, N, y, M, D, center, st, &coord);
    if (rc) return rc;
  }
  if (coord_out) *coord_out = coord;
  float* w_absmax = nullptr;
  if (w != nullptr) {
    // P = w_j e_ij feeds an fp16 GEMM: normalise the weights to max|w| = 1 (undone by the finalize kernel)
    w_absmax = reinterpret_cast<float*>(base + p.off_misc);
    B200OT_CUDA_TRY(cudaMemsetAsync(w_absmax, 0, sizeof(float), st));
    absmax_kernel<<<(unsigned)std::min<int64_t>(ceil_div64(M, 256), 1024), 256, 0, st>>>(w, M, w_absmax);
    B200OT_CUDA_TRY(cudaGetLastError());
  }
  if (w_absmax_out) *w_absmax_out = w_absmax;
  const int threads = 128;
  tc_pack_kernel<<<(unsigned)ceil_div64(p.a_tiles_pad * kTcM, threads), threads, 0, st>>>(
      x, nullptr, nullptr, nullptr, 0.f, 0.f, center, scale, N, D, p.kp, kTcM, 0, a_imgs, lse2, nullptr, kTcRT,
      coord);
  B200OT_CUDA_TRY(cudaGetLastError());
  tc_pack_kernel<<<(unsigned)ceil_div64(p.b_tiles * kTcBN, threads), threads, 0, st>>>(
      y, w, h_a, h_b, h_scale_b, kLog2e, center, scale, M, D, p.kp, kTcBN, 1, b_imgs, nullptr, w_absmax, 1, coord);
  B200OT_CUDA_TRY(cudaGetLastError());
  dim3 grid((unsigned)p.a_tiles, (unsigned)p.n_split);
  // K_xx: exact zero exponent (gaussian) / zero gradient (laplacian, energy) on the diagonal
  const int self_mode = (kind != 1 && x == y && N == M) ? 1 : 0;
  const TcBwdTuning tn = tc_bwd_tuning();
  auto launch = [&](auto kern, int threads) -> int {
    B200OT_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
    kern<<<grid, threads, (size_t)p.smem, st>>>(a_imgs, b_imgs, part, N, p.kp, (int)p.b_tiles, p.tiles_per_split,
                                                p.nstage, D, self_mode, kc, clampq, coord);
    B200OT_CUDA_TRY(cudaGetLastError());
    return B200OT_OK;
  };
  // (MODE, PT, epilogue warps, LDALL, MERGE) -> instantiation
  auto pick3 = [&](auto mode_tag, auto pt_tag, auto merge_tag) -> int {
    constexpr int MODE = decltype(mode_tag)::value, PT = decltype(pt_tag)::value;
    constexpr bool MG = decltype(merge_tag)::value;
    if (tn.epi == 16) return launch(tc_bwd_kernel<TcBwdCfg16, MODE, PT, false, MG>, TcBwdCfg16::THREADS);
    if (tn.ldall) return launch(tc_bwd_kernel<TcBwdCfg, MODE, PT, true, MG>, TcBwdCfg::THREADS);
    return launch(tc_bwd_kernel<TcBwdCfg, MODE, PT, false, MG>, TcBwdCfg::THREADS);
  };
  auto pick = [&](auto mode_tag) -> int {
    using T1 = std::integral_constant<int, 1>;
    using T2 = std::integral_constant<int, 2>;
    if (tn.merge)
      return tn.p_terms == 1 ? pick3(mode_tag, T1{}, std::true_type{}) : pick3(mode_tag, T2{}, std::true_type{});
    return tn.p_terms == 1 ? pick3(mode_tag, T1{}, std::false_type{}) : pick3(mode_tag, T2{}, std::false_type{});
  };
  int rc;
  switch (kind) {
    case 0: rc = pick(std::integral_constant<int, 2>{}); break;
    case 1: rc = pick(std::integral_constant<int, 3>{}); break;
    case 2: rc = pick(std::integral_constant<int, 4>{}); break;
    default: rc = pick(std::integral_constant<int, 5>{}); break;
  }
  if (rc) return rc;
  *part_out = part;
  *n_part_out = p.n_split;  // G of a CTA is complete over its column split (both column halves feed one GEMM)
  return B200OT_OK;
}

// Tensor-core softmin partials (p = 2): packs both clouds, runs the reduction, leaves n_part (m, s) sets in
// `*part_out` (inside scratch) for b200ot_softmin_finalize.
int softmin_partial_tc(const float* x, const float* y, const float* h_a, const float* h_b, float h_scale_b,
                       const float* center, int64_t N, int64_t M, int D, float eps, void* scratch,
                       float** part_out, int* n_part_out, cudaStream_t st) {
  const TcPlan p = make_tc_plan(N, M, D);
  if (p.nstage < 1) return B200OT_EINVAL;
  unsigned char* base = reinterpret_cast<unsigned char*>(scratch);
  unsigned char* a_imgs = base;
  unsigned char* b_imgs = base + p.off_b;
  float* part = reinterpret_cast<float*>(base + p.off_part);
  const float scale = softmin_coord_scale(2, eps);
  const int threads = 128;
  tc_pack_kernel<<<(unsigned)ceil_div64(p.a_tiles_pad * kTcM, threads), threads, 0, st>>>(
      x, nullptr, nullptr, nullptr, 0.f, 0.f, center, scale, N, D, p.kp, kTcM, 0, a_imgs, nullptr, nullptr, kTcRT);
  B200OT_CUDA_TRY(cudaGetLastError());
  tc_pack_kernel<<<(unsigned)ceil_div64(p.b_tiles * kTcBN, threads), threads, 0, st>>>(
      y, nullptr, h_a, h_b, h_scale_b, kLog2e, center, scale, M, D, p.kp, kTcBN, 1, b_imgs);
  B200OT_CUDA_TRY(cudaGetLastError());
  auto kern = tc_reduce_kernel<TcConvCfg, 1>;
  B200OT_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
  dim3 grid((unsigned)(p.a_tiles_pad / kTcRT), (unsigned)p.n_split);
  kern<<<grid, TcConvCfg::THREADS, (size_t)p.smem, st>>>(a_imgs, b_imgs, part, N, p.kp, (int)p.b_tiles,
                                                        p.tiles_per_split, p.nstage, D, 0, 0.f, 0.f, nullptr);
  B200OT_CUDA_TRY(cudaGetLastError());
  *part_out = part;
  *n_part_out = p.n_split * (kTcEpi / 4);
  return B200OT_OK;
}

// kind_flags: gaussian (MODE 0), laplacian (MODE 4) or energy (MODE 5), with or without B200OT_KERNEL_UNCLAMPED
static int conv_fwd_tc(int kind_flags, const float* x, const float* y, const float* w, const float* center, float* out,
                       int64_t N, int64_t M, int D, float blur, void* scratch, cudaStream_t st) {
  const int kind = kind_base(kind_flags);
  const int self_mode = (x == y && N == M) ? 1 : 0;  // K_xx / K_yy: the diagonal exponent is exactly 0 (tcconv.cuh)
  const TcPlan p = make_tc_plan(N, M, D);
  if (p.nstage < 1) return B200OT_EINVAL;
  unsigned char* base = reinterpret_cast<unsigned char*>(scratch);
  unsigned char* a_imgs = base;
  unsigned char* b_imgs = base + p.off_b;
  float* part = reinterpret_cast<float*>(base + p.off_part);
  const bool gauss = kind == B200OT_KERNEL_GAUSSIAN;
  const float scale = gauss ? sqrtf(kLog2e) / blur : 1.f;
  const TcSqrtParams sq = gauss ? TcSqrtParams{0.f, 0.f} : tc_sqrt_params(kind_flags, blur);
  const float* coord = nullptr;
  if (!gauss) {
    const int rc = tc_coord_absmax(p, base, x, N, y, M, D, center, st, &coord);
    if (rc) return rc;
  }
  const int threads = 128;
  tc_pack_kernel<<<(unsigned)ceil_div64(p.a_tiles_pad * kTcM, threads), threads, 0, st>>>(
      x, nullptr, nullptr, nullptr, 0.f, 0.f, center, scale, N, D, p.kp, kTcM, 0, a_imgs, nullptr, nullptr, kTcRT,
      coord);
  B200OT_CUDA_TRY(cudaGetLastError());
  tc_pack_kernel<<<(unsigned)ceil_div64(p.b_tiles * kTcBN, threads), threads, 0, st>>>(
      y, w, nullptr, nullptr, 0.f, 0.f, center, scale, M, D, p.kp, kTcBN, 1, b_imgs, nullptr, nullptr, 1, coord);
  B200OT_CUDA_TRY(cudaGetLastError());
  auto kern = gauss ? tc_reduce_kernel<TcConvCfg, 0>
                    : (kind == B200OT_KERNEL_LAPLACIAN ? tc_reduce_kernel<TcConvCfg, 4> : tc_reduce_kernel<TcConvCfg, 5>);
  B200OT_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
  dim3 grid((unsigned)(p.a_tiles_pad / kTcRT), (unsigned)p.n_split);
  kern<<<grid, TcConvCfg::THREADS, (size_t)p.smem, st>>>(a_imgs, b_imgs, part, N, p.kp, (int)p.b_tiles,
                                                        p.tiles_per_split, p.nstage, D, self_mode, sq.kc, sq.clampq,
                                                        coord);
  B200OT_CUDA_TRY(cudaGetLastError());
  conv_fwd_finalize_kernel<<<(unsigned)ceil_div64(N, 256), 256, 0, st>>>(
      part, p.n_split * (kTcEpi / 4), kind == B200OT_KERNEL_ENERGY ? -1.f : 1.f, out, N);
  B200OT_CUDA_TRY(cudaGetLastError());
  return B200OT_OK;
}

}  // namespace b200ot

using namespace b200ot;

extern "C" {

B200OT_API int64_t b200ot_kernel_conv_scratch_bytes(int64_t N, int64_t M, int32_t D) {
  if (N <= 0 || M <= 0 || D <= 0) return 0;
  if (D > B200OT_MAX_D) return tc_capable_dim(D) ? tc_scratch_bytes(N, M, D) : 0;
  const ReducePlan pl = make_plan(N, M, D);
  const int64_t cols = b200ot_packed_cols_floats(M, D, 2) * 4;
  const int64_t part = (int64_t)pl.n_split * N * 4 * (D + 1);
  const int64_t simt = round_up64(cols, 256) + round_up64(part, 256);
  // (one size for every operator of the shape: the caller does not say which one it is about to run)
  return tc_any_routed(D, N, M) ? std::max(simt, tc_scratch_bytes(N, M, D)) : simt;
}

B200OT_API int b200ot_kernel_conv_finalize(const float* part, int32_t n_part, float* out, int64_t N, int32_t kind,
                                           void* stream) {
  if (!part || !out || n_part <= 0 || N <= 0 || !valid_kind(kind)) return B200OT_EINVAL;
  const int threads = 256;
  conv_fwd_finalize_kernel<<<(unsigned)ceil_div64(N, threads), threads, 0, (cudaStream_t)stream>>>(
      part, n_part, kind_base(kind) == B200OT_KERNEL_ENERGY ? -1.f : 1.f, out, N);
  B200OT_CUDA_TRY(cudaGetLastError());
  return B200OT_OK;
}

B200OT_API int b200ot_kernel_conv_bwd_finalize(const float* part, int32_t n_part, const float* x, const float* center,
                                               const float* grad_out, float* grad_x, int64_t N, int32_t D,
                                               int32_t kind, float blur, void* stream) {
  if (!part || !x || !grad_out || !grad_x || n_part <= 0 || N <= 0 || !supported_simt_dim(D) || !valid_kind(kind))
    return B200OT_EINVAL;
  if (kind_base(kind) != B200OT_KERNEL_ENERGY && !(blur > 0.f)) return B200OT_EINVAL;
  const ConvScales cs = conv_scales(kind, blur);
  const int threads = 256;
  conv_bwd_finalize_kernel<<<(unsigned)ceil_div64(N, threads), threads, 0, (cudaStream_t)stream>>>(
      part, n_part, x, center, grad_out, grad_x, N, D, kind_base(kind), cs.scale, conv_bwd_coef(kind, cs, blur),
      (const float*)nullptr);
  B200OT_CUDA_TRY(cudaGetLastError());
  return B200OT_OK;
}

B200OT_API int b200ot_kernel_conv_pack_gather(const float* y, const float* w, const float* center,
                                              const int32_t* src_index, int64_t n_slots, int32_t D, int32_t kind,
                                              float blur, float* cols_out, void* stream) {
  if (!y || !w || !src_index || !cols_out || n_slots <= 0 || !supported_simt_dim(D) || !valid_kind(kind))
    return B200OT_EINVAL;
  if (kind_base(kind) != B200OT_KERNEL_ENERGY && !(blur > 0.f)) return B200OT_EINVAL;
  if (((uintptr_t)cols_out) & 15) return B200OT_EALIGN;
  return conv_pack(y, w, center, n_slots, D, conv_scales(kind, blur), cols_out, (cudaStream_t)stream,
                   reinterpret_cast<const int*>(src_index));
}

// part: (N) sums (forward) or (N, width) sums (row gradients: width = D + 1 gaussian, D otherwise)
B200OT_API int b200ot_kernel_conv_partial_ranges(const float* x, const float* center, const float* cols,
                                                 const b200ot_segment* seg, int64_t n_seg,
                                                 const b200ot_piece* pieces, float* part, int64_t N, int32_t D,
                                                 int32_t kind, float blur, int32_t backward, int32_t variant,
                                                 void* stream) {
  if (!x || !cols || !seg || !pieces || !part || N <= 0 || n_seg <= 0 || n_seg > 0x7fffffff ||
      !supported_simt_dim(D) || !valid_kind(kind) ||
      (variant != B200OT_RANGES_BIG && variant != B200OT_RANGES_SMALL))
    return B200OT_EINVAL;
  if (kind_base(kind) != B200OT_KERNEL_ENERGY && !(blur > 0.f)) return B200OT_EINVAL;
  if ((((uintptr_t)cols) & 15) || (((uintptr_t)seg) & 15) || (((uintptr_t)pieces) & 7)) return B200OT_EALIGN;
  return conv_partial(kind, backward != 0, ranges_plan(variant, n_seg), (cudaStream_t)stream, x, center,
                      conv_scales(kind, blur), cols, part, N, D, reinterpret_cast<const int4*>(seg),
                      reinterpret_cast<const int2*>(pieces));
}

// Laplacian / energy take the tensor cores above B200OT_MAX_D only: at D <= B200OT_MAX_D they stay on the CUDA cores
// whatever $B200OT_TC_MIN_D / $B200OT_TC_MIN_PAIRS say (tc_routed's cross-over was measured for the gaussian).
static bool conv_tc(int op, int kind_flags, int D, int64_t N, int64_t M) {
  if (kind_base(kind_flags) == B200OT_KERNEL_GAUSSIAN) return tc_routed(op, D, N, M);
  return D > B200OT_MAX_D && tc_capable_dim(D);
}

B200OT_API int b200ot_kernel_conv_fwd(const float* x, const float* y, const float* w, const float* center,
                                      float* out, int64_t N, int64_t M, int32_t D, int32_t kind, float blur,
                                      void* scratch, int64_t scratch_bytes, void* stream) {
  const bool tc = conv_tc(kTcConvFwd, kind, D, N, M);
  if (!x || !y || !w || !out || !scratch || N <= 0 || M <= 0 || (!supported_simt_dim(D) && !tc) || !valid_kind(kind))
    return B200OT_EINVAL;
  if (kind_base(kind) != B200OT_KERNEL_ENERGY && !(blur > 0.f)) return B200OT_EINVAL;
  if (((uintptr_t)scratch) & 15) return B200OT_EALIGN;
  if (scratch_bytes < b200ot_kernel_conv_scratch_bytes(N, M, D)) return B200OT_ESCRATCH;
  if (tc) return conv_fwd_tc(kind, x, y, w, center, out, N, M, D, blur, scratch, (cudaStream_t)stream);
  const ReducePlan pl = make_plan(N, M, D);
  const ConvScales cs = conv_scales(kind, blur);
  float* cols = reinterpret_cast<float*>(scratch);
  float* part = reinterpret_cast<float*>(reinterpret_cast<char*>(scratch) +
                                         round_up64(b200ot_packed_cols_floats(M, D, 2) * 4, 256));
  cudaStream_t st = (cudaStream_t)stream;
  int rc = conv_pack(y, w, center, M, D, cs, cols, st);
  if (rc) return rc;
  rc = conv_partial(kind, false, pl, st, x, center, cs, cols, part, N, D);
  if (rc) return rc;
  return b200ot_kernel_conv_finalize(part, pl.n_split, out, N, kind, stream);
}

// Row gradients (and, with value_out, the forward values from the same pass: gaussian only).
static int conv_bwd_x_impl(const float* x, const float* y, const float* w, const float* center, const float* grad_out,
                           float* grad_x, float* value_out, int64_t N, int64_t M, int32_t D, int32_t kind, float blur,
                           void* scratch, int64_t scratch_bytes, void* stream) {
  const bool gauss = kind_base(kind) == B200OT_KERNEL_GAUSSIAN;
  const bool tc = conv_tc(kTcConvBwd, kind, D, N, M);
  if (!x || !y || !w || !grad_x || !scratch || N <= 0 || M <= 0 || (!supported_simt_dim(D) && !tc) ||
      !valid_kind(kind) || (value_out && !gauss))
    return B200OT_EINVAL;
  if (kind_base(kind) != B200OT_KERNEL_ENERGY && !(blur > 0.f)) return B200OT_EINVAL;
  if (((uintptr_t)scratch) & 15) return B200OT_EALIGN;
  if (scratch_bytes < b200ot_kernel_conv_scratch_bytes(N, M, D)) return B200OT_ESCRATCH;
  if (tc && !gauss) {
    // P = w k'(r)/r without its negative factor (tcbwd.cuh): grad = go (-k'(r)/r factor) (sum P Y - X sum P)
    float* tc_part = nullptr;
    int n_part = 0;
    const float* w_absmax = nullptr;
    const float* coord = nullptr;
    const TcSqrtParams sq = tc_sqrt_params(kind, blur);
    const bool lap = kind_base(kind) == B200OT_KERNEL_LAPLACIAN;
    const int rc = bwd_partial_tc(lap ? 2 : 3, x, y, w, nullptr, nullptr, 0.f, nullptr, center, 1.f, N, M, D, scratch,
                                  &tc_part, &n_part, (cudaStream_t)stream, &w_absmax, sq.kc, sq.clampq, &coord);
    if (rc) return rc;
    conv_bwd_finalize_kernel<<<(unsigned)ceil_div64(N, 256), 256, 0, (cudaStream_t)stream>>>(
        tc_part, n_part, x, center, grad_out, grad_x, N, D, kind_base(kind), 1.f, lap ? 1.0f / blur : 1.0f, w_absmax,
        nullptr, coord);
    B200OT_CUDA_TRY(cudaGetLastError());
    return B200OT_OK;
  }
  if (tc) {
    float* tc_part = nullptr;
    int n_part = 0;
    const float scale = sqrtf(kLog2e) / blur;
    const float* w_absmax = nullptr;
    const int rc = bwd_partial_tc(0, x, y, w, nullptr, nullptr, 0.f, nullptr, center, scale, N, M, D, scratch,
                                  &tc_part, &n_part, (cudaStream_t)stream, &w_absmax);
    if (rc) return rc;
    conv_bwd_finalize_kernel<<<(unsigned)ceil_div64(N, 256), 256, 0, (cudaStream_t)stream>>>(
        tc_part, n_part, x, center, grad_out, grad_x, N, D, 0, scale, 1.0f / (scale * blur * blur), w_absmax,
        value_out);
    B200OT_CUDA_TRY(cudaGetLastError());
    return B200OT_OK;
  }
  const ReducePlan pl = make_plan(N, M, D);
  const ConvScales cs = conv_scales(kind, blur);
  float* cols = reinterpret_cast<float*>(scratch);
  float* part = reinterpret_cast<float*>(reinterpret_cast<char*>(scratch) +
                                         round_up64(b200ot_packed_cols_floats(M, D, 2) * 4, 256));
  cudaStream_t st = (cudaStream_t)stream;
  int rc = conv_pack(y, w, center, M, D, cs, cols, st);
  if (rc) return rc;
  rc = conv_partial(kind, true, pl, st, x, center, cs, cols, part, N, D);
  if (rc) return rc;
  conv_bwd_finalize_kernel<<<(unsigned)ceil_div64(N, 256), 256, 0, st>>>(
      part, pl.n_split, x, center, grad_out, grad_x, N, D, kind_base(kind), cs.scale, conv_bwd_coef(kind, cs, blur),
      (const float*)nullptr, value_out);
  B200OT_CUDA_TRY(cudaGetLastError());
  return B200OT_OK;
}

B200OT_API int b200ot_kernel_conv_bwd_x(const float* x, const float* y, const float* w, const float* center,
                                        const float* grad_out, float* grad_x, int64_t N, int64_t M, int32_t D,
                                        int32_t kind, float blur, void* scratch, int64_t scratch_bytes,
                                        void* stream) {
  if (!grad_out) return B200OT_EINVAL;
  return conv_bwd_x_impl(x, y, w, center, grad_out, grad_x, nullptr, N, M, D, kind, blur, scratch, scratch_bytes,
                         stream);
}

B200OT_API int b200ot_kernel_conv_fwd_bwd_x(const float* x, const float* y, const float* w, const float* center,
                                            float* out, float* grad_unit, int64_t N, int64_t M, int32_t D,
                                            int32_t kind, float blur, void* scratch, int64_t scratch_bytes,
                                            void* stream) {
  if (!out) return B200OT_EINVAL;
  return conv_bwd_x_impl(x, y, w, center, nullptr, grad_unit, out, N, M, D, kind, blur, scratch, scratch_bytes,
                         stream);
}

}  // extern "C"
