// b200ot — host-side helpers shared by the translation units of libb200ot.so.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "b200ot.h"

namespace b200ot {

inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline int64_t round_up64(int64_t a, int64_t b) { return ceil_div64(a, b) * b; }

// Last CUDA error text seen by any entry point (process-wide, best effort; for diagnostics only).
void set_last_cuda_error(cudaError_t e, const char* where);

// SM count of the current device, cached per device ordinal.
int num_sms();

// Dimensions served by the CUDA-core (register tile) kernels that are instantiated in this build.
inline bool supported_simt_dim(int D) { return D >= 1 && D <= B200OT_MAX_D; }

// Cost exponent argument of the C ABI: 1 or 2, optionally or-ed with B200OT_P_UNCLAMPED (p = 1 only matters).
inline int p_exponent(int p) { return p & 0xff; }
inline bool valid_p(int p) {
  const int e = p & 0xff;
  return (e == 1 || e == 2) && (p & ~(0xff | B200OT_P_UNCLAMPED)) == 0;
}
// Clamp on |x-y|^2 under the square root: the reference's tensorized `distances` clamps at 1e-8 (utils.py:61);
// pykeops' Norm2 / sqrt do not (sqrt(0) = 0 with a zero gradient) — emulated by a clamp far below fp32 resolution.
inline float cost_clamp(int flags) { return (flags & B200OT_P_UNCLAMPED) ? 1e-30f : 1e-8f; }

// Coordinate scale of the softmin kernels: the log2-domain exponent is H - |X-Y|^2/2 (p = 2) or
// H - |X-Y| (p = 1) with X = scale * (x - c).
inline float softmin_coord_scale(int p, float eps) {
  return p == 2 ? sqrtf(1.4426950408889634f / eps) : 1.4426950408889634f / eps;
}

// Shared between translation units (defined in b200ot_softmin.cu).
int softmin_pack_impl(const float* y, const float* h_a, const float* h_b, float h_scale_b, const float* center,
                      int64_t M, int D, int p, float eps, float* cols_out, cudaStream_t st, const int* src);

// Tensor-core (tcgen05) path, defined in b200ot_kernel_conv.cu.  The kernels serve any 1 <= D <= 64 (coordinates are
// zero-padded to a multiple of 16); above B200OT_MAX_D they are the only path, at or below it `tc_routed` decides per
// operator from the measured cross-over (see there).
enum TcOp { kTcSoftminFwd = 0, kTcSoftminBwd = 1, kTcConvFwd = 2, kTcConvBwd = 3 };
inline bool tc_capable_dim(int D) { return D >= 1 && D <= 64; }
bool tc_routed(int op, int D, int64_t N, int64_t M);
bool tc_any_routed(int D, int64_t N, int64_t M);  // some operator of this shape takes the tensor-core path (scratch sizing)
int64_t tc_scratch_bytes(int64_t N, int64_t M, int D);
int softmin_partial_tc(const float* x, const float* y, const float* h_a, const float* h_b, float h_scale_b,
                       const float* center, int64_t N, int64_t M, int D, float eps, void* scratch,
                       float** part_out, int* n_part_out, cudaStream_t st);

int bwd_partial_tc(int kind, const float* x, const float* y, const float* w, const float* h_a, const float* h_b,
                   float h_scale_b, const float* lse2, const float* center, float scale, int64_t N, int64_t M, int D,
                   void* scratch, float** part_out, int* n_part_out, cudaStream_t st, const float** w_absmax_out,
                   float kc = 0.f, float clampq = 0.f, const float** coord_out = nullptr);

#define B200OT_STR2(x) #x
#define B200OT_STR(x) B200OT_STR2(x)
#define B200OT_CUDA_TRY(expr)                                                         \
  do {                                                                                \
    cudaError_t e__ = (expr);                                                         \
    if (e__ != cudaSuccess) {                                                         \
      ::b200ot::set_last_cuda_error(e__, __FILE__ ":" B200OT_STR(__LINE__));          \
      return B200OT_ECUDA;                                                            \
    }                                                                                 \
  } while (0)

}  // namespace b200ot
