// Shared helpers for the matten_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/matten_b200.h"

namespace mt {

// ----------------------------------------------------------------- errors --
char* last_error_buf();  // thread-local, defined in api.cu
void count_launch();     // bumps the process-wide kernel-launch counter (mt_launch_count)
int set_error(int code, const char* fmt, ...);
int check_device();  // MT_OK iff current device is cc 10.x

#define MT_CUDA_OK(expr)                                                              \
  do {                                                                                \
    cudaError_t _e = (expr);                                                          \
    if (_e != cudaSuccess)                                                            \
      return ::mt::set_error(MT_ECUDA, "%s failed: %s (%s:%d)", #expr,                \
                             cudaGetErrorString(_e), __FILE__, __LINE__);             \
  } while (0)

#define MT_LAUNCH_OK()                                                                \
  do {                                                                                \
    cudaError_t _e = cudaGetLastError();                                              \
    if (_e != cudaSuccess)                                                            \
      return ::mt::set_error(MT_ECUDA, "kernel launch failed: %s (%s:%d)",            \
                             cudaGetErrorString(_e), __FILE__, __LINE__);             \
    ::mt::count_launch();                                                             \
  } while (0)

#define MT_REQUIRE(cond, ...)                                                         \
  do {                                                                                \
    if (!(cond)) return ::mt::set_error(MT_EINVAL, __VA_ARGS__);                      \
  } while (0)

#define MT_ENTRY_GUARD()                                                              \
  do {                                                                                \
    int _rc = ::mt::check_device();                                                   \
    if (_rc != MT_OK) return _rc;                                                     \
  } while (0)

// dispatch on dtype: calls FN<float>(...) or FN<double>(...)
#define MT_DISPATCH_DTYPE(dtype, ...)                                                 \
  do {                                                                                \
    if ((dtype) == MT_F32) {                                                          \
      using T = float;                                                                \
      __VA_ARGS__                                                                     \
    } else if ((dtype) == MT_F64) {                                                   \
      using T = double;                                                               \
      __VA_ARGS__                                                                     \
    } else {                                                                          \
      return ::mt::set_error(MT_EINVAL, "unknown dtype %d", (int)(dtype));            \
    }                                                                                 \
  } while (0)

inline cudaStream_t as_stream(mt_stream s) { return reinterpret_cast<cudaStream_t>(s); }

constexpr int kNumSMs = 148;  // B200

template <typename I>
__host__ __device__ constexpr I ceil_div(I a, I b) {
  return (a + b - 1) / b;
}

__host__ __device__ __forceinline__ int64_t imin64(int64_t a, int64_t b) { return a < b ? a : b; }

// workspace regions start at multiples of 256 bytes
inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// ------------------------------------------------------------ species-indexed linear (node_ops.cu) --
// MT_OK iff every block has dim 2l+1 <= 9 and lies within in_dim / out_dim, and, when reads_weight, the weight is
// given for every block with input channels.  mt_linear_fwd and mt_linear_bwd check their blocks with it.
// Both are internal to the library: hidden from its dynamic symbol table, which holds the C ABI.
__attribute__((visibility("hidden"))) int linear_check_blocks(const mt_lin_block* blocks, int num_blocks, int in_dim,
                                                              int out_dim, const void* weight, bool reads_weight);
// Backward of mt_linear_fwd w.r.t. x: the transposed weight slices applied to grad_out, for checked blocks.
__attribute__((visibility("hidden"))) int linear_transposed(
    int dtype, const mt_lin_block* blocks, int num_blocks, int in_dim, int out_dim, int num_species,
    const void* grad_out, const void* weight, const int32_t* species_perm, const int32_t* species_ptr, int accumulate,
    void* grad_x, int64_t N, cudaStream_t st);

// padded size (8 / 16 / 32 / 64) of the last hidden layer of the radial MLP in the FMA-pipe kernels; -1: over 64
inline int pad_hp(int h) {
  if (h <= 8) return 8;
  if (h <= 16) return 16;
  if (h <= 32) return 32;
  if (h <= 64) return 64;
  return -1;
}

// ------------------------------------------------------------ packed fp32 --
// Two fp32 lanes in one register pair: sm_100 issues FFMA2 / FMUL2 (two IEEE fp32 FMAs per instruction).  The
// generated CG contractions are templates on the scalar type, so instantiating them with f2 processes two edges per
// instruction stream at half the issue slots -- these kernels are issue-bound, not FMA-pipe-bound.
struct f2 {
  float2 v;
  __device__ __forceinline__ f2() {}
  __device__ __forceinline__ f2(float a, float b) : v(make_float2(a, b)) {}
  __device__ __forceinline__ explicit f2(float a) : v(make_float2(a, a)) {}
  __device__ __forceinline__ explicit f2(double a) : v(make_float2((float)a, (float)a)) {}
  __device__ __forceinline__ explicit f2(int a) : v(make_float2((float)a, (float)a)) {}
};
__device__ __forceinline__ f2 operator-(f2 a) { return f2(-a.v.x, -a.v.y); }  // folds into an operand modifier
__device__ __forceinline__ f2 operator*(f2 a, f2 b) {
  f2 r;
  r.v = __fmul2_rn(a.v, b.v);
  return r;
}
using ::fma;  // keep the scalar overloads visible next to the packed one
__device__ __forceinline__ f2 fma(f2 a, f2 b, f2 c) {
  f2 r;
  r.v = __ffma2_rn(a.v, b.v, c.v);
  return r;
}

// c[0..1] += s * b[0..1] for a register pair (one FFMA2 with a broadcast scalar operand in fp32)
__device__ __forceinline__ void fma_pair(float s, float b0, float b1, float2& c) {
  c = __ffma2_rn(make_float2(s, s), make_float2(b0, b1), c);
}
__device__ __forceinline__ void fma_pair(double s, double b0, double b1, double2& c) {
  c.x = fma(s, b0, c.x);
  c.y = fma(s, b1, c.y);
}
template <typename T> struct pair_of;
template <> struct pair_of<float> { using type = float2; };
template <> struct pair_of<double> { using type = double2; };

// ------------------------------------------------------------ activations --
template <typename T>
__device__ __forceinline__ T act_sigmoid(T v) {
  return T(1) / (T(1) + exp(-v));
}
template <>
__device__ __forceinline__ float act_sigmoid<float>(float v) {
  return 1.0f / (1.0f + expf(-v));
}

template <typename T>
__device__ __forceinline__ T act_softplus(T v) {  // torch.nn.Softplus(beta=1, threshold=20)
  return v > T(20) ? v : log1p(exp(v));
}

template <typename T>
__device__ __forceinline__ T act_tanh(T v) {
  return tanh(v);
}

// value of activation `id` (un-normalised)
template <typename T>
__device__ __forceinline__ T apply_act(int id, T v) {
  switch (id) {
    case MT_ACT_SILU: return v * act_sigmoid(v);
    case MT_ACT_TANH: return act_tanh(v);
    case MT_ACT_SIGMOID: return act_sigmoid(v);
    // softplus(v) - log 2 = log1p(expm1(v) / 2): no cancellation next to v = 0 (NormActivation feeds norms there)
    case MT_ACT_SSP: return v > T(20) ? v - T(0.6931471805599453) : log1p(T(0.5) * expm1(v));
    case MT_ACT_ABS: return fabs(v);
    default: return v;
  }
}

// derivative of activation `id`
template <typename T>
__device__ __forceinline__ T apply_act_grad(int id, T v) {
  switch (id) {
    case MT_ACT_SILU: {
      T s = act_sigmoid(v);
      return s * (T(1) + v * (T(1) - s));
    }
    case MT_ACT_TANH: {
      T t = act_tanh(v);
      return T(1) - t * t;
    }
    case MT_ACT_SIGMOID: {
      T s = act_sigmoid(v);
      return s * (T(1) - s);
    }
    case MT_ACT_SSP: return v > T(20) ? T(1) : act_sigmoid(v);
    case MT_ACT_ABS: return v > T(0) ? T(1) : (v < T(0) ? T(-1) : T(0));
    default: return T(1);
  }
}

}  // namespace mt
