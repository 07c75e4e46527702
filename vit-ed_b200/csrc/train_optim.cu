// The rest of a Hisfrag training iteration after the backward pass (misc/engine.py:189-257, misc/utils.py:206-226):
// overflow detection for the loss-scaled 16-bit gradients, the global gradient norm of clip_grad_norm_ and a fused
// AdamW step. The host side is vit-ed_b200/train.py (LossScaler, AdamW, train_iteration).
//   range_check: the 16-bit conversions of this library saturate (fp16 at +-65504) instead of producing inf, so an
//                overflowing loss-scaled gradient would pass unnoticed; the host checks every buffer a loss-scaled
//                gradient is converted from or to and skips the step when the sticky flag is set.
//   grad_norm:   multi-tensor sum of squares, fp64 per thread over a fixed partition (grid-stride over every tensor
//                with a grid of n_partials blocks), fixed-order block and final reductions: bit-reproducible.
//   adamw:       one multi-tensor launch; the operations of torch.optim.AdamW's single-tensor form, one by one.
// Multi-tensor kernels read a device table with one row per tensor and only do scalar (4-byte) accesses, so a tensor
// may start at any element offset.
#include "kernels.h"

namespace vited {

namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ bool out_of_range(float v, float limit) { return !(fabsf(v) < limit); }   // NaN too

__device__ __forceinline__ bool vec_out_of_range(uint4 u, float limit, float) {
  return out_of_range(__uint_as_float(u.x), limit) | out_of_range(__uint_as_float(u.y), limit) |
         out_of_range(__uint_as_float(u.z), limit) | out_of_range(__uint_as_float(u.w), limit);
}
__device__ __forceinline__ bool vec_out_of_range(uint4 u, float limit, act_t) {
  const float2 a = unpack_act(u.x), b = unpack_act(u.y), c = unpack_act(u.z), d = unpack_act(u.w);
  return out_of_range(a.x, limit) | out_of_range(a.y, limit) | out_of_range(b.x, limit) | out_of_range(b.y, limit) |
         out_of_range(c.x, limit) | out_of_range(c.y, limit) | out_of_range(d.x, limit) | out_of_range(d.y, limit);
}
__device__ __forceinline__ float to_float(float v) { return v; }
__device__ __forceinline__ float to_float(act_t v) { return act2f(v); }

// x[0, head) and x[head + n_vec * W, n) element by element, the 16-byte aligned middle as uint4 loads
template <typename T>
__global__ void range_check_kernel(const T* __restrict__ x, int64_t head, int64_t n_vec, int64_t n, float limit,
                                   int* __restrict__ flag) {
  constexpr int W = 16 / sizeof(T);
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t tail0 = head + n_vec * W, n_scalar = head + (n - tail0);
  bool bad = false;
  for (int64_t i = tid; i < n_scalar; i += stride) bad |= out_of_range(to_float(x[i < head ? i : tail0 + (i - head)]), limit);
  const uint4* xv = reinterpret_cast<const uint4*>(x + head);
  for (int64_t i = tid; i < n_vec; i += stride) bad |= vec_out_of_range(__ldg(xv + i), limit, T());
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) *flag = 1;
}

// table rows of grad_norm: (pointer, numel); of adamw: (param, grad, exp_avg, exp_avg_sq, numel, weight decay as the
// bits of a double)
constexpr int kNormCols = 2, kAdamCols = 6;

__global__ void grad_norm_partial_kernel(const int64_t* __restrict__ table, int n_tensors, double* __restrict__ partials) {
  __shared__ double warp_part[kThreads / 32];
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
  double acc = 0.0;
  for (int t = 0; t < n_tensors; ++t) {
    const float* g = reinterpret_cast<const float*>(table[t * kNormCols]);
    const int64_t n = table[t * kNormCols + 1];
    for (int64_t i = tid; i < n; i += stride) {
      const double v = g[i];
      acc += v * v;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) s += warp_part[w];
    partials[blockIdx.x] = s;
  }
}

// out[0] = (float) sum of the partials; the int32 at out + 1 is the sticky overflow flag, set for a non-finite sum
__global__ void grad_norm_final_kernel(const double* __restrict__ partials, int n_partials, float* __restrict__ out) {
  __shared__ double warp_part[1024 / 32];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n_partials; i += blockDim.x) acc += partials[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += warp_part[w];
    const float sf = (float)s;
    out[0] = sf;
    if (!isfinite(sf)) *reinterpret_cast<int*>(out + 1) = 1;
  }
}

// torch.optim.AdamW (foreach=False, fused=False, amsgrad=False, maximize=False), per element of every tensor:
//   p *= 1 - lr * wd                 (Python double, applied as a float scalar; skipped for wd == 0 as torch does)
//   m.lerp_(g, 1 - beta1)            (torch's lerp: m + w (g - m) for |w| < 0.5, else g - (g - m)(1 - w))
//   v = v * beta2 + (1 - beta2) g g  (mul_ then addcmul_)
//   p += -step_size * m / (sqrt(v) / bc2_sqrt + eps),  step_size = lr / bc1
// with g = grad * clip_coef (clip_grad_norm_'s in-place multiply, here only in registers: grad is not written).
__global__ void adamw_kernel(const int64_t* __restrict__ table, int n_tensors, double lr, float one_minus_beta1,
                             float beta2, float one_minus_beta2, float eps, float clip_coef, float neg_step_size,
                             float bc2_sqrt) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
  const float w1 = one_minus_beta1;
  for (int t = 0; t < n_tensors; ++t) {
    const int64_t* row = table + (int64_t)t * kAdamCols;
    float* p = reinterpret_cast<float*>(row[0]);
    const float* grad = reinterpret_cast<const float*>(row[1]);
    float* m = reinterpret_cast<float*>(row[2]);
    float* v = reinterpret_cast<float*>(row[3]);
    const int64_t n = row[4];
    const double wd = __longlong_as_double(row[5]);
    const float decay = (float)(1.0 - lr * wd);
    for (int64_t i = tid; i < n; i += stride) {
      const float g = grad[i] * clip_coef;
      float pi = p[i];
      if (wd != 0.0) pi = pi * decay;
      float mi = m[i];
      mi = fabsf(w1) < 0.5f ? mi + w1 * (g - mi) : g - (g - mi) * (1.f - w1);
      float vi = v[i] * beta2;
      vi = vi + one_minus_beta2 * g * g;
      const float denom = sqrtf(vi) / bc2_sqrt + eps;
      pi = pi + neg_step_size * (mi / denom);
      p[i] = pi;
      m[i] = mi;
      v[i] = vi;
    }
  }
}

inline int grid_for(int64_t work) {
  int64_t b = (work + kThreads - 1) / kThreads;
  if (b > 148 * 8) b = 148 * 8;
  return b < 1 ? 1 : (int)b;
}

}  // namespace

float train_range_limit() { return kActRangeLimit; }

int train_range_check(const void* x, int is_f32, int64_t n, float limit, int* flag, cudaStream_t s) {
  VITED_CHECK(n >= 0 && flag, "train range check: n < 0 or null flag");
  if (n == 0) return 0;
  const int64_t es = is_f32 ? 4 : 2, w = 16 / es;
  const uintptr_t a = reinterpret_cast<uintptr_t>(x);
  VITED_CHECK(x && a % es == 0, "train range check: null or misaligned input");
  int64_t head = (int64_t)((16 - a % 16) % 16) / es;
  if (head > n) head = n;
  const int64_t n_vec = (n - head) / w;
  const int64_t work = n_vec > n - n_vec * w ? n_vec : n - n_vec * w;
  if (is_f32)
    range_check_kernel<float><<<grid_for(work), kThreads, 0, s>>>((const float*)x, head, n_vec, n, limit, flag);
  else
    range_check_kernel<act_t><<<grid_for(work), kThreads, 0, s>>>((const act_t*)x, head, n_vec, n, limit, flag);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

int train_grad_norm(const int64_t* table, int n_tensors, double* partials, int n_partials, float* out, cudaStream_t s) {
  VITED_CHECK(table && partials && out && n_tensors >= 0 && n_partials >= 1 && n_partials <= 65535,
              "train grad norm: bad arguments (n_tensors %d, n_partials %d)", n_tensors, n_partials);
  VITED_CHECK((reinterpret_cast<uintptr_t>(out) & 7) == 0, "train grad norm: out must be 8-byte aligned");
  grad_norm_partial_kernel<<<n_partials, kThreads, 0, s>>>(table, n_tensors, partials);
  VITED_CUDA_OK(cudaGetLastError());
  grad_norm_final_kernel<<<1, 1024, 0, s>>>(partials, n_partials, out);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

int train_adamw(const int64_t* table, int n_tensors, int64_t max_numel, double lr, double beta1, double beta2, double eps,
                float clip_coef, double bc1, double bc2, cudaStream_t s) {
  VITED_CHECK(table && n_tensors >= 0 && max_numel >= 0, "train adamw: bad arguments");
  VITED_CHECK(bc1 > 0.0 && bc2 > 0.0, "train adamw: bias corrections must be positive (step >= 1)");
  if (n_tensors == 0 || max_numel == 0) return 0;
  // the scalars as torch hands them to its float kernels: Python double arithmetic, then one rounding to float
  adamw_kernel<<<grid_for(max_numel), kThreads, 0, s>>>(table, n_tensors, lr, (float)(1.0 - beta1), (float)beta2,
                                                        (float)(1.0 - beta2), (float)eps, clip_coef, -(float)(lr / bc1),
                                                        (float)sqrt(bc2));
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace vited
