// Shared host/device helpers for libds2_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <atomic>

#include "../../include/ds2_b200.h"

namespace ds2 {

void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;
int precision();
inline bool tensor_core_mode() { return precision() != DS2_PREC_FP32; }   // TF32 or precision-16: tcgen05 kernels
inline bool f16_gemm_mode() { return precision() == DS2_PREC_F16; }       // fp16 operands for the dense RNN GEMMs

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// Host-side "once per device" latch: cudaFuncSetAttribute and the device attributes are per device, so a plain
// function-local static would leave the second GPU of a process without its shared-memory opt-in.
inline int current_device() {
  int d = 0;
  (void)cudaGetDevice(&d);
  return d & 63;
}
struct DeviceOnce {
  std::atomic<unsigned long long> mask{0};
  bool first() const { return !((mask.load(std::memory_order_acquire) >> current_device()) & 1ull); }
  void done() { mask.fetch_or(1ull << current_device(), std::memory_order_release); }
};
int device_sm_count();   // SM count of the current device (cached per device)

// A tensor-core-mode call that had to take the one-launch-per-time-step FFMA kernels (shape not eligible for the
// persistent sweeps): counted and reported once per shape on stderr, never silent.
void note_fallback(const char* what, int rnn, int T, int B, int H, int D);

// Optional side stream (ds2_set_side_stream): deferred work whose results nobody on the main stream needs before
// ds2_join_side_stream.  Workspaces read by side work are protected by per-workspace events.
extern std::atomic<void*> g_side_stream;
int side_wait_for_workspace(const void* ws, cudaStream_t main);
int side_fork(cudaStream_t main, cudaStream_t side);
int side_mark_workspace(const void* ws, cudaStream_t side);

#define DS2_CHECK_CUDA(expr)                                                             \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) {                                                             \
      ds2::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return DS2_ERR_CUDA;                                                               \
    }                                                                                    \
  } while (0)

#define DS2_REQUIRE(cond, ...)                      \
  do {                                              \
    if (!(cond)) {                                  \
      ds2::set_error(__VA_ARGS__);                  \
      return DS2_ERR_INVALID;                       \
    }                                               \
  } while (0)

// Launch bookkeeping: every kernel launch of the library goes through this.
#define DS2_LAUNCH(kernel, grid, block, smem, stream, ...)                \
  do {                                                                    \
    kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);           \
    ds2::g_launches.fetch_add(1, std::memory_order_relaxed);              \
    DS2_CHECK_CUDA(cudaGetLastError());                                   \
  } while (0)

// Device-time ranges (cudaEvent pairs on the launching stream), off unless ds2_prof_enable(1).
void prof_begin(const char* tag, cudaStream_t st);
void prof_end(cudaStream_t st);
struct ProfRange {
  cudaStream_t st;
  ProfRange(const char* tag, cudaStream_t s) : st(s) { prof_begin(tag, s); }
  ~ProfRange() { prof_end(st); }
};
#define DS2_PROF(tag, st) ds2::ProfRange _prof_range_##__LINE__(tag, st)

inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }
#ifdef __CUDACC__
__device__ __forceinline__ int cdiv_dev(int a, int b) { return (a + b - 1) / b; }
#endif
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bump allocator over a caller-provided workspace.
struct Arena {
  char* base;
  size_t cap, off;
  Arena(void* p, size_t n) : base(static_cast<char*>(p)), cap(n), off(0) {}
  template <typename T>
  T* take(size_t count) {
    size_t bytes = align_up(count * sizeof(T), 256);
    if (off + bytes > cap) return nullptr;
    T* r = reinterpret_cast<T*>(base + off);
    off += bytes;
    return r;
  }
};

#ifdef __CUDACC__
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
#endif

// ---- internal cross-file entry points -------------------------------------------------------
// C[M,N] = alpha*op(A)op(B) + beta*C (row-major, fp32 FFMA kernel; any shape/stride)
int gemm_simt(int transA, int transB, int M, int N, int K, float alpha, const float* A, int lda, const float* B,
              int ldb, float beta, float* C, int ldc, void* ws, size_t ws_bytes, cudaStream_t st);
size_t gemm_simt_workspace_bytes(int M, int N, int K);
// tcgen05 TF32 kernel.  Returns 1 if the shape is not eligible (caller falls back to gemm_simt).
int gemm_tc(int transA, int transB, int M, int N, int K, float alpha, const float* A, int lda, const float* B,
            int ldb, float beta, float* C, int ldc, void* ws, size_t ws_bytes, cudaStream_t st);
size_t gemm_tc_workspace_bytes(int transA, int transB, int M, int N, int K);
// precision-16 GEMM: fp16 K-major operands, fp32 accumulation / output (gemm_tc.cu); 1 = not eligible
int gemm_tc_f16(int M, int N, int K, float alpha, const void* A16, int lda, const void* B16, int ldb, float beta,
                float* C, int ldc, const float* alpha_dev, cudaStream_t st);
// fp32 -> fp16 operand copies (convert.cu)
int f32_to_f16_rows(int rows, int cols, const float* in, size_t ld_in, void* out, size_t ld_out, const float* scale_dev,
                    cudaStream_t st);
int f32_to_f16_transpose(int rows, int cols, const float* in, size_t ld_in, void* out, size_t ld_out, void* outT,
                         size_t ld_outT, const float* scale_dev, cudaStream_t st);
int pow2_scale_for(int rows, int cols, const float* x, size_t ld, unsigned int* absmax_ws, float* scale, int top,
                   cudaStream_t st);

// BatchNorm over rows of a (rows, F) matrix (BatchNorm1d under SequenceWise, model.py:18-33,86,196)
// training: batch stats (biased var) -> mean/invstd, running stats updated; else running stats.
// y = (x-mean)*invstd*gamma+beta ; xhat optionally stored.
int bn_rows_fwd(int rows, int F, const float* x, const float* gamma, const float* beta, float* rmean, float* rvar,
                int training, float momentum, float eps, float* y, float* xhat, float* mean_invstd /*2F*/,
                double* ws_sums /*2F doubles*/, cudaStream_t st);
// y / xhat again from saved statistics (backward recomputation)
int bn_rows_reapply(int rows, int F, const float* x, const float* gamma, const float* beta,
                    const float* mean_invstd, float* y, float* xhat, cudaStream_t st);
int transpose(int R, int C, const float* in, float* out, cudaStream_t st);
int transpose_strided(int R, int C, const float* in, size_t ldi, float* out, size_t ldo, cudaStream_t st);
// dx = gamma*invstd*(dy - mean(dy) - xhat*mean(dy*xhat)); dgamma, dbeta written.
int bn_rows_bwd(int rows, int F, const float* xhat, const float* gamma, const float* mean_invstd, const float* dy,
                float* dx, float* dgamma, float* dbeta, double* ws_sums /*2F doubles*/, cudaStream_t st);

}  // namespace ds2
