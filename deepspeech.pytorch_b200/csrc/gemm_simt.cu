// fp32 FFMA GEMM (any shape / stride / transpose).  This is the DS2_PREC_FP32 path and the
// fallback for shapes the tcgen05 kernel does not take (tiny hidden sizes, unaligned strides).
// 128x128x16 CTA tile, 8x8 register micro-tile, smem operands stored k-major so that the
// inner product reads are conflict-free LDS.128.
#include "common.cuh"

namespace ds2 {

constexpr int BM = 128, BN = 128, BK = 16, TM = 8, TN = 8;

template <bool TA, bool TB>
__global__ void __launch_bounds__(256) gemm_simt_kernel(int M, int N, int K, float alpha,
                                                        const float* __restrict__ A, int lda,
                                                        const float* __restrict__ B, int ldb, float beta,
                                                        float* __restrict__ C, int ldc, int k_per_split,
                                                        float* __restrict__ part) {
  // gridDim.z > 1: split-K, every CTA stores alpha * its partial product into part[z] (M x N), summed by
  // splitk_reduce_kernel in a fixed order
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN + 4];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int tx = tid % 16, ty = tid / 16;  // micro-tile position: rows ty*8.., cols tx*8..
  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  const int k_begin = blockIdx.z * k_per_split;
  const int k_end = min(K, k_begin + k_per_split);
  for (int k0 = k_begin; k0 < k_end; k0 += BK) {
    // ---- stage A tile (BM x BK) into As[k][m]
#pragma unroll
    for (int e = 0; e < (BM * BK) / 256; ++e) {
      int idx = tid + e * 256;
      int m, k;
      if (TA) {  // A stored (K, M): m contiguous
        m = idx % BM;
        k = idx / BM;
      } else {   // A stored (M, K): k contiguous
        k = idx % BK;
        m = idx / BK;
      }
      int gm = m0 + m, gk = k0 + k;
      float v = 0.f;
      if (gm < M && gk < k_end) v = TA ? A[(size_t)gk * lda + gm] : A[(size_t)gm * lda + gk];
      As[k][m] = v;
    }
#pragma unroll
    for (int e = 0; e < (BN * BK) / 256; ++e) {
      int idx = tid + e * 256;
      int n, k;
      if (TB) {  // op(B)=B^T, B stored (N, K): k contiguous
        k = idx % BK;
        n = idx / BK;
      } else {   // B stored (K, N): n contiguous
        n = idx % BN;
        k = idx / BN;
      }
      int gn = n0 + n, gk = k0 + k;
      float v = 0.f;
      if (gn < N && gk < k_end) v = TB ? B[(size_t)gn * ldb + gk] : B[(size_t)gk * ldb + gn];
      Bs[k][n] = v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float a[TM], b[TN];
      *reinterpret_cast<float4*>(&a[0]) = *reinterpret_cast<const float4*>(&As[k][ty * TM]);
      *reinterpret_cast<float4*>(&a[4]) = *reinterpret_cast<const float4*>(&As[k][ty * TM + 4]);
      *reinterpret_cast<float4*>(&b[0]) = *reinterpret_cast<const float4*>(&Bs[k][tx * TN]);
      *reinterpret_cast<float4*>(&b[4]) = *reinterpret_cast<const float4*>(&Bs[k][tx * TN + 4]);
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    int gm = m0 + ty * TM + i;
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      int gn = n0 + tx * TN + j;
      if (gn >= N) continue;
      float* c = C + (size_t)gm * ldc + gn;
      float v = alpha * acc[i][j];
      if (gridDim.z > 1) {
        part[((size_t)blockIdx.z * M + gm) * N + gn] = v;
      } else {
        if (beta != 0.f) v += beta * (*c);
        *c = v;
      }
    }
  }
}

// C = beta * C + sum_z part[z], z in increasing order
__global__ void splitk_reduce_kernel(int M, int N, int splits, const float* __restrict__ part, float beta,
                                     float* __restrict__ C, int ldc) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n = (size_t)M * N;
  if (i >= n) return;
  float v = 0.f;
  for (int z = 0; z < splits; ++z) v += part[(size_t)z * n + i];
  float* c = C + (i / N) * ldc + (i % N);
  *c = (beta == 0.f) ? v : fmaf(beta, *c, v);
}

// K split for long reductions onto few output tiles (weight gradients); returns the number of splits (1: none)
static int simt_splits(int M, int N, int K, int* k_per_split) {
  *k_per_split = K > 0 ? K : 1;
  const int tiles = cdiv(N, BN) * cdiv(M, BM);
  if (tiles >= 74 || K < 2048) return 1;
  int splits = 148 / tiles;
  if (splits > K / 256) splits = K / 256;
  if (splits <= 1) return 1;
  const int kps = cdiv(cdiv(K, splits), BK) * BK, gz = cdiv(K, kps);
  if (gz > 1) *k_per_split = kps;
  return gz > 1 ? gz : 1;
}

size_t gemm_simt_workspace_bytes(int M, int N, int K) {
  int kps;
  const int gz = simt_splits(M, N, K, &kps);
  return gz > 1 ? (size_t)gz * M * N * sizeof(float) : 0;
}

int gemm_simt(int transA, int transB, int M, int N, int K, float alpha, const float* A, int lda, const float* B,
              int ldb, float beta, float* C, int ldc, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (M <= 0 || N <= 0) return DS2_OK;
  dim3 grid(cdiv(N, BN), cdiv(M, BM));
  int k_per_split = K > 0 ? K : 1;
  float* part = nullptr;
  {  // long reduction, few output tiles (weight gradients): split K over the SMs when the workspace holds the partials
    int kps;
    const int gz = simt_splits(M, N, K, &kps);
    if (gz > 1 && ws && ws_bytes >= gemm_simt_workspace_bytes(M, N, K)) {
      k_per_split = kps;
      grid.z = gz;
      part = static_cast<float*>(ws);
    }
  }
  if (transA) {
    if (transB) DS2_LAUNCH((gemm_simt_kernel<true, true>), grid, 256, 0, st, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, k_per_split,
               part);
    else DS2_LAUNCH((gemm_simt_kernel<true, false>), grid, 256, 0, st, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, k_per_split,
               part);
  } else {
    if (transB) DS2_LAUNCH((gemm_simt_kernel<false, true>), grid, 256, 0, st, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, k_per_split,
               part);
    else DS2_LAUNCH((gemm_simt_kernel<false, false>), grid, 256, 0, st, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, k_per_split,
               part);
  }
  if (part) DS2_LAUNCH(splitk_reduce_kernel, cdiv((long long)M * N, 256), 256, 0, st, M, N, (int)grid.z, part, beta, C, ldc);
  return DS2_OK;
}

}  // namespace ds2

extern "C" {
size_t ds2_gemm_workspace_bytes(int transA, int transB, int M, int N, int K) {
  const size_t tc = ds2::gemm_tc_workspace_bytes(transA, transB, M, N, K), simt = ds2::gemm_simt_workspace_bytes(M, N, K);
  return tc > simt ? tc : simt;
}

int ds2_gemm(int transA, int transB, int M, int N, int K, float alpha, const float* A, int lda, const float* B,
             int ldb, float beta, float* C, int ldc, void* ws, size_t ws_bytes, void* stream) {
  DS2_REQUIRE(M >= 0 && N >= 0 && K >= 0 && A && B && C, "ds2_gemm: bad arguments");
  cudaStream_t st = ds2::as_stream(stream);
  if (ds2::tensor_core_mode()) {
    int r = ds2::gemm_tc(transA, transB, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, ws, ws_bytes, st);
    if (r <= 0) return r;  // 0 = done, <0 = error, 1 = shape not eligible -> FFMA kernel
  }
  return ds2::gemm_simt(transA, transB, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, ws, ws_bytes, st);
}

// fp16-operand GEMM of the precision-16 mode, exported for tests / the roofline bench: A16 (M,K), B16 (N,K) K-major
// halfs on the device, C fp32.  DS2_ERR_INVALID when the shape / alignment is not eligible (no fallback here).
int ds2_gemm_f16(int M, int N, int K, float alpha, const void* A16, int lda, const void* B16, int ldb, float beta,
                 float* C, int ldc, void* stream) {
  DS2_REQUIRE(M > 0 && N > 0 && K > 0 && A16 && B16 && C, "ds2_gemm_f16: bad arguments");
  int r = ds2::gemm_tc_f16(M, N, K, alpha, A16, lda, B16, ldb, beta, C, ldc, nullptr, ds2::as_stream(stream));
  DS2_REQUIRE(r != 1, "ds2_gemm_f16: shape %dx%dx%d / alignment not eligible for the tcgen05 fp16 kernel", M, N, K);
  return r;
}
}
