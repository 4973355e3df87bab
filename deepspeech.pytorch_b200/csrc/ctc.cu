// CTC loss + gradient w.r.t. logits (model.py:245-248: log_softmax -> CTCLoss(blank, 'sum',
// zero_infinity=True)).  Graves' alpha/beta recursions in log space:
//   kernel 1  log-softmax rows (one warp per (t,b) row)
//   kernel 2  one CTA per (utterance, sweep): the alpha sweep and the beta sweep of an utterance
//             run CONCURRENTLY in two CTAs (they are independent), states across threads, the
//             previous time step double-buffered in shared memory, one __syncthreads per step
//   kernel 3  one warp per (t,b): posterior per class summed over the 2L+1 states in a fixed order,
//             grad = softmax - posterior (fused log-softmax backward), zero for t >= in_len and for
//             infeasible utterances (zero_infinity).
// Integer indexing (extended target, skip rule, lengths) is exact; arithmetic fp32 like ATen.
#include <math_constants.h>

#include "common.cuh"

namespace ds2 {

__global__ void ctc_logsoftmax_kernel(int rows, int C, const float* __restrict__ logits, float* __restrict__ lp) {
  int row = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  int lane = threadIdx.x % 32;
  if (row >= rows) return;
  const float* x = logits + (size_t)row * C;
  float m = -CUDART_INF_F;
  for (int c = lane; c < C; c += 32) m = fmaxf(m, x[c]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += expf(x[c] - m);
  s = warp_sum(s);
  float lz = m + logf(s);
  for (int c = lane; c < C; c += 32) lp[(size_t)row * C + c] = x[c] - lz;
}

__device__ __forceinline__ float lse3(float a, float b, float c) {
  float m = fmaxf(a, fmaxf(b, c));
  if (m == -CUDART_INF_F) return -CUDART_INF_F;
  return m + logf(expf(a - m) + expf(b - m) + expf(c - m));
}

// grid (B, 2); dynamic smem: int ext[Smax] + float buf[2][Smax + 2]
// blockIdx.y = 0: alpha sweep, 1: beta sweep.  The beta recursion is the alpha recursion on the
// mirrored problem (states r = S-1-s, time reversed), so both run the same code.
// Scaled recursion: every RESCALE steps the block maximum is subtracted from all states and
// accumulated (in double) into a per-time offset, so the fp32 log-values stay O(10) instead of
// O(-nll) and keep ~1e-6 absolute precision: table[t][s] + offs[t] = log alpha_t(s).
constexpr int RESCALE = 8;

__global__ void ctc_alpha_beta_kernel(int T, int B, int C, int Smax, const float* __restrict__ lp,
                                      const int64_t* __restrict__ targets, const int32_t* __restrict__ in_len,
                                      const int32_t* __restrict__ tgt_len, int blank, float* __restrict__ alpha,
                                      float* __restrict__ beta, double* __restrict__ offs_a,
                                      double* __restrict__ offs_b, double* __restrict__ loglik) {
  extern __shared__ unsigned char smem_raw[];
  int* ext = reinterpret_cast<int*>(smem_raw);           // mirrored for the beta sweep
  float* buf = reinterpret_cast<float*>(ext + Smax);
  __shared__ float wmax[32];
  __shared__ long long off_s;
  __shared__ double shift_s;
  const int b = blockIdx.x;
  const bool is_beta = blockIdx.y == 1;
  const int Tb = in_len[b], Lb = tgt_len[b];
  const int S = 2 * Lb + 1;
  if (threadIdx.x == 0) {
    long long off = 0;
    for (int i = 0; i < b; ++i) off += tgt_len[i];
    off_s = off;
    shift_s = 0.0;
  }
  __syncthreads();
  for (int r = threadIdx.x; r < S; r += blockDim.x) {
    int s = is_beta ? S - 1 - r : r;
    ext[r] = (s & 1) ? (int)targets[off_s + (s >> 1)] : blank;
  }
  const int W = Smax + 2;  // buffer row: [0,1] = -inf guards, states at [2, 2+S)
  for (int i = threadIdx.x; i < 2 * W; i += blockDim.x) buf[i] = -CUDART_INF_F;
  __syncthreads();
  if (Tb <= 0) {
    if (!is_beta && threadIdx.x == 0) loglik[b] = (Lb == 0) ? 0.0 : -(double)CUDART_INF_F;
    return;
  }
  float* table = (is_beta ? beta : alpha) + (size_t)b * T * Smax;
  double* offs = (is_beta ? offs_b : offs_a) + (size_t)b * T;
  const size_t row_stride = (size_t)B * C;
  const float* lpb = lp + (size_t)b * C;
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32, nwarps = blockDim.x / 32;

  // The log-probability a state adds at step t does not depend on the recursion: with one state per thread (the
  // launcher's choice whenever 2L+1 <= 1024) the values of the NEXT block of 8 steps are fetched into registers while
  // the current block runs (fully unrolled, no register rotation), so the ~600-cycle L2 latency of that load — a third
  // of all stall samples in the round-1 kernel — is off the T-step dependency chain.
  const bool one = S <= (int)blockDim.x;
  const int l_own = (one && (int)threadIdx.x < S) ? ext[threadIdx.x] : blank;
  float nxt[RESCALE];
#pragma unroll
  for (int i = 0; i < RESCALE; ++i) {
    const int t_i = is_beta ? Tb - 1 - i : i;
    nxt[i] = (one && i < Tb) ? lpb[(size_t)t_i * row_stride + l_own] : 0.f;
  }
  int cur = 0;
  for (int t0 = 0; t0 < Tb; t0 += RESCALE) {
    float lpv[RESCALE];
#pragma unroll
    for (int i = 0; i < RESCALE; ++i) {
      lpv[i] = nxt[i];
      const int ta = t0 + RESCALE + i, t_a = is_beta ? Tb - 1 - ta : ta;
      nxt[i] = (one && ta < Tb) ? lpb[(size_t)t_a * row_stride + l_own] : 0.f;
    }
#pragma unroll
    for (int i = 0; i < RESCALE; ++i) {
      const int tt = t0 + i;
      if (tt >= Tb) break;                               // block-uniform
      const int t = is_beta ? Tb - 1 - tt : tt;
      const float* prev = buf + cur * W + 2;
      float* next = buf + (cur ^ 1) * W + 2;
      const float* lpt = lpb + (size_t)t * row_stride;
      float local_max = -CUDART_INF_F;
      for (int r = threadIdx.x; r < S; r += blockDim.x) {
        const int l = ext[r];
        const float lpx = one ? lpv[i] : lpt[l];
        float v;
        if (tt == 0) {
          v = (r < 2) ? lpx : -CUDART_INF_F;
        } else {
          bool skip = (r >= 2) && (l != blank) && (l != ext[r - 2]);
          float a2 = skip ? prev[r - 2] : -CUDART_INF_F;
          v = lse3(prev[r], prev[r - 1], a2) + lpx;       // prev[-1], prev[-2] are the -inf guards
        }
        next[r] = v;
        local_max = fmaxf(local_max, v);
      }
      if (i == RESCALE - 1) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) local_max = fmaxf(local_max, __shfl_xor_sync(0xffffffffu, local_max, o));
        if (lane == 0) wmax[warp] = local_max;
        __syncthreads();
        float m = -CUDART_INF_F;
        for (int w = 0; w < nwarps; ++w) m = fmaxf(m, wmax[w]);
        if (m != -CUDART_INF_F) {
          for (int r = threadIdx.x; r < S; r += blockDim.x) next[r] -= m;   // own states only
          if (threadIdx.x == 0) shift_s += (double)m;
        }
      }
      for (int r = threadIdx.x; r < S; r += blockDim.x) {
        int s = is_beta ? S - 1 - r : r;
        table[(size_t)t * Smax + s] = next[r];
      }
      if (threadIdx.x == 0) offs[t] = shift_s;
      __syncthreads();
      cur ^= 1;
    }
  }
  if (!is_beta && threadIdx.x == 0) {
    const float* last = buf + cur * W + 2;
    float a = last[S - 1], c = (S > 1) ? last[S - 2] : -CUDART_INF_F;
    float m = fmaxf(a, c);
    loglik[b] = (m == -CUDART_INF_F) ? -(double)CUDART_INF_F
                                      : shift_s + (double)m + log((double)expf(a - m) + (double)expf(c - m));
  }
}

// one warp per (t,b)
__global__ void ctc_grad_kernel(int T, int B, int C, int Smax, const float* __restrict__ lp,
                                const int64_t* __restrict__ targets, const int32_t* __restrict__ in_len,
                                const int32_t* __restrict__ tgt_len, const long long* __restrict__ tgt_off,
                                int blank, const float* __restrict__ alpha, const float* __restrict__ beta,
                                const double* __restrict__ offs_a, const double* __restrict__ offs_b,
                                const double* __restrict__ loglik, float* __restrict__ nll,
                                float* __restrict__ grad) {
  extern __shared__ float post_all[];  // warps_per_block * Cpad
  const int wpb = blockDim.x / 32;
  const int w = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int Cpad = (C + 31) / 32 * 32;
  float* post = post_all + w * Cpad;
  long long idx = (long long)blockIdx.x * wpb + w;
  if (idx >= (long long)T * B) return;
  int t = (int)(idx / B), b = (int)(idx % B);
  float* g = grad + ((size_t)t * B + b) * C;
  const double ll = loglik[b];
  const bool feasible = ll > -1e300;
  const int Tb = in_len[b];
  if (t == 0 && lane == 0) nll[b] = feasible ? (float)(-ll) : 0.f;  // zero_infinity
  if (t >= Tb || !feasible) {
    for (int c = lane; c < C; c += 32) g[c] = 0.f;
    return;
  }
  for (int c = lane; c < Cpad; c += 32) post[c] = 0.f;
  __syncwarp();
  const int S = 2 * tgt_len[b] + 1;
  const float* a = alpha + ((size_t)b * T + t) * Smax;
  const float* be = beta + ((size_t)b * T + t) * Smax;
  const float* lpr = lp + ((size_t)t * B + b) * C;
  const int64_t* tg = targets + tgt_off[b];
  // log posterior(s) = alpha + beta - lp - ll, with the big scalars combined in double first
  const float kt = (float)(offs_a[(size_t)b * T + t] + offs_b[(size_t)b * T + t] - ll);
  // lanes with the same label (every even s is the blank; repeated labels) are summed in lane order and added by
  // one lane per pass, so the gradient does not depend on the order in which shared-memory atomics would land
  for (int s0 = 0; s0 < S; s0 += 32) {
    const int s = s0 + lane;
    int l = -1;
    float e = 0.f;
    if (s < S) {
      l = (s & 1) ? (int)tg[s >> 1] : blank;
      const float v = a[s] + be[s];
      if (v != -CUDART_INF_F) e = expf(v - lpr[l] + kt);
    }
    const unsigned grp = __match_any_sync(0xffffffffu, l);
    float tot = 0.f;
    for (int k = 0; k < 32; ++k) {
      const float ek = __shfl_sync(0xffffffffu, e, k);
      if ((grp >> k) & 1u) tot += ek;
    }
    if (l >= 0 && lane == __ffs(grp) - 1) post[l] += tot;
    __syncwarp();
  }
  for (int c = lane; c < C; c += 32) g[c] = expf(lpr[c]) - post[c];
}

__global__ void ctc_offsets_kernel(int B, const int32_t* __restrict__ tgt_len, long long* __restrict__ off) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    long long o = 0;
    for (int b = 0; b < B; ++b) { off[b] = o; o += tgt_len[b]; }
  }
}

}  // namespace ds2

extern "C" {

size_t ds2_ctc_workspace_bytes(int T, int B, int C, int max_tgt_len) {
  size_t Smax = 2 * (size_t)max_tgt_len + 1;
  size_t n = ds2::align_up((size_t)T * B * C * 4, 256)      // lp
             + 2 * ds2::align_up((size_t)B * T * Smax * 4, 256)  // alpha, beta
             + 2 * ds2::align_up((size_t)B * T * 8, 256)         // per-time scale offsets (double)
             + ds2::align_up((size_t)B * 8, 256)                 // loglik (double)
             + ds2::align_up((size_t)B * 8, 256);                // target offsets
  return n;
}

int ds2_ctc_loss_fwd_bwd(int T, int B, int C, const float* logits, const int64_t* targets, const int32_t* in_len,
                         const int32_t* tgt_len, int max_tgt_len, int blank, float* nll, float* grad, void* ws,
                         size_t ws_bytes, void* stream) {
  using namespace ds2;
  DS2_REQUIRE(T > 0 && B > 0 && C > 0 && max_tgt_len >= 0 && blank >= 0 && blank < C, "ds2_ctc: bad shape");
  DS2_REQUIRE(ws_bytes >= ds2_ctc_workspace_bytes(T, B, C, max_tgt_len), "ds2_ctc: workspace too small");
  cudaStream_t st = as_stream(stream);
  const int Smax = 2 * max_tgt_len + 1;
  Arena ar(ws, ws_bytes);
  float* lp = ar.take<float>((size_t)T * B * C);
  float* alpha = ar.take<float>((size_t)B * T * Smax);
  float* beta = ar.take<float>((size_t)B * T * Smax);
  double* offs_a = ar.take<double>((size_t)B * T);
  double* offs_b = ar.take<double>((size_t)B * T);
  double* loglik = ar.take<double>(B);
  long long* off = ar.take<long long>(B);
  if (!lp || !alpha || !beta || !offs_a || !offs_b || !loglik || !off) { set_error("ds2_ctc: arena"); return DS2_ERR_WORKSPACE; }

  int rows = T * B;
  DS2_PROF("ctc", st);
  DS2_LAUNCH(ctc_logsoftmax_kernel, cdiv(rows, 8), 256, 0, st, rows, C, logits, lp);
  DS2_LAUNCH(ctc_offsets_kernel, 1, 32, 0, st, B, tgt_len, off);
  int threads = (Smax + 31) / 32 * 32;
  if (threads > 1024) threads = 1024;
  if (threads < 64) threads = 64;
  size_t smem = (size_t)Smax * 4 + 2 * ((size_t)Smax + 2) * 4;
  if (smem > 48 * 1024)
    DS2_CHECK_CUDA(cudaFuncSetAttribute(ctc_alpha_beta_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  DS2_LAUNCH(ctc_alpha_beta_kernel, dim3(B, 2), threads, smem, st, T, B, C, Smax, lp, targets, in_len, tgt_len, blank,
             alpha, beta, offs_a, offs_b, loglik);
  const int wpb = 8;
  size_t smem3 = (size_t)wpb * ((C + 31) / 32 * 32) * 4;
  DS2_LAUNCH(ctc_grad_kernel, cdiv((long long)T * B, wpb), wpb * 32, smem3, st, T, B, C, Smax, lp, targets, in_len,
             tgt_len, off, blank, alpha, beta, offs_a, offs_b, loglik, nll, grad);
  return DS2_OK;
}

}  // extern "C"
