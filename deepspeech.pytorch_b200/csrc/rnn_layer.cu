// One BatchRNN layer (model.py:80-102): [BatchNorm1d over T*B rows] -> input projection GEMM ->
// recurrent sweep per direction with per-utterance length masking (replaces pack/pad, SURVEY §2b K8)
// -> sum of directions.  Backward: reverse sweep producing gate gradients in place of the saved
// gate activations, then three dense GEMMs (dW_ih, dW_hh, dX) and the BatchNorm backward.
//
// This file holds the host orchestration and the generic FFMA step kernels (any H, any B): one
// launch per time step covering both directions.  rnn_persistent_tc.cu provides the tcgen05
// persistent sweep that replaces the step launches when the shape is eligible.
//
// reserve layout (floats):  gates (T,B,D,G*H) | hseq (D,T,B,H) | aux (D,T,B,H: LSTM cell states /
//                           GRU W_hn h + b_hn; absent for tanh) | bn mean,invstd (2*In)
#include <cuda_fp16.h>

#include <mutex>
#include <unordered_set>

#include "common.cuh"
#include "rnn_cells.cuh"
#include "rnn_common.cuh"

namespace ds2 {

constexpr int UT = 8;   // hidden units per CTA
constexpr int KC = 64;  // reduction chunk staged in shared memory

__device__ __forceinline__ int gates_per(int rnn) { return rnn == DS2_RNN_LSTM ? 4 : (rnn == DS2_RNN_GRU ? 3 : 1); }

// grid (ceil(H/UT), D), block (32, UT)
template <int RNN>
__global__ void __launch_bounds__(32 * UT) rnn_step_fwd_kernel(SeqArgs a, int step) {
  constexpr int G = RNN == DS2_RNN_LSTM ? 4 : (RNN == DS2_RNN_GRU ? 3 : 1);
  __shared__ float hs[32][KC + 1];
  __shared__ float ws[G * UT][KC + 1];
  const int d = blockIdx.y, T = a.T, B = a.B, H = a.H, D = a.D;
  const int t = d == 0 ? step : T - 1 - step;
  const int tp = d == 0 ? t - 1 : t + 1;
  const bool tp_in = tp >= 0 && tp < T;
  const int lane = threadIdx.x, uy = threadIdx.y, tid = uy * 32 + lane;
  const int u0 = blockIdx.x * UT, u = u0 + uy;
  const float* __restrict__ W = a.w_hh[d];
  const float* hprev = a.hseq + ((size_t)d * T + (tp_in ? tp : 0)) * B * H;
  const float* cprev = a.aux ? a.aux + ((size_t)d * T + (tp_in ? tp : 0)) * B * H : nullptr;
  const int GH = G * H;

  for (int bt = 0; bt < (B + 31) / 32; ++bt) {
    const int b = bt * 32 + lane;
    float acc[G];
#pragma unroll
    for (int g = 0; g < G; ++g) acc[g] = 0.f;
    for (int k0 = 0; k0 < H; k0 += KC) {
      for (int idx = tid; idx < 32 * KC; idx += 32 * UT) {
        int kk = idx % KC, bb = idx / KC, gb = bt * 32 + bb, gk = k0 + kk;
        float v = 0.f;
        if (gb < B && gk < H) {
          bool pin = tp_in && (d == 0 || tp < a.len[gb]);
          v = pin ? hprev[(size_t)gb * H + gk] : (a.h0 ? a.h0[((size_t)d * B + gb) * H + gk] : 0.f);
        }
        hs[bb][kk] = v;
      }
      for (int idx = tid; idx < G * UT * KC; idx += 32 * UT) {
        int kk = idx % KC, rr = idx / KC, g = rr / UT, gu = u0 + rr % UT, gk = k0 + kk;
        ws[rr][kk] = (gu < H && gk < H) ? W[((size_t)g * H + gu) * H + gk] : 0.f;
      }
      __syncthreads();
#pragma unroll 8
      for (int kk = 0; kk < KC; ++kk) {
        float hv = hs[lane][kk];
#pragma unroll
        for (int g = 0; g < G; ++g) acc[g] = fmaf(hv, ws[g * UT + uy][kk], acc[g]);
      }
      __syncthreads();
    }
    if (b < B && u < H) {
      const bool valid = t < a.len[b];
      const bool pin = tp_in && (d == 0 || tp < a.len[b]);
      float* gp = a.gates + (((size_t)t * B + b) * D + d) * GH + u;
      float* hp = a.hseq + (((size_t)d * T + t) * B + b) * H + u;
      float* xp = a.aux ? a.aux + (((size_t)d * T + t) * B + b) * H + u : nullptr;
      const float* bi = a.b_ih[d] + u;
      const float* bh = a.b_hh[d] + u;
      if (!valid) {
        *hp = 0.f;
        if (xp) *xp = 0.f;
#pragma unroll
        for (int g = 0; g < G; ++g) gp[g * H] = 0.f;
      } else if constexpr (RNN == DS2_RNN_LSTM) {
        float c_prev = pin ? cprev[(size_t)b * H + u] : (a.c0 ? a.c0[((size_t)d * B + b) * H + u] : 0.f);
        LstmFwd r = lstm_cell_fwd(gp[0] + bi[0] + acc[0] + bh[0], gp[H] + bi[H] + acc[1] + bh[H],
                                  gp[2 * H] + bi[2 * H] + acc[2] + bh[2 * H],
                                  gp[3 * H] + bi[3 * H] + acc[3] + bh[3 * H], c_prev);
        gp[0] = r.i; gp[H] = r.f; gp[2 * H] = r.g; gp[3 * H] = r.o;
        *hp = r.h;
        *xp = r.c;
      } else if constexpr (RNN == DS2_RNN_GRU) {
        float h_prev = pin ? hprev[(size_t)b * H + u] : (a.h0 ? a.h0[((size_t)d * B + b) * H + u] : 0.f);
        float hn = acc[2] + bh[2 * H];
        GruFwd r = gru_cell_fwd(gp[0] + bi[0], gp[H] + bi[H], gp[2 * H] + bi[2 * H], acc[0] + bh[0],
                                acc[1] + bh[H], hn, h_prev);
        gp[0] = r.r; gp[H] = r.z; gp[2 * H] = r.n;
        *hp = r.h;
        *xp = hn;
      } else {
        float h = tanhf(gp[0] + bi[0] + acc[0] + bh[0]);
        gp[0] = h;
        *hp = h;
      }
    }
  }
}

// Backward step.  w_hh[d] here is the TRANSPOSED recurrent matrix (H, G*H).
template <int RNN>
__global__ void __launch_bounds__(32 * UT) rnn_step_bwd_kernel(SeqArgs a, int step) {
  constexpr int G = RNN == DS2_RNN_LSTM ? 4 : (RNN == DS2_RNN_GRU ? 3 : 1);
  __shared__ float gs[32][KC + 1];
  __shared__ float ws[UT][KC + 1];
  const int d = blockIdx.y, T = a.T, B = a.B, H = a.H, D = a.D;
  const int t = d == 0 ? T - 1 - step : step;
  const int tn = d == 0 ? t + 1 : t - 1;   // processed just before (later in this direction's time)
  const int tp = d == 0 ? t - 1 : t + 1;   // source of the previous state in the forward sweep
  const bool tn_in = tn >= 0 && tn < T, tp_in = tp >= 0 && tp < T;
  const int lane = threadIdx.x, uy = threadIdx.y, tid = uy * 32 + lane;
  const int u0 = blockIdx.x * UT, u = u0 + uy;
  const int GH = G * H;
  const float* __restrict__ WT = a.w_hh[d];

  for (int bt = 0; bt < (B + 31) / 32; ++bt) {
    const int b = bt * 32 + lane;
    float acc = 0.f;
    if (tn_in) {
      for (int k0 = 0; k0 < GH; k0 += KC) {
        for (int idx = tid; idx < 32 * KC; idx += 32 * UT) {
          int kk = idx % KC, bb = idx / KC, gb = bt * 32 + bb, row = k0 + kk;
          float v = 0.f;
          if (gb < B && row < GH) {
            if (RNN == DS2_RNN_GRU && row >= 2 * H)
              v = a.aux[(((size_t)d * T + tn) * B + gb) * H + (row - 2 * H)];   // dGh_n
            else
              v = a.gates[(((size_t)tn * B + gb) * D + d) * GH + row];
          }
          gs[bb][kk] = v;
        }
        for (int idx = tid; idx < UT * KC; idx += 32 * UT) {
          int kk = idx % KC, rr = idx / KC, gu = u0 + rr, row = k0 + kk;
          ws[rr][kk] = (gu < H && row < GH) ? WT[(size_t)gu * GH + row] : 0.f;
        }
        __syncthreads();
#pragma unroll 8
        for (int kk = 0; kk < KC; ++kk) acc = fmaf(gs[lane][kk], ws[uy][kk], acc);
        __syncthreads();
      }
    }
    if (b < B && u < H) {
      const bool valid = t < a.len[b];
      const bool pin = tp_in && (d == 0 || tp < a.len[b]);
      float* gp = a.gates + (((size_t)t * B + b) * D + d) * GH + u;
      const size_t si = (((size_t)d * T + t) * B + b) * H + u;
      const size_t sp = (((size_t)d * T + (tp_in ? tp : 0)) * B + b) * H + u;
      float* carry = a.carry ? a.carry + ((size_t)d * B + b) * H + u : nullptr;
      if (!valid) {
#pragma unroll
        for (int g = 0; g < G; ++g) gp[g * H] = 0.f;
        if (RNN == DS2_RNN_GRU) a.aux[si] = 0.f;
      } else {
        float dh = a.dy[((size_t)t * B + b) * H + u] + acc;
        if constexpr (RNN == DS2_RNN_LSTM) {
          float c_prev = pin ? a.aux[sp] : 0.f;
          LstmBwd r = lstm_cell_bwd(gp[0], gp[H], gp[2 * H], gp[3 * H], a.aux[si], c_prev, dh, *carry);
          gp[0] = r.di; gp[H] = r.df; gp[2 * H] = r.dg; gp[3 * H] = r.d_o;
          *carry = r.dc_prev;
        } else if constexpr (RNN == DS2_RNN_GRU) {
          float h_prev = pin ? a.hseq[sp] : 0.f;
          dh += *carry;
          GruBwd r = gru_cell_bwd(gp[0], gp[H], gp[2 * H], a.aux[si], h_prev, dh);
          gp[0] = r.dr; gp[H] = r.dz; gp[2 * H] = r.dxn;
          a.aux[si] = r.dhn;
          *carry = r.dh_prev;
        } else {
          float h = a.hseq[si];
          gp[0] = dh * (1.f - h * h);
        }
      }
    }
  }
}

__global__ void sum_dirs_kernel(size_t n, int D, const float* __restrict__ hseq, float* __restrict__ y) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) y[i] = D == 2 ? hseq[i] + hseq[n + i] : hseq[i];
}

// hn[d,b,u] = state after the last valid step (fwd: t=len-1, reverse: t=0); h0 when len == 0
__global__ void final_state_kernel(int T, int B, int H, int D, const int32_t* __restrict__ len,
                                   const float* __restrict__ seq, const float* __restrict__ init,
                                   float* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)D * B * H) return;
  int u = (int)(i % H), b = (int)((i / H) % B), d = (int)(i / ((size_t)H * B));
  int L = min(len[b], T);
  float v;
  if (L <= 0) v = init ? init[i] : 0.f;
  else v = seq[(((size_t)d * T + (d == 0 ? L - 1 : 0)) * B + b) * H + u];
  out[i] = v;
}

// dst[f] = sum_r src[r*ld + f]   (dst zeroed by the caller); grid (ceil(F/32), chunks), block (32,8)
__global__ void colsum_strided_kernel(int rows, int F, const float* __restrict__ src, size_t ld,
                                      float* __restrict__ dst) {
  __shared__ float red[8][33];
  int f = blockIdx.x * 32 + threadIdx.x;
  int per = cdiv_dev(rows, gridDim.y), r0 = blockIdx.y * per, r1 = min(rows, r0 + per);
  float acc = 0.f;
  if (f < F)
    for (int r = r0 + threadIdx.y; r < r1; r += 8) acc += src[(size_t)r * ld + f];
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && f < F) {
    for (int i = 1; i < 8; ++i) acc += red[i][threadIdx.x];
    atomicAdd(&dst[f], acc);
  }
}

static int colsum(int rows, int F, const float* src, size_t ld, float* dst, cudaStream_t st) {
  DS2_CHECK_CUDA(cudaMemsetAsync(dst, 0, sizeof(float) * F, st));
  int chunks = rows / 256;
  chunks = chunks < 1 ? 1 : (chunks > 64 ? 64 : chunks);
  DS2_LAUNCH(colsum_strided_kernel, dim3(cdiv(F, 32), chunks), dim3(32, 8), 0, st, rows, F, src, ld, dst);
  return DS2_OK;
}

static inline int num_gates(int rnn) { return rnn == DS2_RNN_LSTM ? 4 : (rnn == DS2_RNN_GRU ? 3 : 1); }

struct Reserve {
  float *gates, *hseq, *aux, *bnstats;
  __half* wT16;   // (D, H, G*H) fp16 W_hh^T, written by a tensor-core-mode training forward for the backward sweep
  size_t total;
};
static Reserve carve_reserve(const ds2_rnn_desc* d, float* base) {
  const size_t D = d->bidirectional ? 2 : 1, G = num_gates(d->rnn_type);
  const size_t TB = (size_t)d->T * d->B;
  Reserve r;
  size_t off = 0;
  r.gates = base + off; off += TB * D * G * d->H;
  r.hseq = base + off; off += D * TB * d->H;
  if (d->rnn_type != DS2_RNN_TANH) { r.aux = base + off; off += D * TB * d->H; } else r.aux = nullptr;
  r.bnstats = base + off; off += 2 * (size_t)d->In;
  off = (off + 3) & ~(size_t)3;                           // 16-byte aligned (TMA source)
  r.wT16 = reinterpret_cast<__half*>(base + off); off += (D * G * d->H * d->H + 1) / 2;
  r.total = off;
  return r;
}

// Which reserve buffers hold a valid fp16 W_hh^T (the forward pass that wrote it registers the pointer, the backward
// pass that consumes the reserve removes it): a backward without the copy simply converts the weights itself.
static std::mutex g_wT16_mu;
static std::unordered_set<const void*> g_wT16_valid;
static void wT16_set(const void* reserve, bool valid) {
  std::lock_guard<std::mutex> lk(g_wT16_mu);
  if (valid) g_wT16_valid.insert(reserve); else g_wT16_valid.erase(reserve);
}
static bool wT16_take(const void* reserve) {
  std::lock_guard<std::mutex> lk(g_wT16_mu);
  return g_wT16_valid.erase(reserve) > 0;
}

// lazily materialised fp32 W_hh^T of the backward pass (SeqArgs::fill_w_hh)
struct FillWhh {
  int GH, H, D, done;
  const float* const* w_hh;
  float* wT[2];
};
static int fill_w_hh_cb(void* ctx, void* stream) {
  FillWhh* f = static_cast<FillWhh*>(ctx);
  if (f->done) return DS2_OK;
  for (int dir = 0; dir < f->D; ++dir) {
    int rc = transpose(f->GH, f->H, f->w_hh[dir], f->wT[dir], static_cast<cudaStream_t>(stream));
    if (rc) return rc;
  }
  f->done = 1;
  return DS2_OK;
}

// tcgen05 persistent sweeps (rnn_persistent_tc.cu).  Return 1 when the shape is not eligible.
int rnn_sweep_fwd_tc(int rnn, const SeqArgs& a, void* ws, size_t ws_bytes, cudaStream_t st);
int rnn_sweep_bwd_tc(int rnn, const SeqArgs& a, void* ws, size_t ws_bytes, cudaStream_t st);
size_t rnn_sweep_tc_workspace_bytes(int rnn, int T, int B, int H, int D);

static int sweep_fwd(int rnn, const SeqArgs& a, cudaStream_t st) {
  dim3 grid(cdiv(a.H, UT), a.D), block(32, UT);
  for (int s = 0; s < a.T; ++s) {
    if (rnn == DS2_RNN_LSTM) DS2_LAUNCH(rnn_step_fwd_kernel<DS2_RNN_LSTM>, grid, block, 0, st, a, s);
    else if (rnn == DS2_RNN_GRU) DS2_LAUNCH(rnn_step_fwd_kernel<DS2_RNN_GRU>, grid, block, 0, st, a, s);
    else DS2_LAUNCH(rnn_step_fwd_kernel<DS2_RNN_TANH>, grid, block, 0, st, a, s);
  }
  return DS2_OK;
}
static int sweep_bwd(int rnn, const SeqArgs& a, cudaStream_t st) {
  dim3 grid(cdiv(a.H, UT), a.D), block(32, UT);
  for (int s = 0; s < a.T; ++s) {
    if (rnn == DS2_RNN_LSTM) DS2_LAUNCH(rnn_step_bwd_kernel<DS2_RNN_LSTM>, grid, block, 0, st, a, s);
    else if (rnn == DS2_RNN_GRU) DS2_LAUNCH(rnn_step_bwd_kernel<DS2_RNN_GRU>, grid, block, 0, st, a, s);
    else DS2_LAUNCH(rnn_step_bwd_kernel<DS2_RNN_TANH>, grid, block, 0, st, a, s);
  }
  return DS2_OK;
}

}  // namespace ds2

extern "C" {
using namespace ds2;

size_t ds2_rnn_reserve_floats(const ds2_rnn_desc* d) {
  if (!d) return 0;
  return carve_reserve(d, nullptr).total;
}

size_t ds2_rnn_workspace_bytes(const ds2_rnn_desc* d) {
  if (!d) return 0;
  const size_t D = d->bidirectional ? 2 : 1, G = num_gates(d->rnn_type);
  const size_t TB = (size_t)d->T * d->B, GH = G * d->H;
  size_t n = 0;
  n += 3 * align_up(TB * d->In * 4, 256);                 // xbn, xhat, dxbn
  n += align_up(2 * (size_t)d->In * 8, 256);              // BN double sums
  n += D * align_up(GH * d->H * 4, 256);                  // W_hh^T per direction
  n += align_up(D * (size_t)d->B * d->H * 4, 256);        // carry
  if (f16_gemm_mode()) {
    // precision-16 operand copies: x16, W16 (fwd); dG16, dG16^T, x16^T, h16^T, aux16^T, W16^T, scale (bwd)
    n += 2 * align_up(TB * d->In * 2, 256) + 2 * align_up(D * GH * d->In * 2, 256) + 2 * align_up(TB * D * GH * 2, 256) +
         2 * align_up(D * d->H * TB * 2, 256) + 512;
  }
  n += rnn_sweep_tc_workspace_bytes(d->rnn_type, d->T, d->B, d->H, (int)D);
  {  // one slot shared by every ds2_gemm of the layer: the largest need among its shapes (the FFMA path keeps its
     // split-K partials there; a narrower dW_hh splits K more ways than dW_ih)
    const int T = d->T, B = d->B, In = d->In, H = d->H, gh = (int)GH, tb = (int)TB, kr = (T - 1) * B;
    const int rows_x = d->rnn_type == DS2_RNN_GRU ? 2 * H : gh;
    const size_t need[] = {ds2_gemm_workspace_bytes(0, 1, tb, gh, In), ds2_gemm_workspace_bytes(1, 0, gh, In, tb),
                           ds2_gemm_workspace_bytes(1, 0, rows_x, H, kr), ds2_gemm_workspace_bytes(1, 0, H, H, kr),
                           ds2_gemm_workspace_bytes(0, 0, tb, In, gh)};
    size_t g = 0;
    for (size_t v : need) g = v > g ? v : g;
    n += g;
  }
  return n + 4096;
}

static int check_desc(const ds2_rnn_desc* d) {
  DS2_REQUIRE(d, "rnn: null descriptor");
  DS2_REQUIRE(d->rnn_type >= DS2_RNN_LSTM && d->rnn_type <= DS2_RNN_TANH, "rnn: unknown rnn_type %d", d->rnn_type);
  DS2_REQUIRE(d->T > 0 && d->B > 0 && d->In > 0 && d->H > 0, "rnn: bad shape T=%d B=%d In=%d H=%d", d->T, d->B,
              d->In, d->H);
  return DS2_OK;
}

int ds2_rnn_layer_fwd(const ds2_rnn_desc* d, const float* x, const int32_t* len, const float* bn_gamma,
                      const float* bn_beta, float* bn_rmean, float* bn_rvar, const float* const* w_ih,
                      const float* const* w_hh, const float* const* b_ih, const float* const* b_hh, const float* h0,
                      const float* c0, float* y, float* hn, float* cn, float* reserve, void* ws, size_t ws_bytes,
                      void* stream) {
  int rc = check_desc(d);
  if (rc) return rc;
  DS2_REQUIRE(ws_bytes >= ds2_rnn_workspace_bytes(d), "rnn fwd: workspace too small");
  cudaStream_t st = as_stream(stream);
  const int D = d->bidirectional ? 2 : 1, G = num_gates(d->rnn_type), T = d->T, B = d->B, In = d->In, H = d->H;
  const int TB = T * B, GH = G * H;
  Reserve R = carve_reserve(d, reserve);
  Arena ar(ws, ws_bytes);
  const float* xin = x;
  if (bn_gamma) {
    float* xbn = ar.take<float>((size_t)TB * In);
    double* sums = ar.take<double>(2 * (size_t)In);
    rc = bn_rows_fwd(TB, In, x, bn_gamma, bn_beta, bn_rmean, bn_rvar, d->training, d->bn_momentum, d->bn_eps, xbn,
                     nullptr, R.bnstats, sums, st);
    if (rc) return rc;
    xin = xbn;
  }
  void* gws = ar.base + ar.off;
  size_t gws_bytes = ar.cap - ar.off;
  // input projection for every time step and both directions: gates[:, d*GH:(d+1)*GH] = xin . W_ih[d]^T
  {
    DS2_PROF("rnn_fwd_proj_gemm", st);
    bool done = false;
    if (f16_gemm_mode() && B % 8 == 0 && In % 8 == 0 && H % 8 == 0) {
      // precision 16: fp16 copies of the layer input and of both directions' W_ih (stacked: one N = D*G*H GEMM)
      __half* x16 = ar.take<__half>((size_t)TB * In);
      __half* w16 = ar.take<__half>((size_t)D * GH * In);
      if (x16 && w16) {
        rc = f32_to_f16_rows(TB, In, xin, In, x16, In, nullptr, st);
        if (rc) return rc;
        for (int dir = 0; dir < D; ++dir) {
          rc = f32_to_f16_rows(GH, In, w_ih[dir], In, w16 + (size_t)dir * GH * In, In, nullptr, st);
          if (rc) return rc;
        }
        rc = gemm_tc_f16(TB, D * GH, In, 1.f, x16, In, w16, In, 0.f, R.gates, D * GH, nullptr, st);
        if (rc < 0) return rc;
        done = rc == 0;
      }
      gws = ar.base + ar.off;
      gws_bytes = ar.cap - ar.off;
    }
    for (int dir = 0; dir < D && !done; ++dir) {
      rc = ds2_gemm(0, 1, TB, GH, In, 1.f, xin, In, w_ih[dir], In, 0.f, R.gates + (size_t)dir * GH, D * GH, gws,
                    gws_bytes, stream);
      if (rc) return rc;
    }
  }
  SeqArgs a{};
  a.T = T; a.B = B; a.H = H; a.D = D; a.G = G; a.len = len;
  a.gates = R.gates; a.hseq = R.hseq; a.aux = R.aux;
  for (int dir = 0; dir < D; ++dir) { a.w_hh[dir] = w_hh[dir]; a.b_ih[dir] = b_ih[dir]; a.b_hh[dir] = b_hh[dir]; }
  a.h0 = h0; a.c0 = c0; a.training = d->training;
  {
    DS2_PROF("rnn_fwd_sweep", st);
    rc = 1;
    if (tensor_core_mode()) {
      rc = rnn_sweep_fwd_tc(d->rnn_type, a, gws, gws_bytes, st);
      if (rc == 1) note_fallback("forward sweep", d->rnn_type, T, B, H, D);
    }
    if (rc == 1) rc = sweep_fwd(d->rnn_type, a, st);
    if (rc) return rc;
  }
  // fp16 W_hh^T for the backward sweep of this step (the weights cannot change in between): one pass here instead of a
  // transpose + a conversion on the backward critical path; on the side stream when there is one
  wT16_set(reserve, false);
  if (d->training && tensor_core_mode() && H % 8 == 0) {
    cudaStream_t side = as_stream(g_side_stream.load());
    cudaStream_t cst = st;
    if (side) {
      rc = side_fork(st, side);
      if (rc) return rc;
      cst = side;
    }
    for (int dir = 0; dir < D; ++dir) {
      rc = f32_to_f16_transpose(GH, H, w_hh[dir], (size_t)H, nullptr, 0, R.wT16 + (size_t)dir * H * GH, (size_t)GH,
                                nullptr, cst);
      if (rc) return rc;
    }
    if (side) {
      rc = side_mark_workspace(reserve, side);
      if (rc) return rc;
    }
    wT16_set(reserve, true);
  }
  size_t n = (size_t)TB * H;
  int blocks = (int)((n + 1023) / 1024);
  blocks = blocks > 148 * 16 ? 148 * 16 : blocks;
  DS2_LAUNCH(sum_dirs_kernel, blocks, 256, 0, st, n, D, R.hseq, y);
  if (hn) DS2_LAUNCH(final_state_kernel, cdiv((long long)D * B * H, 256), 256, 0, st, T, B, H, D, len, R.hseq, h0, hn);
  if (cn && d->rnn_type == DS2_RNN_LSTM)
    DS2_LAUNCH(final_state_kernel, cdiv((long long)D * B * H, 256), 256, 0, st, T, B, H, D, len, R.aux, c0, cn);
  return DS2_OK;
}

int ds2_rnn_layer_bwd(const ds2_rnn_desc* d, const float* x, const int32_t* len, const float* bn_gamma,
                      const float* bn_beta, const float* const* w_ih, const float* const* w_hh,
                      const float* const* b_ih, const float* const* b_hh, const float* dy, float* reserve, float* dx,
                      float* dbn_gamma, float* dbn_beta, float* const* dw_ih, float* const* dw_hh,
                      float* const* db_ih, float* const* db_hh, void* ws, size_t ws_bytes, void* stream) {
  int rc = check_desc(d);
  if (rc) return rc;
  DS2_REQUIRE(ws_bytes >= ds2_rnn_workspace_bytes(d), "rnn bwd: workspace too small");
  cudaStream_t st = as_stream(stream);
  cudaStream_t side = as_stream(g_side_stream.load());
  if (side) {   // deferred weight-gradient GEMMs of an earlier layer may still read operand copies in this workspace
    rc = side_wait_for_workspace(ws, st);
    if (rc) return rc;
  }
  const int D = d->bidirectional ? 2 : 1, G = num_gates(d->rnn_type), T = d->T, B = d->B, In = d->In, H = d->H;
  const int TB = T * B, GH = G * H;
  Reserve R = carve_reserve(d, reserve);
  Arena ar(ws, ws_bytes);
  float *xbn = nullptr, *xhat = nullptr, *dxbn = nullptr;
  double* sums = nullptr;
  if (bn_gamma) {
    xbn = ar.take<float>((size_t)TB * In);
    xhat = ar.take<float>((size_t)TB * In);
    dxbn = ar.take<float>((size_t)TB * In);
    sums = ar.take<double>(2 * (size_t)In);
  }
  float* wT[2] = {nullptr, nullptr};
  for (int dir = 0; dir < D; ++dir) wT[dir] = ar.take<float>((size_t)GH * H);
  float* carry = ar.take<float>((size_t)D * B * H);
  void* gws = ar.base + ar.off;
  size_t gws_bytes = ar.cap - ar.off;

  // W_hh^T: fp16 copy from the forward pass when there is one (the fp32 transposes are then made only if a path that
  // streams fp32 weights is taken), otherwise transposed here
  FillWhh fill{GH, H, D, 0, w_hh, {wT[0], wT[1]}};
  const bool have_wT16 = tensor_core_mode() && wT16_take(reserve);
  if (have_wT16) {
    if (side) {   // written on the side stream by the forward pass
      rc = side_wait_for_workspace(reserve, st);
      if (rc) return rc;
    }
  } else {
    rc = fill_w_hh_cb(&fill, st);
    if (rc) return rc;
  }
  DS2_CHECK_CUDA(cudaMemsetAsync(carry, 0, sizeof(float) * (size_t)D * B * H, st));
  SeqArgs a{};
  a.T = T; a.B = B; a.H = H; a.D = D; a.G = G; a.len = len;
  a.gates = R.gates; a.hseq = R.hseq; a.aux = R.aux;
  for (int dir = 0; dir < D; ++dir) { a.w_hh[dir] = wT[dir]; a.b_ih[dir] = b_ih[dir]; a.b_hh[dir] = b_hh[dir]; }
  a.dy = dy; a.carry = carry; a.training = 1;
  a.fill_w_hh = fill_w_hh_cb; a.fill_w_hh_ctx = &fill;
  if (have_wT16)
    for (int dir = 0; dir < D; ++dir) a.w_hhT16[dir] = R.wT16 + (size_t)dir * H * GH;
  // bias gradients are column sums of the gate gradients: the tensor-core sweep can accumulate them on the fly
  int dbias_done = 0;
  const bool gru_l = d->rnn_type == DS2_RNN_GRU;
  for (int dir = 0; dir < D; ++dir) {
    a.dbias[dir] = db_ih[dir];
    a.dbias_hn[dir] = gru_l ? db_hh[dir] + 2 * H : nullptr;
    DS2_CHECK_CUDA(cudaMemsetAsync(db_ih[dir], 0, sizeof(float) * GH, st));
    if (gru_l) DS2_CHECK_CUDA(cudaMemsetAsync(db_hh[dir] + 2 * H, 0, sizeof(float) * H, st));
  }
  a.dbias_done = &dbias_done;
  // ---- precision 16: scaled fp16 copies of the gate gradients (row-major for dX, transposed for the weight
  // gradients), transposed fp16 copies of the layer input / the hidden sequence / W_ih; every GEMM K-major fp16.
  // The split-K sweep writes the gate-gradient copies itself (scale from max|dY|); other sweeps leave f16_done = 0
  // and the copies are converted from the fp32 gate gradients afterwards.
  const bool gru = d->rnn_type == DS2_RNN_GRU;
  __half *dG16 = nullptr, *dG16T = nullptr, *x16T = nullptr, *h16T = nullptr, *aux16T = nullptr, *w16T = nullptr;
  float* scale = nullptr;
  int f16_done = 0;
  bool f16 = f16_gemm_mode() && B % 8 == 0 && In % 8 == 0 && H % 8 == 0 && TB >= 128;
  if (f16) {
    const size_t DGH = (size_t)D * GH;
    dG16 = ar.take<__half>((size_t)TB * DGH);
    dG16T = ar.take<__half>((size_t)TB * DGH);
    x16T = ar.take<__half>((size_t)TB * In);
    h16T = ar.take<__half>((size_t)D * H * TB);
    aux16T = gru ? ar.take<__half>((size_t)D * H * TB) : nullptr;
    w16T = ar.take<__half>((size_t)In * DGH);
    scale = ar.take<float>(16);
    f16 = dG16 && dG16T && x16T && h16T && w16T && scale && (!gru || aux16T);
    gws = ar.base + ar.off;
    gws_bytes = ar.cap - ar.off;
  }
  if (f16) {
    rc = pow2_scale_for(TB, H, dy, (size_t)H, reinterpret_cast<unsigned int*>(scale + 8), scale, 5, st);
    if (rc) return rc;
    a.f16_dg = dG16; a.f16_dgT = dG16T; a.f16_auxT = aux16T; a.f16_scale = scale; a.f16_done = &f16_done;
  }
  {
    DS2_PROF("rnn_bwd_sweep", st);
    rc = 1;
    if (tensor_core_mode()) {
      rc = rnn_sweep_bwd_tc(d->rnn_type, a, gws, gws_bytes, st);
      if (rc == 1) note_fallback("backward sweep", d->rnn_type, T, B, H, D);
    }
    if (rc == 1) {
      rc = fill_w_hh_cb(&fill, st);
      if (rc) return rc;
      rc = sweep_bwd(d->rnn_type, a, st);
    }
    if (rc) return rc;
  }

  // the layer input as the projection saw it (BN applied) and its normalised form for the BN backward
  const float* xin = x;
  if (bn_gamma) {
    // recompute xhat and xbn from the saved batch statistics
    rc = bn_rows_reapply(TB, In, x, bn_gamma, bn_beta, R.bnstats, xbn, xhat, st);
    if (rc) return rc;
    xin = xbn;
  }
  DS2_PROF("rnn_bwd_gemms", st);
  if (f16) {
    const size_t DGH = (size_t)D * GH;
    if (!f16_done) {
      unsigned int* absmax_ws = reinterpret_cast<unsigned int*>(scale + 8);
      rc = pow2_scale_for(TB, (int)DGH, R.gates, DGH, absmax_ws, scale, 10, st);
      if (rc) return rc;
      rc = f32_to_f16_transpose(TB, (int)DGH, R.gates, DGH, dG16, DGH, dG16T, (size_t)TB, scale, st);
      if (rc) return rc;
    }
    for (int dir = 0; dir < D; ++dir) {
      rc = f32_to_f16_transpose(GH, In, w_ih[dir], (size_t)In, nullptr, 0, w16T + (size_t)dir * GH, DGH, nullptr, st);
      if (rc) return rc;
    }
  }
  // weight-gradient GEMMs: nobody needs dW_ih / dW_hh before the optimizer, so (precision-16 path, caller opted in)
  // they go to the side stream together with the operand copies only they read (x16T, h16T), ordered after the sweep,
  // and overlap the next layer's sweep.  The side stream then reads x / reserve until ds2_join_side_stream.
  cudaStream_t gst = st;
  if (f16 && side && d->deferred_dw) {
    rc = side_fork(st, side);
    if (rc) return rc;
    gst = side;
  }
  if (f16) {
    rc = f32_to_f16_transpose(TB, In, xin, (size_t)In, nullptr, 0, x16T, (size_t)TB, nullptr, gst);
    if (rc) return rc;
    for (int dir = 0; dir < D; ++dir) {
      rc = f32_to_f16_transpose(TB, H, R.hseq + (size_t)dir * TB * H, (size_t)H, nullptr, 0, h16T + (size_t)dir * H * TB,
                                (size_t)TB, nullptr, gst);
      if (rc) return rc;
      if (gru && !f16_done) {
        rc = f32_to_f16_transpose(TB, H, R.aux + (size_t)dir * TB * H, (size_t)H, nullptr, 0,
                                  aux16T + (size_t)dir * H * TB, (size_t)TB, scale, gst);
        if (rc) return rc;
      }
    }
  }
  bool dx_done = false;
  if (f16 && dx) {   // dX = dG (TB x D*GH) . [W_ih fwd ; W_ih rev] : one K = D*G*H GEMM for both directions
    rc = gemm_tc_f16(TB, In, D * GH, 1.f, dG16, D * GH, w16T, D * GH, 0.f, bn_gamma ? dxbn : dx, In, scale + 1, st);
    if (rc < 0) return rc;
    dx_done = rc == 0;
  }
  for (int dir = 0; dir < D; ++dir) {
    const float* dG = R.gates + (size_t)dir * GH;   // (TB, GH) with row stride D*GH : dGx
    const int ldg = D * GH;
    const float* aux_d = R.aux ? R.aux + (size_t)dir * TB * H : nullptr;   // GRU: dGh_n (TB,H)
    const float* hseq_d = R.hseq + (size_t)dir * TB * H;
    // dW_ih = dGx^T . xin
    rc = 1;
    if (f16) {
      rc = gemm_tc_f16(GH, In, TB, 1.f, dG16T + (size_t)dir * GH * TB, TB, x16T, TB, 0.f, dw_ih[dir], In, scale + 1, gst);
      if (rc < 0) return rc;
    }
    if (rc == 1) rc = ds2_gemm(1, 0, GH, In, TB, 1.f, dG, ldg, xin, In, 0.f, dw_ih[dir], In, gws, gws_bytes, stream);
    if (rc) return rc;
    if (!dbias_done) {
      rc = colsum(TB, GH, dG, ldg, db_ih[dir], st);
      if (rc) return rc;
    }
    // dW_hh = sum_t dGh[t]^T . h_prev[t]; h_prev[t] = hseq[t-1] (forward) / hseq[t+1] (reverse)
    const int Kr = (T - 1) * B;
    const size_t a_off = dir == 0 ? (size_t)B : 0, h_off = dir == 0 ? 0 : (size_t)B;
    const int rows_x = gru ? 2 * H : GH;   // rows whose dGh == dGx
    if (Kr > 0) {
      rc = 1;
      if (f16) {   // in the transposed copies a shift by one time step is a shift by B columns
        rc = gemm_tc_f16(rows_x, H, Kr, 1.f, dG16T + (size_t)dir * GH * TB + a_off, TB, h16T + (size_t)dir * H * TB + h_off,
                         TB, 0.f, dw_hh[dir], H, scale + 1, gst);
        if (rc < 0) return rc;
      }
      if (rc == 1)
        rc = ds2_gemm(1, 0, rows_x, H, Kr, 1.f, dG + a_off * ldg, ldg, hseq_d + h_off * H, H, 0.f, dw_hh[dir], H, gws,
                      gws_bytes, stream);
      if (rc) return rc;
      if (gru) {
        rc = 1;
        if (f16) {
          rc = gemm_tc_f16(H, H, Kr, 1.f, aux16T + (size_t)dir * H * TB + a_off, TB, h16T + (size_t)dir * H * TB + h_off,
                           TB, 0.f, dw_hh[dir] + (size_t)2 * H * H, H, scale + 1, gst);
          if (rc < 0) return rc;
        }
        if (rc == 1)
          rc = ds2_gemm(1, 0, H, H, Kr, 1.f, aux_d + a_off * H, H, hseq_d + h_off * H, H, 0.f,
                        dw_hh[dir] + (size_t)2 * H * H, H, gws, gws_bytes, stream);
        if (rc) return rc;
      }
    } else {
      DS2_CHECK_CUDA(cudaMemsetAsync(dw_hh[dir], 0, sizeof(float) * (size_t)GH * H, st));
    }
    if (gru) {
      DS2_CHECK_CUDA(cudaMemcpyAsync(db_hh[dir], db_ih[dir], sizeof(float) * 2 * H, cudaMemcpyDeviceToDevice, st));
      if (!dbias_done) {
        rc = colsum(TB, H, aux_d, H, db_hh[dir] + 2 * H, st);
        if (rc) return rc;
      }
    } else {
      DS2_CHECK_CUDA(cudaMemcpyAsync(db_hh[dir], db_ih[dir], sizeof(float) * GH, cudaMemcpyDeviceToDevice, st));
    }
    // dX (pre-BN-affine) += dGx . W_ih
    if (dx && !dx_done) {
      rc = ds2_gemm(0, 0, TB, In, GH, 1.f, dG, ldg, w_ih[dir], In, dir == 0 ? 0.f : 1.f, bn_gamma ? dxbn : dx, In,
                    gws, gws_bytes, stream);
      if (rc) return rc;
    }
  }
  if (gst != st) {
    rc = side_mark_workspace(ws, side);
    if (rc) return rc;
  }
  if (bn_gamma) {
    DS2_REQUIRE(dx && dbn_gamma && dbn_beta, "rnn bwd: BN layer needs dx, dbn_gamma, dbn_beta");
    rc = bn_rows_bwd(TB, In, xhat, bn_gamma, R.bnstats, dxbn, dx, dbn_gamma, dbn_beta, sums, st);
    if (rc) return rc;
  }
  return DS2_OK;
}

}  // extern "C"
