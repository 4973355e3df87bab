// Conv front-end of DeepSpeech2 (model.py:157-164 under MaskConv :53-69) + the (B,C,D,T)->(T,B,C*D)
// re-layout of model.py:219-221, forward and backward, as im2col-free direct convolutions:
// each CTA stages an input slab (rows x cols of one input channel) and that channel's packed
// filter taps [kh][kw][32 co] in shared memory; a thread owns 8 output channels x 4 consecutive
// time steps in registers and slides along kw (vectorised LDS.128 on both operands).
//
//   z1 = mask(conv1(x)+b1)            (B,32,81,T')   stats accumulated in the conv epilogue
//   a1 = mask(clamp(BN1(z1),0,20))    (B,32,81,T')
//   z2 = mask(conv2(a1)+b2)           (B,32,41,T')
//   y  = mask(clamp(BN2(z2),0,20))    written time-major (T',B,32*41), feature = c*41+d
//
// BatchNorm statistics include the masked (zeroed) positions exactly like the reference
// (count = B*D*T', SURVEY.md §8c).  The mask is applied from the device-resident length vector, so
// the reference's CPU-built Bool masks / 6 H2D copies / .item() syncs disappear (SURVEY §2b K4).
//
// Backward: BN/Hardtanh/mask backward fused into two passes per BN (reduce, apply); conv2 data
// gradient = two stride-1 convolutions (even / odd input rows) run through the SAME forward kernel
// with re-packed (flipped, transposed) taps; weight gradients by dedicated reduction kernels.
#include <stdlib.h>

#include "common.cuh"

namespace ds2 {

constexpr int CO = 32;           // output channels of both convolutions
constexpr int TD = 4, TT = 64;   // output tile: 4 rows x 64 time steps x 32 channels per CTA

template <int KH, int KW, int SH, int SW>
struct ConvGeom {
  static constexpr int ROWS = (TD - 1) * SH + KH;
  static constexpr int XIN = (4 - 1) * SW + KW;                     // inputs a thread needs per row
  static constexpr int XVEC = (XIN + 3) / 4;                        // as float4 loads
  static constexpr int COLS = ((15 * 4 * SW + XVEC * 4) + 3) / 4 * 4;  // slab width (16B aligned rows)
  static constexpr int SLAB = ROWS * COLS;
  static constexpr int WTS = KH * KW * CO;
  static constexpr size_t SMEM = (size_t)(SLAB + WTS) * sizeof(float);
};

// out[b,co,d,t] = bias[co] + sum_{ci,kh,kw} wpk[ci][kh][kw][co] * in[b,ci,d*SH+kh-PH,t*SW+kw-PW]
// out address = b*ob + co*oc + d*orow + t ; positions t >= out_len[b] are written as 0 (if out_len)
// stat_sums (double[64]) += per-channel sum / sum of squares of what was written (if non-null)
template <int KH, int KW, int SH, int SW>
__global__ void __launch_bounds__(256) conv_fwd_kernel(const float* __restrict__ in, int Cin, int Hin, int Win,
                                                       const float* __restrict__ wpk, const float* __restrict__ bias,
                                                       float* __restrict__ out, int Hout, int Wout, size_t ob,
                                                       size_t oc, size_t orow, int PH, int PW,
                                                       const int32_t* __restrict__ out_len,
                                                       double* __restrict__ stat_sums) {
  using Gm = ConvGeom<KH, KW, SH, SW>;
  extern __shared__ __align__(16) float smem[];
  float* slab = smem;
  float* wsm = smem + Gm::SLAB;
  const int tid = threadIdx.x;
  const int b = blockIdx.z, d0 = blockIdx.y * TD, t0 = blockIdx.x * TT;
  const int cg = tid / 64, pos = tid % 64, dl = pos / 16, tg = pos % 16;
  float acc[4][8];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[j][c] = 0.f;

  const int in_r0 = d0 * SH - PH, in_c0 = t0 * SW - PW;
  for (int ci = 0; ci < Cin; ++ci) {
    const float* src = in + ((size_t)b * Cin + ci) * Hin * Win;
    for (int idx = tid; idx < Gm::SLAB; idx += 256) {
      int r = idx / Gm::COLS, c = idx % Gm::COLS;
      int gr = in_r0 + r, gc = in_c0 + c;
      slab[idx] = (gr >= 0 && gr < Hin && gc >= 0 && gc < Win) ? src[(size_t)gr * Win + gc] : 0.f;
    }
    const float4* wsrc = reinterpret_cast<const float4*>(wpk + (size_t)ci * Gm::WTS);
    for (int idx = tid; idx < Gm::WTS / 4; idx += 256) reinterpret_cast<float4*>(wsm)[idx] = wsrc[idx];
    __syncthreads();
#pragma unroll 1
    for (int kh = 0; kh < KH; ++kh) {
      const float4* row = reinterpret_cast<const float4*>(slab + (dl * SH + kh) * Gm::COLS + tg * 4 * SW);
      float xin[Gm::XVEC * 4];
#pragma unroll
      for (int v = 0; v < Gm::XVEC; ++v) *reinterpret_cast<float4*>(&xin[v * 4]) = row[v];
      const float* wrow = wsm + kh * KW * CO + cg * 8;
#pragma unroll
      for (int kw = 0; kw < KW; ++kw) {
        float4 w0 = *reinterpret_cast<const float4*>(wrow + kw * CO);
        float4 w1 = *reinterpret_cast<const float4*>(wrow + kw * CO + 4);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float xv = xin[j * SW + kw];
          acc[j][0] = fmaf(xv, w0.x, acc[j][0]); acc[j][1] = fmaf(xv, w0.y, acc[j][1]);
          acc[j][2] = fmaf(xv, w0.z, acc[j][2]); acc[j][3] = fmaf(xv, w0.w, acc[j][3]);
          acc[j][4] = fmaf(xv, w1.x, acc[j][4]); acc[j][5] = fmaf(xv, w1.y, acc[j][5]);
          acc[j][6] = fmaf(xv, w1.z, acc[j][6]); acc[j][7] = fmaf(xv, w1.w, acc[j][7]);
        }
      }
    }
    __syncthreads();
  }
  // epilogue: bias, mask, store, statistics
  const int d = d0 + dl;
  const int L = out_len ? out_len[b] : Wout;
  float s1[8], s2[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) s1[c] = s2[c] = 0.f;
  if (d < Hout) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const int co = cg * 8 + c;
      const float bv = bias ? bias[co] : 0.f;
      float* op = out + (size_t)b * ob + (size_t)co * oc + (size_t)d * orow;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        int t = t0 + tg * 4 + j;
        if (t < Wout) {
          float v = (t < L) ? acc[j][c] + bv : 0.f;
          op[t] = v;
          s1[c] += v;
          s2[c] = fmaf(v, v, s2[c]);
        }
      }
    }
  }
  if (stat_sums) {
    __shared__ float red[2][8][CO];   // [sum|sumsq][warp][co]
    const int warp = tid / 32, lane = tid % 32;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float a = warp_sum(s1[c]), q = warp_sum(s2[c]);
      if (lane == 0) { red[0][warp][(warp / 2) * 8 + c] = a; red[1][warp][(warp / 2) * 8 + c] = q; }
    }
    __syncthreads();
    if (tid < 2 * CO) {
      int which = tid / CO, co = tid % CO, w0 = (co / 8) * 2;
      double v = (double)red[which][w0][co] + (double)red[which][w0 + 1][co];
      atomicAdd(&stat_sums[which * CO + co], v);
    }
  }
}

// ---- filter re-packing ------------------------------------------------------------------------
// forward: wpk[ci][kh][kw][co] = w[co][ci][kh][kw]
__global__ void pack_fwd_kernel(int Cin, int KH, int KW, const float* __restrict__ w, float* __restrict__ wpk) {
  int i = blockIdx.x * blockDim.x + threadIdx.x, n = Cin * KH * KW * CO;
  if (i >= n) return;
  int co = i % CO, kw = (i / CO) % KW, kh = (i / (CO * KW)) % KH, ci = i / (CO * KW * KH);
  wpk[i] = w[(((size_t)co * Cin + ci) * KH + kh) * KW + kw];
}
// conv2 data gradient (32->32, 21x11, stride (2,1), pad (10,5)): rows of parity p of d(a1) are a
// stride-1 correlation of dz2 with taps  wT[co][m][k][ci] = w2[co][ci][2*(M-1-m)+p][10-k],
// M = 11 (p=0) / 10 (p=1), pad_h = 5 - p, pad_w = 5.
__global__ void pack_bwd_data_kernel(int parity, const float* __restrict__ w2, float* __restrict__ wT) {
  const int M = parity ? 10 : 11;
  int i = blockIdx.x * blockDim.x + threadIdx.x, n = CO * M * 11 * CO;
  if (i >= n) return;
  int ci = i % CO, k = (i / CO) % 11, m = (i / (CO * 11)) % M, co = i / (CO * 11 * M);
  int kh = 2 * (M - 1 - m) + parity, kw = 10 - k;
  wT[i] = w2[(((size_t)co * CO + ci) * 21 + kh) * 11 + kw];
}

// ---- BatchNorm2d pieces -----------------------------------------------------------------------
__global__ void bn2d_finalize_kernel(double count, const double* __restrict__ sums, const float* __restrict__ gamma,
                                     const float* __restrict__ beta, float* __restrict__ rmean,
                                     float* __restrict__ rvar, int training, float momentum, float eps,
                                     float* __restrict__ mean_invstd /*[2][32]*/) {
  int c = threadIdx.x;
  if (c >= CO) return;
  float mean, var;
  if (training) {
    double m = sums[c] / count, v = sums[CO + c] / count - m * m;
    if (v < 0.0) v = 0.0;
    mean = (float)m;
    var = (float)v;
    double unb = count > 1.0 ? v * count / (count - 1.0) : v;
    rmean[c] = (1.f - momentum) * rmean[c] + momentum * mean;
    rvar[c] = (1.f - momentum) * rvar[c] + momentum * (float)unb;
  } else {
    mean = rmean[c];
    var = rvar[c];
  }
  mean_invstd[c] = mean;
  mean_invstd[CO + c] = rsqrtf(var + eps);
}

// a = mask(clamp(gamma*(z-mean)*invstd+beta, 0, 20)) over (B,32,D,T)
__global__ void bn_act_kernel(int B, int D, int T, const float* __restrict__ z, const float* __restrict__ mi,
                              const float* __restrict__ gamma, const float* __restrict__ beta,
                              const int32_t* __restrict__ len, float* __restrict__ a) {
  size_t total = (size_t)B * CO * D * T;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    int t = (int)(i % T);
    int c = (int)((i / ((size_t)T * D)) % CO), b = (int)(i / ((size_t)T * D * CO));
    float v = 0.f;
    if (t < len[b]) {
      float u = fmaf((z[i] - mi[c]) * mi[CO + c], gamma[c], beta[c]);
      v = fminf(fmaxf(u, 0.f), 20.f);
    }
    a[i] = v;
  }
}

// y[t][b][c*D+d] = mask(clamp(BN(z[b][c][d][t]))) ; 32x32 tile transposes; grid (ceil(T/32), ceil(CD/32), B)
__global__ void bn_act_transpose_kernel(int B, int D, int T, const float* __restrict__ z,
                                        const float* __restrict__ mi, const float* __restrict__ gamma,
                                        const float* __restrict__ beta, const int32_t* __restrict__ len,
                                        float* __restrict__ y) {
  __shared__ float tile[32][33];
  const int CD = CO * D, b = blockIdx.z, t0 = blockIdx.x * 32, f0 = blockIdx.y * 32;
  const int L = len[b];
  for (int j = threadIdx.y; j < 32; j += 8) {
    int f = f0 + j, t = t0 + threadIdx.x;
    float v = 0.f;
    if (f < CD && t < T && t < L) {
      int c = f / D;
      float u = fmaf((z[((size_t)b * CD + f) * T + t] - mi[c]) * mi[CO + c], gamma[c], beta[c]);
      v = fminf(fmaxf(u, 0.f), 20.f);
    }
    tile[j][threadIdx.x] = v;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += 8) {
    int t = t0 + j, f = f0 + threadIdx.x;
    if (t < T && f < CD) y[((size_t)t * B + b) * CD + f] = tile[threadIdx.x][j];
  }
}

// Backward pass 1 of a BN+Hardtanh+mask stage:  du = dy * 1[0<u<20] * 1[t<len]   (written to du)
// and per-channel sums  S1 = sum du, S2 = sum du*zhat  (double atomics into sums[64]).
// TRANSPOSED=true reads dy as (T,B,C*D) (the RNN-side layout), else as (B,C,D,T).
template <bool TRANSPOSED>
__global__ void bn_bwd_reduce_kernel(int B, int D, int T, const float* __restrict__ z,
                                     const float* __restrict__ mi, const float* __restrict__ gamma,
                                     const float* __restrict__ beta, const int32_t* __restrict__ len,
                                     const float* dy, float* du /* may alias dy (same index) */,
                                     double* __restrict__ sums) {
  // grid (ceil(T/32), ceil(CD/32), B), block (32, 8): thread (x = t lane, rows f)
  __shared__ float tile[32][33];
  __shared__ float r1[8][32], r2[8][32];
  const int CD = CO * D, b = blockIdx.z, t0 = blockIdx.x * 32, f0 = blockIdx.y * 32;
  const int L = len[b];
  if (TRANSPOSED) {
    for (int j = threadIdx.y; j < 32; j += 8) {
      int t = t0 + j, f = f0 + threadIdx.x;
      tile[j][threadIdx.x] = (t < T && f < CD) ? dy[((size_t)t * B + b) * CD + f] : 0.f;
    }
    __syncthreads();
  }
  // each thread walks rows f = f0 + threadIdx.y + 8*k at time t0 + threadIdx.x
  for (int j = threadIdx.y; j < 32; j += 8) {
    int f = f0 + j, t = t0 + threadIdx.x;
    float g = 0.f, zh = 0.f;
    if (f < CD && t < T) {
      int c = f / D;
      size_t zi = ((size_t)b * CD + f) * T + t;
      zh = (z[zi] - mi[c]) * mi[CO + c];
      float u = fmaf(zh, gamma[c], beta[c]);
      float dyv = TRANSPOSED ? tile[threadIdx.x][j] : dy[zi];
      g = (t < L && u > 0.f && u < 20.f) ? dyv : 0.f;
      du[zi] = g;
    }
    // reduce over the 32 time lanes (same f => same channel)
    float a = warp_sum(g), q = warp_sum(g * zh);
    if (threadIdx.x == 0) { r1[threadIdx.y][j] = a; r2[threadIdx.y][j] = q; }
  }
  __syncthreads();
  // rows j handled by warp (j % 8); combine rows of the same channel, then one atomic per channel
  if (threadIdx.y == 0) {
    int j = threadIdx.x, f = f0 + j;
    float a = (f < CD) ? r1[j % 8][j] : 0.f, q = (f < CD) ? r2[j % 8][j] : 0.f;
    int c = (f < CD) ? f / D : -1;
    // serial merge by lane 0 of runs with equal channel (at most 2-3 channels per 32 rows)
    int c0 = __shfl_sync(0xffffffffu, c, 0);
    (void)c0;
    for (int cc = f0 / D; cc <= min(CO - 1, (f0 + 31) / D); ++cc) {
      float sa = warp_sum(c == cc ? a : 0.f), sq = warp_sum(c == cc ? q : 0.f);
      if (threadIdx.x == 0) { atomicAdd(&sums[cc], (double)sa); atomicAdd(&sums[CO + cc], (double)sq); }
    }
  }
}

// Backward pass 2:  dz = 1[t<len] * gamma*invstd*(du - S1/N - zhat*S2/N)  in place over du,
// plus the block's share of db[c] = sum dz (bias gradient of the producing convolution) in db_part[c][b][block],
// summed by bias_grad_kernel in a fixed order.
__global__ void bn_bwd_apply_kernel(int B, int D, int T, double inv_count, const float* __restrict__ z,
                                    const float* __restrict__ mi, const float* __restrict__ gamma,
                                    const int32_t* __restrict__ len, const double* __restrict__ sums,
                                    float* __restrict__ du_dz, float* __restrict__ db_part) {
  // grid (ceil(T*D/256), CO, B)
  const int c = blockIdx.y, b = blockIdx.z;
  const size_t base = ((size_t)b * CO + c) * D * T;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const float m1 = (float)(sums[c] * inv_count), m2 = (float)(sums[CO + c] * inv_count);
  const float k = gamma[c] * mi[CO + c];
  float v = 0.f;
  if (i < D * T) {
    int t = i % T;
    if (t < len[b]) {
      float zh = (z[base + i] - mi[c]) * mi[CO + c];
      v = k * (du_dz[base + i] - m1 - zh * m2);
    }
    du_dz[base + i] = v;
  }
  __shared__ float red[8];
  float s = warp_sum(v);
  if (threadIdx.x % 32 == 0) red[threadIdx.x / 32] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int w = 0; w < (int)blockDim.x / 32; ++w) tot += red[w];
    db_part[((size_t)c * gridDim.z + b) * gridDim.x + blockIdx.x] = tot;
  }
}

// dbias[c] = sum of the n partials of channel c; grid CO, block 256; fixed summation order
__global__ void bias_grad_kernel(int n, const float* __restrict__ db_part, float* __restrict__ dbias) {
  __shared__ float red[256];
  const float* src = db_part + (size_t)blockIdx.x * n;
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) acc += src[i];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) dbias[blockIdx.x] = red[0];
}

__global__ void bn_bwd_params2d_kernel(const double* __restrict__ sums, float* __restrict__ dgamma,
                                       float* __restrict__ dbeta) {
  int c = threadIdx.x;
  if (c < CO) { dbeta[c] = (float)sums[c]; dgamma[c] = (float)sums[CO + c]; }
}

// ---- weight gradients -------------------------------------------------------------------------
// conv2: dw2[co][ci][kh][kw] = sum_{b,d,t} dz2[b,co,d,t] * a1[b,ci,2d+kh-10,t+kw-5]
// CTA = (kh, b); thread = (4 co, 1 ci) x 11 kw accumulators; atomics merge the batch.
__global__ void __launch_bounds__(256) conv2_dw_kernel(int B, int T, const float* __restrict__ dz2,
                                                       const float* __restrict__ a1, float* __restrict__ dw2) {
  constexpr int D1 = DS2_CONV1_D, D2 = DS2_CONV2_D, TW = 64, AW = TW + 12;  // 76 columns staged (74 used)
  __shared__ __align__(16) float dsm[TW][36];   // [t][co]
  __shared__ float asmx[AW][33];                // [t+kw][ci]
  const int kh = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const int cog = tid / 32, ci = tid % 32;
  float acc[4][11];
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int k = 0; k < 11; ++k) acc[c][k] = 0.f;
  for (int d = 0; d < D2; ++d) {
    const int r = 2 * d + kh - 10;
    if (r < 0 || r >= D1) continue;
    for (int t0 = 0; t0 < T; t0 += TW) {
      for (int idx = tid; idx < CO * TW; idx += 256) {
        int tt = idx % TW, co = idx / TW, t = t0 + tt;
        dsm[tt][co] = (t < T) ? dz2[(((size_t)b * CO + co) * D2 + d) * T + t] : 0.f;
      }
      for (int idx = tid; idx < CO * AW; idx += 256) {
        int tt = idx % AW, c2 = idx / AW, t = t0 + tt - 5;
        asmx[tt][c2] = (t >= 0 && t < T) ? a1[(((size_t)b * CO + c2) * D1 + r) * T + t] : 0.f;
      }
      __syncthreads();
#pragma unroll 1
      for (int tb = 0; tb < TW; tb += 4) {
        float win[14];
#pragma unroll
        for (int i = 0; i < 14; ++i) win[i] = asmx[tb + i][ci];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float4 dv = *reinterpret_cast<const float4*>(&dsm[tb + j][cog * 4]);
#pragma unroll
          for (int k = 0; k < 11; ++k) {
            float a = win[j + k];
            acc[0][k] = fmaf(dv.x, a, acc[0][k]); acc[1][k] = fmaf(dv.y, a, acc[1][k]);
            acc[2][k] = fmaf(dv.z, a, acc[2][k]); acc[3][k] = fmaf(dv.w, a, acc[3][k]);
          }
        }
      }
      __syncthreads();
    }
  }
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int k = 0; k < 11; ++k)
      atomicAdd(&dw2[((((size_t)(cog * 4 + c)) * CO + ci) * 21 + kh) * 11 + k], acc[c][k]);
}

// conv1: dw1[co][kh][kw] = sum_{b,d,t} dz1[b,co,d,t] * x[b,2d+kh-20,2t+kw-5]
// CTA = (group of 14 kh, b, half of the d range); thread = (kh_local, group of 4 co) with 4 x 11 kw accumulators:
// per 4 time steps 17 window loads + 4 vector loads feed 176 FFMAs (the earlier 1 co x 11 kw blocking was
// shared-memory bound at 21 loads per 44 FFMAs).
constexpr int C1_KG = 14, C1_TW = 64, C1_XW = 2 * C1_TW + 12, C1_DSPLIT = 6;
__global__ void __launch_bounds__(128) conv1_dw_kernel(int B, int Tin, int T, const float* __restrict__ dz1,
                                                       const float* __restrict__ x, float* __restrict__ dw1) {
  constexpr int D1 = DS2_CONV1_D, F = DS2_NUM_FREQ, TW = C1_TW, XW = C1_XW;
  __shared__ __align__(16) float dsm[TW][CO];     // [t][co]
  __shared__ float xsm[C1_KG][XW];                // [kh_local][2t+kw]
  const int kh0 = blockIdx.x * C1_KG, b = blockIdx.y, tid = threadIdx.x;
  const int dper = (D1 + C1_DSPLIT - 1) / C1_DSPLIT, d0 = blockIdx.z * dper, d1 = min(D1, d0 + dper);
  const int cog = tid % 8, khl = tid / 8, kh = kh0 + khl;      // khl 14, 15: loaders only
  const bool worker = khl < C1_KG && kh < 41;
  const int khr = worker ? khl : 0;
  float acc[4][11];
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int k = 0; k < 11; ++k) acc[c][k] = 0.f;
  for (int d = d0; d < d1; ++d) {
    for (int t0 = 0; t0 < T; t0 += TW) {
      for (int idx = tid; idx < CO * TW; idx += 128) {
        const int tt = idx % TW, c2 = idx / TW, t = t0 + tt;
        dsm[tt][c2] = (t < T) ? dz1[(((size_t)b * CO + c2) * D1 + d) * T + t] : 0.f;
      }
      for (int idx = tid; idx < C1_KG * XW; idx += 128) {
        const int cc = idx % XW, kl = idx / XW, r = 2 * d + kh0 + kl - 20, c = 2 * t0 + cc - 5;
        xsm[kl][cc] = (kh0 + kl < 41 && r >= 0 && r < F && c >= 0 && c < Tin) ? x[((size_t)b * F + r) * Tin + c] : 0.f;
      }
      __syncthreads();
      if (worker) {
#pragma unroll 1
        for (int tb = 0; tb < TW; tb += 4) {
          float win[17];
#pragma unroll
          for (int i = 0; i < 17; ++i) win[i] = xsm[khr][2 * tb + i];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 dv = *reinterpret_cast<const float4*>(&dsm[tb + j][cog * 4]);
#pragma unroll
            for (int k = 0; k < 11; ++k) {
              const float a = win[2 * j + k];
              acc[0][k] = fmaf(dv.x, a, acc[0][k]); acc[1][k] = fmaf(dv.y, a, acc[1][k]);
              acc[2][k] = fmaf(dv.z, a, acc[2][k]); acc[3][k] = fmaf(dv.w, a, acc[3][k]);
            }
          }
        }
      }
      __syncthreads();
    }
  }
  if (worker) {
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int k = 0; k < 11; ++k) atomicAdd(&dw1[((size_t)(cog * 4 + c) * 41 + kh) * 11 + k], acc[c][k]);
  }
}

// ---- host helpers -------------------------------------------------------------------------------
template <int KH, int KW, int SH, int SW>
static int launch_conv(const float* in, int B, int Cin, int Hin, int Win, const float* wpk, const float* bias,
                       float* out, int Hout, int Wout, size_t ob, size_t oc, size_t orow, int PH, int PW,
                       const int32_t* out_len, double* sums, cudaStream_t st) {
  using Gm = ConvGeom<KH, KW, SH, SW>;
  auto kern = conv_fwd_kernel<KH, KW, SH, SW>;
  DS2_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Gm::SMEM));
  dim3 grid(cdiv(Wout, TT), cdiv(Hout, TD), B);
  DS2_LAUNCH(kern, grid, 256, Gm::SMEM, st, in, Cin, Hin, Win, wpk, bias, out, Hout, Wout, ob, oc, orow, PH, PW,
             out_len, sums);
  return DS2_OK;
}

// tensor-core 32->32 convolution (conv_tc.cu)
int conv_tc_run(const float* in_cl, int B, int T, int R_in, int R_out, const float* taps, int n_taps, int J,
                int row_mul, int row_off, int row_step, int w_off, int w_step, float* out, size_t ob, size_t oc,
                size_t orow, int out_row_mul, int out_row_off, const float* bias, const int32_t* out_len,
                double* stat_sums, cudaStream_t st);
int nchw_to_cl(int B, int R, int T, const float* in, float* out, cudaStream_t st);
int pack_conv2_tc(const float* w2, float* wn_fwd, float* wd_bwd, cudaStream_t st);
int conv2_wgrad_tc(const float* dz2, const float* a1, float* a1_shifted, int B, int T, float* dw2, float* part,
                   cudaStream_t st);
int conv1_wgrad_tc(const float* dz1, const float* x, float* xs, int B, int T, int Tp, float* dw1, float* part,
                   cudaStream_t st);
size_t conv_wgrad_tc_part_floats();

struct ConvWs {
  float *wpk1, *wpk2, *wTe, *wTo, *du2, *da1;
  float *taps_f, *taps_b, *cl;     // tensor-core path: packed taps (21x352x32 each), channels-last staging
  float* shifted;                  // tensor-core weight gradient: a1 delayed by 0,1,2,3 time steps
  float* wpart;                    // tensor-core weight gradients: per-CTA partial sums
  float* dbpart;                   // conv bias gradients: per-block partial sums (CO x B x blocks)
  double* sums;   // 4 x 64 doubles: fwd stats 1, fwd stats 2, bwd sums 2, bwd sums 1
};
static size_t conv_ws_carve(int B, int T, void* base, ConvWs* w) {
  const size_t Tp = (size_t)(T - 1) / 2 + 1;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes, 256); return base ? (char*)base + o : nullptr; };
  float* p;
  p = (float*)take((size_t)41 * 11 * CO * 4); if (w) w->wpk1 = p;
  p = (float*)take((size_t)CO * 21 * 11 * CO * 4); if (w) w->wpk2 = p;
  p = (float*)take((size_t)CO * 11 * 11 * CO * 4); if (w) w->wTe = p;
  p = (float*)take((size_t)CO * 10 * 11 * CO * 4); if (w) w->wTo = p;
  double* s = (double*)take(4 * 64 * sizeof(double)); if (w) w->sums = s;
  p = (float*)take((size_t)B * CO * DS2_CONV2_D * Tp * 4); if (w) w->du2 = p;
  p = (float*)take((size_t)B * CO * DS2_CONV1_D * Tp * 4); if (w) w->da1 = p;
  p = (float*)take((size_t)21 * 352 * 32 * 4); if (w) w->taps_f = p;
  p = (float*)take((size_t)21 * 352 * 32 * 4); if (w) w->taps_b = p;
  p = (float*)take((size_t)B * CO * DS2_CONV1_D * Tp * 4); if (w) w->cl = p;
  p = (float*)take((size_t)4 * B * CO * DS2_CONV1_D * (Tp + 4) * 4); if (w) w->shifted = p;
  p = (float*)take(conv_wgrad_tc_part_floats() * 4); if (w) w->wpart = p;
  p = (float*)take((size_t)CO * B * cdiv((long long)DS2_CONV1_D * Tp, 256) * 4); if (w) w->dbpart = p;
  return off;
}

}  // namespace ds2

extern "C" {
using namespace ds2;

size_t ds2_conv_frontend_workspace_bytes(int B, int T) {
  if (B <= 0 || T <= 0) return 0;
  return conv_ws_carve(B, T, nullptr, nullptr) + 256;
}

int ds2_conv_frontend_fwd(int B, int T, const float* x, const int32_t* out_len, const float* w1, const float* b1,
                          const float* g1, const float* be1, float* rm1, float* rv1, const float* w2,
                          const float* b2, const float* g2, const float* be2, float* rm2, float* rv2, int training,
                          float momentum, float eps, float* y, float* z1, float* a1, float* z2, float* stats,
                          void* ws, size_t ws_bytes, void* stream) {
  DS2_REQUIRE(B > 0 && T > 0, "conv fwd: bad shape B=%d T=%d", B, T);
  DS2_REQUIRE(ws_bytes >= ds2_conv_frontend_workspace_bytes(B, T), "conv fwd: workspace too small");
  cudaStream_t st = as_stream(stream);
  const int Tp = (T - 1) / 2 + 1, D1 = DS2_CONV1_D, D2 = DS2_CONV2_D, F = DS2_NUM_FREQ;
  ConvWs W;
  conv_ws_carve(B, T, ws, &W);
  DS2_PROF("conv_fwd", st);
  DS2_CHECK_CUDA(cudaMemsetAsync(W.sums, 0, 4 * 64 * sizeof(double), st));
  DS2_LAUNCH(pack_fwd_kernel, cdiv(41 * 11 * CO, 256), 256, 0, st, 1, 41, 11, w1, W.wpk1);
  DS2_LAUNCH(pack_fwd_kernel, cdiv(CO * 21 * 11 * CO, 256), 256, 0, st, CO, 21, 11, w2, W.wpk2);
  int rc = launch_conv<41, 11, 2, 2>(x, B, 1, F, T, W.wpk1, b1, z1, D1, Tp, (size_t)CO * D1 * Tp, (size_t)D1 * Tp,
                                     (size_t)Tp, 20, 5, out_len, training ? W.sums : nullptr, st);
  if (rc) return rc;
  DS2_LAUNCH(bn2d_finalize_kernel, 1, 32, 0, st, (double)B * D1 * Tp, W.sums, g1, be1, rm1, rv1, training, momentum,
             eps, stats);
  DS2_LAUNCH(bn_act_kernel, 148 * 8, 256, 0, st, B, D1, Tp, z1, stats, g1, be1, out_len, a1);
  if (tensor_core_mode() && !getenv("DS2_NO_CONV_TC") && !getenv("DS2_NO_CONV_TC_FWD")) {
    // conv2 on tcgen05: channels-last copy of a1, packed taps, implicit GEMM with the kw taps folded into N
    rc = nchw_to_cl(B, D1, Tp, a1, W.cl, st);
    if (rc) return rc;
    rc = pack_conv2_tc(w2, W.taps_f, nullptr, st);
    if (rc) return rc;
    rc = conv_tc_run(W.cl, B, Tp, D1, D2, W.taps_f, 21, 21, 2, -10, 1, 0, 1, z2, (size_t)CO * D2 * Tp, (size_t)D2 * Tp,
                     (size_t)Tp, 1, 0, b2, out_len, training ? W.sums + 64 : nullptr, st);
  } else {
    rc = launch_conv<21, 11, 2, 1>(a1, B, CO, D1, Tp, W.wpk2, b2, z2, D2, Tp, (size_t)CO * D2 * Tp, (size_t)D2 * Tp,
                                   (size_t)Tp, 10, 5, out_len, training ? W.sums + 64 : nullptr, st);
  }
  if (rc) return rc;
  DS2_LAUNCH(bn2d_finalize_kernel, 1, 32, 0, st, (double)B * D2 * Tp, W.sums + 64, g2, be2, rm2, rv2, training,
             momentum, eps, stats + 64);
  DS2_LAUNCH(bn_act_transpose_kernel, dim3(cdiv(Tp, 32), cdiv(CO * D2, 32), B), dim3(32, 8), 0, st, B, D2, Tp, z2,
             stats + 64, g2, be2, out_len, y);
  return DS2_OK;
}

int ds2_conv_frontend_bwd(int B, int T, const float* x, const int32_t* out_len, const float* w1, const float* g1,
                          const float* be1, const float* w2, const float* g2, const float* be2, const float* z1,
                          const float* a1, const float* z2, const float* stats, const float* dy, float* dw1,
                          float* db1, float* dg1, float* dbe1, float* dw2, float* db2, float* dg2, float* dbe2,
                          void* ws, size_t ws_bytes, void* stream) {
  DS2_REQUIRE(B > 0 && T > 0, "conv bwd: bad shape B=%d T=%d", B, T);
  DS2_REQUIRE(ws_bytes >= ds2_conv_frontend_workspace_bytes(B, T), "conv bwd: workspace too small");
  (void)w1;
  cudaStream_t st = as_stream(stream);
  const int Tp = (T - 1) / 2 + 1, D1 = DS2_CONV1_D, D2 = DS2_CONV2_D;
  ConvWs W;
  conv_ws_carve(B, T, ws, &W);
  double* s2 = W.sums + 128;
  double* s1 = W.sums + 192;
  DS2_PROF("conv_bwd", st);
  DS2_CHECK_CUDA(cudaMemsetAsync(s2, 0, 128 * sizeof(double), st));
  DS2_CHECK_CUDA(cudaMemsetAsync(dw2, 0, sizeof(float) * CO * CO * 21 * 11, st));
  DS2_CHECK_CUDA(cudaMemsetAsync(dw1, 0, sizeof(float) * CO * 41 * 11, st));

  // ---- stage 2: BN2 + Hardtanh + mask backward (dy arrives time-major)
  DS2_LAUNCH(bn_bwd_reduce_kernel<true>, dim3(cdiv(Tp, 32), cdiv(CO * D2, 32), B), dim3(32, 8), 0, st, B, D2, Tp, z2,
             stats + 64, g2, be2, out_len, dy, W.du2, s2);
  DS2_LAUNCH(bn_bwd_params2d_kernel, 1, 32, 0, st, s2, dg2, dbe2);
  DS2_LAUNCH(bn_bwd_apply_kernel, dim3(cdiv(D2 * Tp, 256), CO, B), 256, 0, st, B, D2, Tp, 1.0 / ((double)B * D2 * Tp),
             z2, stats + 64, g2, out_len, s2, W.du2, W.dbpart);
  DS2_LAUNCH(bias_grad_kernel, CO, 256, 0, st, B * cdiv(D2 * Tp, 256), W.dbpart, db2);
  // ---- conv2 gradients.  Nobody needs dW2 before the optimizer: with a side stream set the weight gradient runs there,
  // next to the data gradient and the (elementwise, HBM-bound) BN1 backward of the main stream, and is joined before
  // the conv1 weight gradient reuses its staging buffer.
  cudaStream_t side = as_stream(g_side_stream.load());
  bool forked = false;
  {
    int wrc = 1;
    if (tensor_core_mode() && !getenv("DS2_NO_CONV_TC") && !getenv("DS2_NO_CONV_TC_WGRAD")) {
      cudaStream_t wst = st;
      if (side && Tp % 4 == 0) {
        int frc = side_fork(st, side);
        if (frc) return frc;
        wst = side;
        forked = true;
      }
      wrc = conv2_wgrad_tc(W.du2, a1, W.shifted, B, Tp, dw2, W.wpart, wst);
      if (wrc < 0) return wrc;
      if (forked) {
        int mrc = side_mark_workspace(ws, side);
        if (mrc) return mrc;
      }
    }
    if (wrc == 1) DS2_LAUNCH(conv2_dw_kernel, dim3(21, B), 256, 0, st, B, Tp, W.du2, a1, dw2);
  }
  DS2_LAUNCH(pack_bwd_data_kernel, cdiv(CO * 11 * 11 * CO, 256), 256, 0, st, 0, w2, W.wTe);
  DS2_LAUNCH(pack_bwd_data_kernel, cdiv(CO * 10 * 11 * CO, 256), 256, 0, st, 1, w2, W.wTo);
  // even rows y=2j (41 rows), odd rows y=2j+1 (40 rows) of d(a1) (B,32,81,T')
  const size_t ob = (size_t)CO * D1 * Tp, oc = (size_t)D1 * Tp;
  int rc;
  if (tensor_core_mode() && !getenv("DS2_NO_CONV_TC") && !getenv("DS2_NO_CONV_TC_DGRAD")) {
    // data gradient on tcgen05: rows y=2i use taps kh=2m (d = i+5-m), rows y=2i+1 taps kh=2m+1
    rc = nchw_to_cl(B, D2, Tp, W.du2, W.cl, st);
    if (rc) return rc;
    rc = pack_conv2_tc(w2, nullptr, W.taps_b, st);
    if (rc) return rc;
    rc = conv_tc_run(W.cl, B, Tp, D2, 41, W.taps_b, 21, 11, 1, 5, -1, 0, 2, W.da1, ob, oc, (size_t)Tp, 2, 0, nullptr,
                     nullptr, nullptr, st);
    if (rc) return rc;
    rc = conv_tc_run(W.cl, B, Tp, D2, 40, W.taps_b, 21, 10, 1, 5, -1, 1, 2, W.da1, ob, oc, (size_t)Tp, 2, 1, nullptr,
                     nullptr, nullptr, st);
    if (rc) return rc;
  } else {
    rc = launch_conv<11, 11, 1, 1>(W.du2, B, CO, D2, Tp, W.wTe, nullptr, W.da1, 41, Tp, ob, oc, (size_t)2 * Tp, 5, 5,
                                   nullptr, nullptr, st);
    if (rc) return rc;
    rc = launch_conv<10, 11, 1, 1>(W.du2, B, CO, D2, Tp, W.wTo, nullptr, W.da1 + Tp, 40, Tp, ob, oc, (size_t)2 * Tp, 4, 5,
                                   nullptr, nullptr, st);
    if (rc) return rc;
  }
  // ---- stage 1: BN1 + Hardtanh + mask backward (natural layout, in place over da1)
  DS2_LAUNCH(bn_bwd_reduce_kernel<false>, dim3(cdiv(Tp, 32), cdiv(CO * D1, 32), B), dim3(32, 8), 0, st, B, D1, Tp,
             z1, stats, g1, be1, out_len, W.da1, W.da1, s1);
  DS2_LAUNCH(bn_bwd_params2d_kernel, 1, 32, 0, st, s1, dg1, dbe1);
  DS2_LAUNCH(bn_bwd_apply_kernel, dim3(cdiv(D1 * Tp, 256), CO, B), 256, 0, st, B, D1, Tp, 1.0 / ((double)B * D1 * Tp),
             z1, stats, g1, out_len, s1, W.da1, W.dbpart);
  DS2_LAUNCH(bias_grad_kernel, CO, 256, 0, st, B * cdiv(D1 * Tp, 256), W.dbpart, db1);
  if (forked) {   // dW2 done (and its staging buffer free) before this call returns
    int jrc = side_wait_for_workspace(ws, st);
    if (jrc) return jrc;
  }
  {
    // conv1 weight gradient on tcgen05 (reuses the conv2 weight gradient's staging buffer, which is free by now)
    int wrc = 1;
    if (tensor_core_mode() && !getenv("DS2_NO_CONV_TC") && !getenv("DS2_NO_CONV1_TC_WGRAD")) {
      wrc = conv1_wgrad_tc(W.da1, x, W.shifted, B, T, Tp, dw1, W.wpart, st);
      if (wrc < 0) return wrc;
    }
    if (wrc == 1) DS2_LAUNCH(conv1_dw_kernel, dim3(3, B, C1_DSPLIT), 128, 0, st, B, T, Tp, W.da1, x, dw1);
  }
  return DS2_OK;
}

}  // extern "C"
