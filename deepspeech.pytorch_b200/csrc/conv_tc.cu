// 32->32 channel convolution (conv2 forward and its data gradient) on tcgen05 tensor cores as an
// im2col-free implicit GEMM with the horizontal taps folded into N ("tap-in-N"):
//
//   for an output row and one vertical tap j, with the input row r_j in channels-last layout (t, ci):
//       D[p, (kw, co)] += sum_ci  X[r_j][p][ci] * Wn[j][(kw, co)][ci]          (M = 128 positions p,
//                                                                               N = 11*32 = 352, K = 32)
//   and after all vertical taps   out[t][co] = sum_kw D[t + kw - 5][(kw, co)]   (shifted sum, epilogue)
//
// The A tile of a tap is ONE contiguous TMA box (128 positions x 32 channels = 128-byte rows, 128B
// swizzle, out-of-range rows / positions zero-filled by TMA = the convolution padding), the B tile is
// the packed tap matrix (352 x 32); no descriptor tricks, no im2col buffer.  A tile produces 118
// outputs (128 positions minus the 10-position halo).  Accumulators: 352 TMEM columns (two N=176 MMAs
// per K=8 step).  Epilogue: per kw the 32-column block is read from TMEM and added into a shared-memory
// output tile at row p-kw; then bias, length mask, NCHW store and the BatchNorm sum / sum-of-squares
// partials of the forward pass.
//
// The data gradient of the stride-(2,1) convolution is the same kernel run twice (even / odd output
// rows) with transposed, horizontally flipped taps (see pack kernels below).
#include "common.cuh"
#include "tc_common.cuh"

namespace ds2 {
int make_tmap_4d_f32(CUtensorMap* out, const float* base, const unsigned long long dims[4],
                     const unsigned long long strides_bytes[3], const unsigned int box[4]);
int make_tmap_nd_f32(CUtensorMap* out, const float* base, int rank, const unsigned long long* dims,
                     const unsigned long long* strides_bytes, const unsigned int* box);

namespace cv {
constexpr int CH = 32, KW = 11, NN = KW * CH;      // 352
constexpr int MP = 128, TO = MP - (KW - 1);         // positions per tile, outputs per tile (118)
constexpr int A_BYTES = MP * 128;                   // 16 KB
constexpr int W_HALF = (NN / 2) * 128;              // 176 rows x 128 B = 22528
constexpr int STAGE_BYTES = A_BYTES + 2 * W_HALF;   // 61440
constexpr int STAGES = 3;
constexpr int OUT_LD = 33;
constexpr int THREADS = 192;
constexpr int SMEM_BYTES = 1024 + STAGES * STAGE_BYTES + (TO + 10) * OUT_LD * 4 + 256;
}  // namespace cv

// Warp-converged TMA issue (see tc_common.cuh): 4-D / 5-D boxes of the conv kernels
__device__ __forceinline__ void tma_load_4d_w(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                              int c3) {
  asm volatile(
      "{\n\t.reg .pred pe;\n\telect.sync _|pe, 0xffffffff;\n\t"
      "@pe cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n\t}"
      ::"r"(tc::smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(tc::smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
        "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d_w(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                              int c3, int c4) {
  asm volatile(
      "{\n\t.reg .pred pe;\n\telect.sync _|pe, 0xffffffff;\n\t"
      "@pe cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];\n\t}"
      ::"r"(tc::smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(tc::smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
        "r"(c3), "r"(c4)
      : "memory");
}

struct ConvTcParams {
  CUtensorMap tmA;   // 4-D (32 c, T, R_in, B) channels-last input
  CUtensorMap tmW;   // 3-D (32 c, 352 n, taps) packed tap matrices
  int B, T, R_in, R_out;
  int J;                                   // vertical taps per output row
  int row_mul, row_off, row_step;          // input row  = row_mul * d + row_off + j * row_step
  int w_off, w_step;                       // tap matrix = w_off + j * w_step
  float* out;                              // out[b*ob + c*oc + (out_row_mul*d + out_row_off)*orow + t]
  size_t ob, oc, orow;
  int out_row_mul, out_row_off;
  const float* bias;                       // [32] or null
  const int32_t* out_len;                  // [B] or null: positions t >= out_len[b] are written as 0
  double* stat_sums;                       // [64] or null
};

__global__ void __launch_bounds__(cv::THREADS, 1) conv_tc_kernel(const __grid_constant__ ConvTcParams p) {
  using namespace cv;
  using namespace tc;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  float* out_s = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES);       // [TO+10][33]
  uint64_t* full = reinterpret_cast<uint64_t*>(out_s + (TO + 10) * OUT_LD);   // 128*33 floats: 8-byte aligned
  uint64_t* empty = full + STAGES;
  uint64_t* accum_bar = empty + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);

  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int t0 = blockIdx.x * TO, d = blockIdx.y, b = blockIdx.z;

  // vertical taps whose input row exists (the others contribute zeros: skip them)
  int j_lo = 0, j_hi = p.J;
  {
    const int r0 = p.row_mul * d + p.row_off;
    while (j_lo < j_hi && (r0 + j_lo * p.row_step < 0 || r0 + j_lo * p.row_step >= p.R_in)) ++j_lo;
    while (j_hi > j_lo && (r0 + (j_hi - 1) * p.row_step < 0 || r0 + (j_hi - 1) * p.row_step >= p.R_in)) --j_hi;
  }
  const int nj = j_hi - j_lo;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmA);
    tma_prefetch_desc(&p.tmW);
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(accum_bar, 1);
    fence_barrier_init();
  }
  for (int i = threadIdx.x; i < (TO + 10) * OUT_LD; i += THREADS) out_s[i] = 0.f;
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    int s = 0;
    uint32_t ph = 0;
    for (int jj = 0; jj < nj; ++jj) {
      const int j = j_lo + jj;
      const int r = p.row_mul * d + p.row_off + j * p.row_step;
      const int wi = p.w_off + j * p.w_step;
      mbar_wait(&empty[s], ph ^ 1);
      mbar_arrive_expect_tx_w(&full[s], (uint32_t)STAGE_BYTES);
      uint8_t* st = smem + s * STAGE_BYTES;
      // A: 128 positions starting at t0-5 (negative / beyond-T coordinates are zero-filled = padding)
      tma_load_4d_w(st, &p.tmA, &full[s], 0, t0 - 5, r, b);
      tma_load_3d_w(st + A_BYTES, &p.tmW, &full[s], 0, 0, wi);
      tma_load_3d_w(st + A_BYTES + W_HALF, &p.tmW, &full[s], 0, NN / 2, wi);
      if (++s == STAGES) { s = 0; ph ^= 1; }
    }
  } else if (warp == 1) {
    // the whole warp runs the loop, one elected lane issues (a single divergent lane pays ~76 cycles per MMA
    // in uniform-register round trips; see tc_common.cuh)
    const uint32_t idesc = instr_desc(FMT_TF32, MP, NN / 2);
    int s = 0;
    uint32_t ph = 0;
    for (int jj = 0; jj < nj; ++jj) {
      mbar_wait(&full[s], ph);
      tc_fence_after();
      const uint64_t ad = smem_desc_sw128(smem_u32(smem + s * STAGE_BYTES));
      const uint64_t b0 = smem_desc_sw128(smem_u32(smem + s * STAGE_BYTES + A_BYTES));
      const uint64_t b1 = smem_desc_sw128(smem_u32(smem + s * STAGE_BYTES + A_BYTES + W_HALF));
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        mma_tf32_w(tmem_base, ad + (uint64_t)(2 * k), b0 + (uint64_t)(2 * k), idesc, (jj | k) != 0);
        mma_tf32_w(tmem_base + (uint32_t)(NN / 2), ad + (uint64_t)(2 * k), b1 + (uint64_t)(2 * k), idesc, (jj | k) != 0);
      }
      mma_commit_w(&empty[s]);
      if (++s == STAGES) { s = 0; ph ^= 1; }
    }
    mma_commit_w(accum_bar);
  } else {
    const int q = warp % 4, e = threadIdx.x - 64;
    const int pl = q * 32 + lane;                     // position inside the tile (TMEM lane)
    if (nj > 0) {
      mbar_wait(accum_bar, 0);
      tc_fence_after();
      for (int kw = 0; kw < KW; ++kw) {
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(kw * CH), v);
        const int to = pl - kw;                       // output this position feeds through tap kw
        if (to >= 0 && to < TO) {
          float* row = out_s + to * OUT_LD;
#pragma unroll
          for (int c = 0; c < CH; ++c) row[c] += v[c];
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
    } else {
      asm volatile("bar.sync 1, 128;" ::: "memory");
    }
    // bias, mask, NCHW store: warp q owns channels 8q..8q+7, lanes run along time (128-byte stores);
    // per-channel sum / sum of squares for the BatchNorm of the forward pass
    const int L = p.out_len ? p.out_len[b] : p.T;
    const int orow_idx = p.out_row_mul * d + p.out_row_off;
    (void)e;
    for (int cc = 0; cc < 8; ++cc) {
      const int c = q * 8 + cc;
      const float bv = p.bias ? p.bias[c] : 0.f;
      float* op = p.out + (size_t)b * p.ob + (size_t)c * p.oc + (size_t)orow_idx * p.orow;
      float s1 = 0.f, s2 = 0.f;
      for (int to = lane; to < TO; to += 32) {
        const int t = t0 + to;
        if (t < p.T) {
          const float val = (t < L) ? out_s[to * OUT_LD + c] + bv : 0.f;
          op[t] = val;
          s1 += val;
          s2 = fmaf(val, val, s2);
        }
      }
      if (p.stat_sums) {
        s1 = warp_sum(s1);
        s2 = warp_sum(s2);
        if (lane == 0) {
          atomicAdd(&p.stat_sums[c], (double)s1);
          atomicAdd(&p.stat_sums[CH + c], (double)s2);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<512>(tmem_base);
}

// ---- packing ----------------------------------------------------------------------------------------
// forward taps: Wn[kh][kw*32 + co][ci] = w2[co][ci][kh][kw]
__global__ void pack_conv2_tc_fwd_kernel(const float* __restrict__ w2, float* __restrict__ wn) {
  int i = blockIdx.x * blockDim.x + threadIdx.x, n = 21 * cv::NN * 32;
  if (i >= n) return;
  int ci = i % 32, nn = (i / 32) % cv::NN, kh = i / (32 * cv::NN);
  int kw = nn / 32, co = nn % 32;
  wn[i] = w2[(((size_t)co * 32 + ci) * 21 + kh) * 11 + kw];
}
// data-gradient taps: Wd[kh][kwi*32 + ci][co] = w2[co][ci][kh][10 - kwi]   (K runs over co)
__global__ void pack_conv2_tc_bwd_kernel(const float* __restrict__ w2, float* __restrict__ wd) {
  int i = blockIdx.x * blockDim.x + threadIdx.x, n = 21 * cv::NN * 32;
  if (i >= n) return;
  int co = i % 32, nn = (i / 32) % cv::NN, kh = i / (32 * cv::NN);
  int kwi = nn / 32, ci = nn % 32;
  wd[i] = w2[(((size_t)co * 32 + ci) * 21 + kh) * 11 + (10 - kwi)];
}

// NCHW (B,32,R,T) -> channels-last (B,R,T,32); grid (ceil(T/32), R, B), block (32, 8)
__global__ void nchw_to_cl_kernel(int R, int T, const float* __restrict__ in, float* __restrict__ out) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, r = blockIdx.y, t0 = blockIdx.x * 32;
  for (int c = threadIdx.y; c < 32; c += 8) {
    int t = t0 + threadIdx.x;
    tile[c][threadIdx.x] = (t < T) ? in[(((size_t)b * 32 + c) * R + r) * T + t] : 0.f;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += 8) {
    int t = t0 + j;
    if (t < T) out[(((size_t)b * R + r) * T + t) * 32 + threadIdx.x] = tile[threadIdx.x][j];
  }
}

int nchw_to_cl(int B, int R, int T, const float* in, float* out, cudaStream_t st) {
  DS2_LAUNCH(nchw_to_cl_kernel, dim3(cdiv(T, 32), R, B), dim3(32, 8), 0, st, R, T, in, out);
  return DS2_OK;
}

int pack_conv2_tc(const float* w2, float* wn_fwd, float* wd_bwd, cudaStream_t st) {
  const int n = 21 * cv::NN * 32;
  if (wn_fwd) DS2_LAUNCH(pack_conv2_tc_fwd_kernel, cdiv(n, 256), 256, 0, st, w2, wn_fwd);
  if (wd_bwd) DS2_LAUNCH(pack_conv2_tc_bwd_kernel, cdiv(n, 256), 256, 0, st, w2, wd_bwd);
  return DS2_OK;
}

// 4-D channels-last tensor map (32 c, T, R, B), box (32, 128, 1, 1)
static int make_tmap_cl(CUtensorMap* out, const float* base, int T, int R, int B);

// Runs the 32->32 tap-in-N convolution.  in_cl: (B, R_in, T, 32) channels-last; taps: (n_taps, 352, 32).
int conv_tc_run(const float* in_cl, int B, int T, int R_in, int R_out, const float* taps, int n_taps, int J,
                int row_mul, int row_off, int row_step, int w_off, int w_step, float* out, size_t ob, size_t oc,
                size_t orow, int out_row_mul, int out_row_off, const float* bias, const int32_t* out_len,
                double* stat_sums, cudaStream_t st) {
  ConvTcParams p{};
  int rc = make_tmap_cl(&p.tmA, in_cl, T, R_in, B);
  if (rc) return rc;
  rc = make_tmap_3d(&p.tmW, taps, 32, cv::NN, n_taps, 32, (size_t)32 * cv::NN, 32, cv::NN / 2, 1);
  if (rc) return rc;
  p.B = B; p.T = T; p.R_in = R_in; p.R_out = R_out; p.J = J;
  p.row_mul = row_mul; p.row_off = row_off; p.row_step = row_step; p.w_off = w_off; p.w_step = w_step;
  p.out = out; p.ob = ob; p.oc = oc; p.orow = orow; p.out_row_mul = out_row_mul; p.out_row_off = out_row_off;
  p.bias = bias; p.out_len = out_len; p.stat_sums = stat_sums;
  static DeviceOnce attr_once;
  if (attr_once.first()) {
    DS2_CHECK_CUDA(cudaFuncSetAttribute(conv_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, cv::SMEM_BYTES));
    attr_once.done();
  }
  dim3 grid(cdiv(T, cv::TO), R_out, B);
  DS2_LAUNCH(conv_tc_kernel, grid, cv::THREADS, cv::SMEM_BYTES, st, p);
  return DS2_OK;
}

// ---- weight gradient of conv2 on tensor cores ---------------------------------------------------------
//   dW[co][ci][kh][kw] = sum_{b,d,t} dz2[b,co,d,t] * a1[b,ci,2d+kh-10,t+kw-5]
// GEMM over time (K = t), organised around the INPUT row r = 2d+kh-10: one fetch of the row's eleven shifted tiles
// (B operand, N = (kw,ci) = 352) serves every vertical tap kh of r's parity, whose dz2 rows d = (r+10-kh)/2 are
// stacked in M: a CTA owns a group of 4 taps (M = 4 x 32 co = 128) and a slice of the (b, r) pairs, accumulates them
// all in TMEM (352 columns) and finally stores its 128 x 352 tile into its slice of the partial sums (summed per slice in a fixed order).  Rows d outside the output
// are zero-filled by TMA.  (The first version looped over (b, d) for one kh with M = 32 of 64: every input row was
// fetched once per tap, 19 GB of L2 -> shared-memory traffic per launch = 11 TB/s, the limit; stacking the taps cuts
// it to 7.6 GB and fills the M = 128 data path.)
// The producer needs ~110 cycles per TMA instruction, so the eleven shifted 4 KB tiles are fetched with four boxes
// that span the "shift copy" dimension of a 4-copy tensor (see shift_copies_kernel); the N blocks then sit in the
// order KW_OF_BLOCK.
namespace wg {
constexpr int KT = 32;                               // time steps per K chunk (128 bytes)
constexpr int KH = 21;                               // vertical taps of conv2
constexpr int KH_PER = 4;                            // vertical taps stacked in M
constexpr int GROUPS = 3;                            // tap groups per parity: kh = parity + 2 * (4 * g + i)
constexpr int A_BYTES = KH_PER * 32 * 128;           // 128 M rows
constexpr int B_BYTES = cv::NN * 128;                // 352 rows
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;       // 61440
constexpr int STAGES = 3;
constexpr int THREADS = 192;
constexpr int SMEM_BYTES = 1024 + STAGES * STAGE_BYTES + 256;
}  // namespace wg

struct WgradParams {
  CUtensorMap tmDz;   // 4-D (T, 41, 32 co, B)
  CUtensorMap tmS4;   // 5-D (T+4, 81, 32 ci, B, 4 copies): a1 delayed by 0, 1, 2, 3 time steps; box = 4 copies
  CUtensorMap tmS2;   // same tensor, box = 2 copies
  CUtensorMap tmS1;   // same tensor, box = 1 copy
  int B, T, slices;
  float* part;        // slices x 32*32*21*11: each CTA stores its partial sum, summed per slice in a fixed order
};
// shared-memory N block j (32 ci rows each) holds tap kw = KW_OF_BLOCK[j]:
//   box (t0-4, copies 0,1) -> kw 1,0 | (t0, copies 0..3) -> kw 5,4,3,2 | (t0+4, copies 0..3) -> kw 9,8,7,6 | (t0+8, copy 3) -> kw 10
__constant__ int KW_OF_BLOCK[11] = {1, 0, 5, 4, 3, 2, 9, 8, 7, 6, 10};

// TMA needs 16-byte aligned box starts in the innermost dimension, so a shift by sh = kw-5 time steps is
// split into a multiple of 4 (the box coordinate) and s = 0..3 (which delayed copy is read):
//   a1r[s][row][t'] = a1[row][t'-s]  for t' in [0, T+4)  (0 outside the row; rows padded to T+4 so that the
//   shifted tail stays in bounds),  a1[t + sh] = a1r[s][t + sh + s]  with (sh + s) % 4 == 0.
__global__ void shift_copies_kernel(size_t rows, int T, const float* __restrict__ a1, float* __restrict__ a1r) {
  const int Tp = T + 4;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n = rows * Tp, stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    const int t = (int)(i % Tp);
    const float* src = a1 + (i / Tp) * T;
#pragma unroll
    for (int sft = 0; sft <= 3; ++sft) {
      const int ts = t - sft;
      a1r[(size_t)sft * n + i] = (ts >= 0 && ts < T) ? src[ts] : 0.f;
    }
  }
}

__global__ void __launch_bounds__(wg::THREADS, 1) conv2_wgrad_tc_kernel(const __grid_constant__ WgradParams p) {
  using namespace wg;
  using namespace tc;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* accum_bar = empty + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int parity = blockIdx.x / GROUPS, kh0 = parity + 2 * KH_PER * (blockIdx.x % GROUPS);   // taps kh0 + 2 i
  const int nkh = min(KH_PER, (KH - 1 - kh0) / 2 + 1);
  const int nr = (DS2_CONV1_D - parity + 1) / 2;        // input rows of this parity: r = 2 r' + parity
  const int pairs = p.B * nr;
  const int per = (pairs + (int)gridDim.y - 1) / (int)gridDim.y;
  const int p0 = blockIdx.y * per, p1 = min(pairs, p0 + per);
  const int nkt = (p.T + KT - 1) / KT;
  // a row takes part when at least one of the group's taps has its output row d = (r + 10 - kh) / 2 inside [0, 41)
  auto row_active = [&](int r) {
    const int d_hi = (r + 10 - kh0) / 2, d_lo = (r + 10 - (kh0 + 2 * (nkh - 1))) / 2;   // same parity: exact
    return d_hi >= 0 && d_lo < DS2_CONV2_D;
  };

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmDz);
    tma_prefetch_desc(&p.tmS4);
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(accum_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  int nchunks = 0;
  for (int pi = p0; pi < p1; ++pi)
    if (row_active(2 * (pi % nr) + parity)) nchunks += nkt;

  if (warp == 0) {
    int s = 0;
    uint32_t ph = 0;
    for (int pi = p0; pi < p1; ++pi) {
      const int b = pi / nr, r = 2 * (pi % nr) + parity;
      if (!row_active(r)) continue;
      for (int kt = 0; kt < nkt; ++kt) {
        mbar_wait(&empty[s], ph ^ 1);
        mbar_arrive_expect_tx_w(&full[s], (uint32_t)(nkh * 32 * 128 + cv::NN * 128));
        uint8_t* st = smem + s * STAGE_BYTES;
        for (int i = 0; i < nkh; ++i)    // dz2 rows of the stacked taps; d outside [0, 41) arrives as zeros
          tma_load_4d_w(st + i * 4096, &p.tmDz, &full[s], kt * KT, (r + 10 - kh0) / 2 - i, 0, b);
        uint8_t* nb = st + A_BYTES;                      // N blocks of 32 rows x 128 B
        tma_load_5d_w(nb, &p.tmS2, &full[s], kt * KT - 4, r, 0, b, 0);
        tma_load_5d_w(nb + 2 * 4096, &p.tmS4, &full[s], kt * KT, r, 0, b, 0);
        tma_load_5d_w(nb + 6 * 4096, &p.tmS4, &full[s], kt * KT + 4, r, 0, b, 0);
        tma_load_5d_w(nb + 10 * 4096, &p.tmS1, &full[s], kt * KT + 8, r, 0, b, 3);
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // warp-converged issue (one elected lane), as in conv_tc_kernel
    const uint32_t idesc = instr_desc(FMT_TF32, 128, cv::NN / 2);
    int s = 0;
    uint32_t ph = 0;
    for (int c = 0; c < nchunks; ++c) {
      mbar_wait(&full[s], ph);
      tc_fence_after();
      const uint64_t ad = smem_desc_sw128(smem_u32(smem + s * STAGE_BYTES));
      const uint64_t b0 = smem_desc_sw128(smem_u32(smem + s * STAGE_BYTES + A_BYTES));
      const uint64_t b1 = smem_desc_sw128(smem_u32(smem + s * STAGE_BYTES + A_BYTES + cv::W_HALF));
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        mma_tf32_w(tmem_base, ad + (uint64_t)(2 * k), b0 + (uint64_t)(2 * k), idesc, (c | k) != 0);
        mma_tf32_w(tmem_base + (uint32_t)(cv::NN / 2), ad + (uint64_t)(2 * k), b1 + (uint64_t)(2 * k), idesc, (c | k) != 0);
      }
      mma_commit_w(&empty[s]);
      if (++s == STAGES) { s = 0; ph ^= 1; }
    }
    if (nchunks > 0) mma_commit_w(accum_bar);
  } else if (nchunks > 0) {
    // M = 128: row m = 32 i + co lives in TMEM lane m; warp quadrant q reads tap i = q, lane = co
    const int q = warp % 4;
    mbar_wait(accum_bar, 0);
    tc_fence_after();
    if (q < nkh) {      // rows of taps beyond the last one were never loaded
      const int kh = kh0 + 2 * q, co = lane;
      for (int blk = 0; blk < cv::KW; ++blk) {
        const int kw = KW_OF_BLOCK[blk];
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(blk * 32), v);
#pragma unroll
        for (int ci = 0; ci < 32; ++ci)
          p.part[(size_t)blockIdx.y * (32 * 32 * KH * 11) + (((size_t)co * 32 + ci) * KH + kh) * 11 + kw] = v[ci];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<512>(tmem_base);
}

// out[e] = sum_s part[s * n + e], s in increasing order: the weight gradients do not depend on which CTA finishes first
__global__ void sum_slices_kernel(size_t n, int slices, const float* __restrict__ part, float* __restrict__ out) {
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    float acc = 0.f;
    for (int s = 0; s < slices; ++s) acc += part[(size_t)s * n + e];
    out[e] = acc;
  }
}

constexpr int WGRAD_SLICES = 24;
// dz2: (B,32,41,T) NCHW gate... conv2 output gradient; a1: (B,32,81,T) NCHW; dw2 (32,32,21,11) is overwritten;
// part: conv_wgrad_tc_part_floats() floats.
// Returns 1 when the shape is not eligible (row pitch T*4 bytes must be a multiple of 16).
int conv2_wgrad_tc(const float* dz2, const float* a1, float* a1_shifted /* 4*B*32*81*(T+4) floats */, int B, int T,
                   float* dw2, float* part, cudaStream_t st) {
  if (T % 4 != 0) return 1;
  WgradParams p{};
  {
    const size_t rows = (size_t)B * 32 * 81;
    DS2_LAUNCH(shift_copies_kernel, 148 * 8, 256, 0, st, rows, T, a1, a1_shifted);
    const unsigned long long Tq = (unsigned long long)T + 4;
    unsigned long long dims[5] = {Tq, 81ull, 32ull, (unsigned long long)B, 4ull};
    unsigned long long str[4] = {Tq * 4, 81ull * Tq * 4, 32ull * 81 * Tq * 4, (unsigned long long)rows * Tq * 4};
    unsigned int box[5] = {32u, 1u, 32u, 1u, 4u};
    int rc = make_tmap_nd_f32(&p.tmS4, a1_shifted, 5, dims, str, box);
    if (rc) return rc;
    box[4] = 2u;
    rc = make_tmap_nd_f32(&p.tmS2, a1_shifted, 5, dims, str, box);
    if (rc) return rc;
    box[4] = 1u;
    rc = make_tmap_nd_f32(&p.tmS1, a1_shifted, 5, dims, str, box);
    if (rc) return rc;
  }
  {
    unsigned long long dims[4] = {(unsigned long long)T, 41ull, 32ull, (unsigned long long)B};
    unsigned long long str[3] = {(unsigned long long)T * 4, (unsigned long long)41 * T * 4, (unsigned long long)32 * 41 * T * 4};
    unsigned int box[4] = {32u, 1u, 32u, 1u};
    int rc = make_tmap_4d_f32(&p.tmDz, dz2, dims, str, box);
    if (rc) return rc;
  }
  p.B = B; p.T = T; p.slices = WGRAD_SLICES; p.part = part;   // 2 parities x 3 tap groups x 24 slices = 144 CTAs
  const size_t n = (size_t)32 * 32 * 21 * 11;
  DS2_CHECK_CUDA(cudaMemsetAsync(part, 0, sizeof(float) * n * p.slices, st));
  static DeviceOnce attr_once;
  if (attr_once.first()) {
    DS2_CHECK_CUDA(cudaFuncSetAttribute(conv2_wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, wg::SMEM_BYTES));
    attr_once.done();
  }
  DS2_LAUNCH(conv2_wgrad_tc_kernel, dim3(2 * wg::GROUPS, p.slices), wg::THREADS, wg::SMEM_BYTES, st, p);
  DS2_LAUNCH(sum_slices_kernel, cdiv((int)n, 256), 256, 0, st, n, p.slices, part, dw2);
  return DS2_OK;
}

// ---- weight gradient of conv1 (1 -> 32 channels, 41 x 11 taps, stride 2 x 2) on tensor cores -----------------
//   dW1[co][kh][kw] = sum_{b,d,t} dz1[b,co,d,t] * x[b, 2d+kh-20, 2t+kw-5]
// GEMM over time (K = t) between four stacked output rows (M = (co, i): dz1 rows d0..d0+3) and eight stacked input
// rows (N = (tap column, j): x rows r0..r0+7, each in its twelve time-shifted / de-interleaved variants), so that one
// MMA chunk covers 32 (i, j) pairs = 14 vertical taps kh = 8c + j - 2i of class c (r0 = 2 d0 - 20 + 8c; six classes
// cover kh = 0..40).  The stride-2 time axis is de-interleaved (q = parity of 2t+kw-5) and, because TMA boxes start
// on 16-byte boundaries, kept in four delayed copies s (conv1_shift_copies_kernel):
//   xs[s][q][b][r][u'] = x[b][r][2(u'-s)+q],   x[2t+kw-5] = xs[s][q][t + m + s]  with kw-5 = 2m+q, (m+s) % 4 == 0
// Two boxes per chunk fetch all of them: (t0; s=0..3, q=0..1) and (t0+4; s=2..3, q=0..1); shared-memory N row
// n = (2s+q) * 8 + j  resp.  64 + (2(s-2)+q) * 8 + j, whose tap column is KW1_OF_GROUP[n / 8].  Rows outside the
// image / the output arrive as TMA zero fill.  37 GFLOP: 1.38 ms on FFMA (shared-memory bound) before.
namespace w1 {
constexpr int KT = 32;                               // time steps per K chunk (128 bytes)
constexpr int DI = 4, RJ = 8;                        // stacked output rows / input rows
constexpr int NROWS = 12 * RJ;                       // 96 N rows (11 tap columns + 1 unused variant)
constexpr int CLASSES = 6;
constexpr int A_BYTES = 32 * DI * 128;               // 128 M rows
constexpr int B_BYTES = NROWS * 128;                 // 12 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;       // 28672
constexpr int STAGES = 6;
constexpr int THREADS = 192;
constexpr int SMEM_BYTES = 1024 + STAGES * STAGE_BYTES + 256;
}  // namespace w1
__constant__ int KW1_OF_GROUP[12] = {5, 6, 3, 4, 1, 2, -1, 0, 9, 10, 7, 8};

struct Wgrad1Params {
  CUtensorMap tmDz;   // 4-D (T', 81, 32 co, B), box (32, 4, 32, 1)
  CUtensorMap tmX8;   // 5-D (T'+4, 161, B, 2 q, 4 s), box (32, 8, 1, 2, 4)
  CUtensorMap tmX4;   // same tensor, box (32, 8, 1, 2, 2)
  int B, Tp;
  float* part;        // (24 slices x DI output rows) x 32*41*11, summed in a fixed order like conv2's
};

__global__ void conv1_shift_copies_kernel(int B, int T, int Tp, const float* __restrict__ x, float* __restrict__ xs) {
  const int U = Tp + 4;
  const size_t rows = (size_t)B * DS2_NUM_FREQ, n = rows * U, total = 8 * n;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int up = (int)(i % U);
    const size_t row = (i / U) % rows;
    const int sq = (int)(i / n), q = sq & 1, sft = sq >> 1;
    const int u = up - sft, tx = 2 * u + q;
    xs[i] = (u >= 0 && tx < T) ? x[row * T + tx] : 0.f;
  }
}

__global__ void __launch_bounds__(w1::THREADS, 1) conv1_wgrad_tc_kernel(const __grid_constant__ Wgrad1Params p) {
  using namespace w1;
  using namespace tc;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* accum_bar = empty + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int cls = blockIdx.x;
  const int ndb = (DS2_CONV1_D + DI - 1) / DI;              // 21 blocks of output rows
  const int pairs = p.B * ndb;
  const int per = (pairs + (int)gridDim.y - 1) / (int)gridDim.y;
  const int p0 = blockIdx.y * per, p1 = min(pairs, p0 + per);
  const int nkt = (p.Tp + KT - 1) / KT;
  auto block_active = [&](int db) {   // some input row of the block lies inside the image
    const int r0 = 2 * DI * db - 20 + RJ * cls;
    return r0 + RJ - 1 >= 0 && r0 < DS2_NUM_FREQ;
  };

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmDz);
    tma_prefetch_desc(&p.tmX8);
    tma_prefetch_desc(&p.tmX4);
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(accum_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<128>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  int nchunks = 0;
  for (int pi = p0; pi < p1; ++pi)
    if (block_active(pi % ndb)) nchunks += nkt;

  if (warp == 0) {
    int s = 0;
    uint32_t ph = 0;
    for (int pi = p0; pi < p1; ++pi) {
      const int b = pi / ndb, db = pi % ndb;
      if (!block_active(db)) continue;
      const int d0 = DI * db, r0 = 2 * d0 - 20 + RJ * cls;
      for (int kt = 0; kt < nkt; ++kt) {
        mbar_wait(&empty[s], ph ^ 1);
        mbar_arrive_expect_tx_w(&full[s], (uint32_t)STAGE_BYTES);
        uint8_t* st = smem + s * STAGE_BYTES;
        tma_load_4d_w(st, &p.tmDz, &full[s], kt * KT, d0, 0, b);                       // rows m = co * 4 + i
        tma_load_5d_w(st + A_BYTES, &p.tmX8, &full[s], kt * KT, r0, b, 0, 0);           // 64 rows
        tma_load_5d_w(st + A_BYTES + 64 * 128, &p.tmX4, &full[s], kt * KT + 4, r0, b, 0, 2);   // 32 rows
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = instr_desc(FMT_TF32, 128, NROWS);
    int s = 0;
    uint32_t ph = 0;
    for (int c = 0; c < nchunks; ++c) {
      mbar_wait(&full[s], ph);
      tc_fence_after();
      const uint64_t ad = smem_desc_sw128(smem_u32(smem + s * STAGE_BYTES));
      const uint64_t bd = smem_desc_sw128(smem_u32(smem + s * STAGE_BYTES + A_BYTES));
#pragma unroll
      for (int k = 0; k < 4; ++k) mma_tf32_w(tmem_base, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (c | k) != 0);
      mma_commit_w(&empty[s]);
      if (++s == STAGES) { s = 0; ph ^= 1; }
    }
    if (nchunks > 0) mma_commit_w(accum_bar);
  } else if (nchunks > 0) {
    // accumulator row m = co * 4 + i sits in TMEM lane m
    const int q = warp % 4, m = q * 32 + lane, co = m / DI, i = m % DI;
    mbar_wait(accum_bar, 0);
    tc_fence_after();
    for (int blk = 0; blk < NROWS / 32; ++blk) {
      float v[32];
      tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(blk * 32), v);
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        const int n = blk * 32 + c, kw = KW1_OF_GROUP[n / RJ], kh = RJ * cls + (n % RJ) - 2 * i;
        if (kw >= 0 && kh >= 0 && kh < 41)
          p.part[((size_t)blockIdx.y * DI + i) * (32 * 41 * 11) + ((size_t)co * 41 + kh) * 11 + kw] = v[c];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<128>(tmem_base);
}

size_t conv_wgrad_tc_part_floats() {
  const size_t n2 = (size_t)32 * 32 * 21 * 11, n1 = (size_t)w1::DI * 32 * 41 * 11;
  return (size_t)WGRAD_SLICES * (n2 > n1 ? n2 : n1);
}

// dz1: (B,32,81,T') gradient of the conv1 output (after the BN1 / Hardtanh backward); x: (B,1,161,T); dw1 (32,1,41,11)
// is overwritten.  xs: 8 * B * 161 * (T'+4) floats; part: conv_wgrad_tc_part_floats() floats.  Returns 1 when the
// shape is not eligible (T' % 4 != 0).
int conv1_wgrad_tc(const float* dz1, const float* x, float* xs, int B, int T, int Tp, float* dw1, float* part,
                   cudaStream_t st) {
  if (Tp % 4 != 0) return 1;
  Wgrad1Params p{};
  const unsigned long long U = (unsigned long long)Tp + 4, F = DS2_NUM_FREQ;
  DS2_LAUNCH(conv1_shift_copies_kernel, 148 * 8, 256, 0, st, B, T, Tp, x, xs);
  {
    unsigned long long dims[5] = {U, F, (unsigned long long)B, 2ull, 4ull};
    unsigned long long str[4] = {U * 4, F * U * 4, (unsigned long long)B * F * U * 4, 2ull * B * F * U * 4};
    unsigned int box[5] = {32u, (unsigned int)w1::RJ, 1u, 2u, 4u};
    int rc = make_tmap_nd_f32(&p.tmX8, xs, 5, dims, str, box);
    if (rc) return rc;
    box[4] = 2u;
    rc = make_tmap_nd_f32(&p.tmX4, xs, 5, dims, str, box);
    if (rc) return rc;
  }
  {
    unsigned long long dims[4] = {(unsigned long long)Tp, (unsigned long long)DS2_CONV1_D, 32ull, (unsigned long long)B};
    unsigned long long str[3] = {(unsigned long long)Tp * 4, (unsigned long long)DS2_CONV1_D * Tp * 4,
                                 32ull * DS2_CONV1_D * Tp * 4};
    unsigned int box[4] = {32u, (unsigned int)w1::DI, 32u, 1u};
    int rc = make_tmap_4d_f32(&p.tmDz, dz1, dims, str, box);
    if (rc) return rc;
  }
  p.B = B; p.Tp = Tp; p.part = part;
  const size_t n = (size_t)32 * 41 * 11;
  const int slices = WGRAD_SLICES * w1::DI;
  DS2_CHECK_CUDA(cudaMemsetAsync(part, 0, sizeof(float) * n * slices, st));
  static DeviceOnce attr_once;
  if (attr_once.first()) {
    DS2_CHECK_CUDA(cudaFuncSetAttribute(conv1_wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, w1::SMEM_BYTES));
    attr_once.done();
  }
  DS2_LAUNCH(conv1_wgrad_tc_kernel, dim3(w1::CLASSES, WGRAD_SLICES), w1::THREADS, w1::SMEM_BYTES, st, p);
  DS2_LAUNCH(sum_slices_kernel, cdiv((int)n, 256), 256, 0, st, n, slices, part, dw1);
  return DS2_OK;
}

}  // namespace ds2

// tensor-map helper lives next to the other encoders (needs the driver entry point loaded in gemm_tc.cu)
namespace ds2 {
int make_tmap_4d_f32(CUtensorMap* out, const float* base, const unsigned long long dims[4],
                     const unsigned long long strides_bytes[3], const unsigned int box[4]);
static int make_tmap_cl(CUtensorMap* out, const float* base, int T, int R, int B) {
  unsigned long long dims[4] = {32ull, (unsigned long long)T, (unsigned long long)R, (unsigned long long)B};
  unsigned long long str[3] = {128ull, (unsigned long long)T * 128ull, (unsigned long long)R * T * 128ull};
  unsigned int box[4] = {32u, (unsigned int)cv::MP, 1u, 1u};
  return make_tmap_4d_f32(out, base, dims, str, box);
}
}  // namespace ds2
