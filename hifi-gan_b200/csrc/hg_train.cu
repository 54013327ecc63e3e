// hg_train.cu — the bandwidth-bound pieces of the training step (UPSTREAM train.py restated in SURVEY.md §3.3;
// every op below is what torch autograd / torch.optim would run for the reference's src/models.py modules):
//   * bias gradients (column sums)
//   * conv_post + tanh backward (src/models.py:112-114), the Cin = 1 / Cout = 1 discriminator ends' backward
//     (src/models.py:134,141,146-151,196,204), AvgPool1d(4,2,2) backward (:227-230)
//   * loss gradients (src/models.py:251-282 + the mel L1), L1 sums over internal bf16 feature maps
//   * the single-layer weight preparation and weight-gradient finishes (dgrad / discriminator packs, unpacking of
//     hg_conv1d_wgrad results to the parameter layout, weight_norm backward = torch._weight_norm_interface_backward;
//     reparametrisation at src/models.py:16-31,81,86-88,96,132-140): one job of hg_batched.cu each
//   * AdamW (torch.optim.AdamW semantics, decoupled weight decay), and the gradient norm of
//     torch.nn.utils.clip_grad_norm_ with the skip of a non-finite step that guards it
#include "hg_common.cuh"

#include <atomic>

#include "../../include/hifigan_b200.h"

extern std::atomic<int64_t> g_hg_launches;

namespace {

inline cudaStream_t S(void* s) { return static_cast<cudaStream_t>(s); }
inline void count() { g_hg_launches.fetch_add(1, std::memory_order_relaxed); }

__device__ __forceinline__ float warp_sum(float v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float sgn(float d) { return d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f); }

// out[c] (+)= sum over (b, t < t_valid) of x[b][t][c];  x bf16 [B][t_rows][C]
// thread = (row lane, 8-channel vector); a block reduces its rows in registers, then across row lanes through
// shared memory, and issues ONE atomic per channel.
__global__ void __launch_bounds__(256)
colsum_kernel(const __nv_bfloat16* __restrict__ x, int t_valid, int t_rows, int c, int rows_per_block,
              float* __restrict__ out) {
  extern __shared__ float part[];                // [lanes][c]
  const int vecs = c / 8;
  const int b = blockIdx.y;
  const int r0 = blockIdx.x * rows_per_block;
  const int r1 = min(t_valid, r0 + rows_per_block);
  const int lanes = blockDim.x / vecs;           // rows processed in parallel (vecs <= 256)
  const int vq = threadIdx.x % vecs, rl = threadIdx.x / vecs;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (rl < lanes) {
    for (int r = r0 + rl; r < r1; r += lanes) {
      const uint4 v = *reinterpret_cast<const uint4*>(x + (static_cast<size_t>(b) * t_rows + r) * c + vq * 8);
      const float2 a0 = hg::unpack_bf16x2(v.x), a1 = hg::unpack_bf16x2(v.y), a2 = hg::unpack_bf16x2(v.z),
                   a3 = hg::unpack_bf16x2(v.w);
      acc[0] += a0.x; acc[1] += a0.y; acc[2] += a1.x; acc[3] += a1.y;
      acc[4] += a2.x; acc[5] += a2.y; acc[6] += a3.x; acc[7] += a3.y;
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) part[rl * c + vq * 8 + e] = acc[e];
  }
  __syncthreads();
  for (int ch = threadIdx.x; ch < c; ch += blockDim.x) {
    float sum = 0.f;
    for (int l = 0; l < lanes; ++l) sum += part[l * c + ch];
    atomicAdd(out + ch, sum);
  }
}

// conv_post + tanh backward, data half: dpre = dy * (1 - y^2);
// dx[b,t,c] = dx_scale * lrelu'(x[b,t,c]; slope) * sum_j dpre[b, t - j + pad] * w[c][j]  (x = the activated conv_post input)
// bsum*[c] += sum_{b,t} dx[b,t,c] in fp32 (the bias gradient of the convs that produced x's pre-activation)
__global__ void __launch_bounds__(256)
conv_post_bwd_dx_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w,
                        const float* __restrict__ y, const float* __restrict__ dy, int t, int c, int k,
                        float slope, float dx_scale, __nv_bfloat16* __restrict__ dx, float* __restrict__ dpre_out,
                        float* __restrict__ bsum0, float* __restrict__ bsum1, float* __restrict__ bsum2) {
  extern __shared__ float smf[];
  float* ws = smf;                 // [c][k]
  float* dp = smf + c * k;         // [256 + k - 1]
  float* cs = dp + 256 + k - 1;    // [c] column sums of the block
  const int b = blockIdx.y, t0 = blockIdx.x * 256, pad = k / 2;
  for (int i = threadIdx.x; i < c * k; i += blockDim.x) ws[i] = w[i];
  for (int i = threadIdx.x; i < c; i += blockDim.x) cs[i] = 0.f;
  for (int i = threadIdx.x; i < 256 + k - 1; i += blockDim.x) {
    const int tt = t0 + i - (k - 1 - pad);
    float v = 0.f;
    if (tt >= 0 && tt < t) {
      const float yy = y[static_cast<size_t>(b) * t + tt];
      v = dy[static_cast<size_t>(b) * t + tt] * (1.f - yy * yy);
    }
    dp[i] = v;
  }
  __syncthreads();
  const int tt = t0 + threadIdx.x;
  const bool live = tt < t;
  const int lane = threadIdx.x & 31;
  if (live && dpre_out) dpre_out[static_cast<size_t>(b) * t + tt] = dp[threadIdx.x + (k - 1 - pad)];
  const __nv_bfloat16* xr = x + (static_cast<size_t>(b) * t + (live ? tt : 0)) * c;
  __nv_bfloat16* dr = dx + (static_cast<size_t>(b) * t + (live ? tt : 0)) * c;
  for (int c0 = 0; c0 < c; c0 += 8) {
    float g8[8];
    if (live) {
      const uint4 xv = *reinterpret_cast<const uint4*>(xr + c0);
      const uint32_t xw[4] = {xv.x, xv.y, xv.z, xv.w};
      uint32_t ow[4];
#pragma unroll
      for (int h = 0; h < 4; ++h) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int cc = c0 + 2 * h + e;
          float a = 0.f;
          // input position tt feeds output tt - j + pad through tap j
          for (int j = 0; j < k; ++j) a += dp[threadIdx.x + (k - 1 - pad) - j + pad] * ws[cc * k + j];
          g8[2 * h + e] = a * dx_scale;
        }
        const float2 xs = hg::unpack_bf16x2(xw[h]);
        if (!(xs.x > 0.f)) g8[2 * h] *= slope;
        if (!(xs.y > 0.f)) g8[2 * h + 1] *= slope;
        ow[h] = hg::pack_bf16x2(g8[2 * h], g8[2 * h + 1]);
      }
      *reinterpret_cast<uint4*>(dr + c0) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) g8[e] = 0.f;
    }
    if (bsum0) {
      int col;
      const float sum = hg::warp_colsum<8>(g8, lane, col);
      if (!(lane & 3)) atomicAdd(cs + c0 + col, sum);
    }
  }
  if (bsum0) {
    __syncthreads();
    for (int i = threadIdx.x; i < c; i += blockDim.x) {
      const float sum = cs[i];
      atomicAdd(bsum0 + i, sum);
      if (bsum1) atomicAdd(bsum1 + i, sum);
      if (bsum2) atomicAdd(bsum2 + i, sum);
    }
  }
}

// weight half: dw[c][j] += sum_{b,t} dpre[b,t] * x[b, t + j - pad, c];  db += sum dpre
__global__ void __launch_bounds__(256)
conv_post_bwd_dw_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ dpre, int t, int c, int k,
                        int tile, float* __restrict__ dw, float* __restrict__ db) {
  extern __shared__ float smf[];
  float* dp = smf;                                   // [tile]
  __shared__ float red[32];
  const int b = blockIdx.y, t0 = blockIdx.x * tile, pad = k / 2;
  float bsum = 0.f;
  for (int i = threadIdx.x; i < tile; i += blockDim.x) {
    const int tt = t0 + i;
    const float v = tt < t ? dpre[static_cast<size_t>(b) * t + tt] : 0.f;
    dp[i] = v;
    bsum += v;
  }
  __syncthreads();
  bsum = hg::block_sum(bsum, red);
  if (threadIdx.x == 0 && db) atomicAdd(db, bsum);
  for (int idx = threadIdx.x; idx < c * k; idx += blockDim.x) {
    const int j = idx / c, cc = idx % c;             // adjacent threads read adjacent channels
    float a = 0.f;
    for (int i = 0; i < tile; ++i) {
      const int ti = t0 + i + j - pad;
      if (ti >= 0 && ti < t) a += dp[i] * __bfloat162float(x[(static_cast<size_t>(b) * t + ti) * c + cc]);
    }
    atomicAdd(dw + cc * k + j, a);
  }
}

// discriminator conv_post (Cout = 1) backward.
// data half: dx[s,h,c] = (sum_j dl[s, h - j + pad] * w[c][j] + fm_coef * sgn(fm_g - fm_r) + pre_add) * lrelu'(x[s,h,c])
// A block owns kLastRows positions of one sequence; bsum[c] += sum dx[s,h,c] in fp32 (one atomic per channel per
// block): the bias gradient of the layer that produced x.
constexpr int kLastRows = 16;
__global__ void __launch_bounds__(256)
disc_last_bwd_dx_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w,
                        const float* __restrict__ dl, int h, int h_rows, int c, int k, float slope,
                        const __nv_bfloat16* __restrict__ fm_r, float fm_coef,
                        const __nv_bfloat16* __restrict__ pre_add, __nv_bfloat16* __restrict__ dx,
                        float* __restrict__ bsum) {
  const int s = blockIdx.y, h0 = blockIdx.x * kLastRows, pad = k / 2;
  const int h1 = min(h, h0 + kLastRows);
  __shared__ float dls[kLastRows + 8];
  for (int i = threadIdx.x; i < kLastRows + 8; i += blockDim.x) {
    const int o = h0 - 4 + i;
    dls[i] = (o >= 0 && o < h) ? dl[static_cast<size_t>(s) * h + o] : 0.f;
  }
  __syncthreads();
  for (int cc = threadIdx.x; cc < c; cc += blockDim.x) {
    float wk[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) wk[j] = j < k ? w[cc * k + j] : 0.f;
    float csum = 0.f;
    for (int ho = h0; ho < h1; ++ho) {
      const size_t off = (static_cast<size_t>(s) * h_rows + ho) * c + cc;
      float a = 0.f;
#pragma unroll
      for (int j = 0; j < 7; ++j)
        if (j < k) a += dls[ho - h0 + 4 - j + pad] * wk[j];                    // k <= 7, pad = k / 2: index in [1, 22]
      const float xv = __bfloat162float(x[off]);
      if (fm_r) a += fm_coef * sgn(xv - __bfloat162float(fm_r[off]));
      if (pre_add) a += __bfloat162float(pre_add[off]);
      if (!(xv > 0.f)) a *= slope;
      dx[off] = __float2bfloat16(a);
      csum += a;
    }
    if (bsum) atomicAdd(bsum + cc, csum);
  }
}
// weight half: dw[c][j] += sum_{s,h} dl[s,h] * x[s, h + j - pad, c]; db += sum dl.
// Thread = (channel pair, row lane): a block covers 256 channels with two row lanes, blockIdx.y strides over the
// flat (sequence, position) list, so every thread sees a short chain of independent loads; the two lanes meet in
// shared memory and issue one atomic per (channel, tap).
__global__ void __launch_bounds__(256)
disc_last_bwd_dw_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ dl, int nseq, int h,
                        int h_rows, int c, int k, float* __restrict__ dw, float* __restrict__ db) {
  __shared__ float part[128][17];
  const int cp = threadIdx.x & 127, lane = threadIdx.x >> 7;
  const int c0 = blockIdx.x * 256 + cp * 2;
  const int pad = k / 2;
  const int total = nseq * h;
  const int q0 = blockIdx.y * 2 + lane, qstep = gridDim.y * 2;
  float acc[8][2];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j][0] = acc[j][1] = 0.f;
  float bsum = 0.f;
  const bool live = c0 < c;
  for (int q = q0; q < total; q += qstep) {
    const int s = q / h, ho = q - s * h;
    const float d = dl[q];
    bsum += d;
    if (live) {
      const __nv_bfloat16* xs = x + static_cast<size_t>(s) * h_rows * c + c0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int hi = ho + j - pad;
        if (j < k && hi >= 0 && hi < h) {
          const float2 v = hg::unpack_bf16x2(*reinterpret_cast<const uint32_t*>(xs + static_cast<size_t>(hi) * c));
          acc[j][0] += d * v.x;
          acc[j][1] += d * v.y;
        }
      }
    }
  }
  if (lane == 1) {
#pragma unroll
    for (int j = 0; j < 8; ++j) { part[cp][2 * j] = acc[j][0]; part[cp][2 * j + 1] = acc[j][1]; }
    part[cp][16] = bsum;
  }
  __syncthreads();
  if (lane == 0) {
    if (live) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (j < k) {
          atomicAdd(dw + static_cast<size_t>(c0) * k + j, acc[j][0] + part[cp][2 * j]);
          atomicAdd(dw + static_cast<size_t>(c0 + 1) * k + j, acc[j][1] + part[cp][2 * j + 1]);
        }
      }
    }
    // every channel pair of a lane accumulated the same bsum; one thread of the first channel block reports it
    if (blockIdx.x == 0 && cp == 0 && db) atomicAdd(db, bsum + part[0][16]);
  }
}

// discriminator first conv (Cin = 1) backward.  dpre bf16 [S][h_rows][cout] is the gradient at the conv output
// (leaky_relu mask already applied by the producer).
//   dw[co][j] += sum dpre[s,ho,co] * yin(s, ho*stride + j - pad);  db[co] += sum dpre
//   dy[b, i]  += sum_{co,j} dpre[s,ho,co] * w[co][j]   (reflect-padded tail folded back, src/models.py:146-151)
// A block walks kFirstChunk output positions of one sequence in tiles of 128: the dpre tile and the k input
// samples of every position are staged in shared memory; the weight gradient is a [cout x 128] x [128 x (k+1)]
// product accumulated in registers across tiles (column k is the bias), the audio gradient one thread pair per
// position.  One atomic per output per block.
constexpr int kFirstTile = 128;
constexpr int kFirstChunk = 256;    // 2 tiles per block: the MSD launches (16-32 sequences of 8192) fill the GPU (was 1024: 48-128 blocks)
constexpr int kFirstK = 16;
constexpr int kXPitch = 20;   // floats per staged input row (16-byte multiple)

__global__ void __launch_bounds__(256)
disc_first_bwd_kernel(const float* __restrict__ y, const float* __restrict__ w, const __nv_bfloat16* __restrict__ dpre,
                      int t, int period, int h_in, int h_out, int h_rows, int k, int stride, int pad, int cout,
                      float* __restrict__ dw, float* __restrict__ db, float* __restrict__ dy) {
  extern __shared__ __align__(16) uint8_t smb[];
  const int pitch = cout + 2;                                   // odd word pitch: column reads are conflict-free
  float* ws = reinterpret_cast<float*>(smb);                    // [kFirstK][cout], zero for taps >= k
  float* xin = ws + kFirstK * cout;                             // [tile][kXPitch]: taps, then 1 (bias) at column k
  int* xidx = reinterpret_cast<int*>(xin + kFirstTile * kXPitch);   // [tile][kFirstK]
  float* gsm = reinterpret_cast<float*>(xidx + kFirstTile * kFirstK);          // [2][tile][kFirstK] tap sums
  __nv_bfloat16* dp = reinterpret_cast<__nv_bfloat16*>(gsm + 2 * kFirstTile * kFirstK);   // [tile][pitch]
  const int tid = threadIdx.x;
  if (dy) {
    for (int i = tid; i < kFirstK * cout; i += 256) {
      const int j = i / cout, co = i % cout;
      ws[i] = j < k ? w[co * k + j] : 0.f;
    }
  }
  const int seq = blockIdx.y;
  const int b = seq / period, wcol = seq % period;
  const int p0 = blockIdx.x * kFirstChunk;
  const int p1 = min(h_out, p0 + kFirstChunk);
  // weight-gradient register tile: thread = (4 channels, 4 columns of [taps | bias], row group)
  const int cgs = cout / 4;
  const int cg = tid % cgs, jg = (tid / cgs) & 3, rh = tid / cout, rgroups = 256 / cout;
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[a][c] = 0.f;
  for (int q0 = p0; q0 < p1; q0 += kFirstTile) {
    __syncthreads();
    // stage dpre rows (zero past the end) and the input samples of each position
    const int vec_per_row = cout / 2;                           // bf16x2 words
    for (int i = tid; i < kFirstTile * vec_per_row; i += 256) {
      const int r = i / vec_per_row, v = i % vec_per_row;
      const int ho = q0 + r;
      uint32_t val = 0;
      if (ho < p1) val = reinterpret_cast<const uint32_t*>(dpre + (static_cast<size_t>(seq) * h_rows + ho) * cout)[v];
      reinterpret_cast<uint32_t*>(dp + r * pitch)[v] = val;
    }
    for (int i = tid; i < kFirstTile * kFirstK; i += 256) {
      const int r = i / kFirstK, j = i % kFirstK;
      const int ho = q0 + r;
      float v = 0.f;
      int idx = -1;
      if (j == k) {
        v = ho < p1 ? 1.f : 0.f;
      } else if (j < k && ho < p1) {
        const int hh = ho * stride + j - pad;
        if (hh >= 0 && hh < h_in) {
          int ii = hh * period + wcol;
          if (ii >= t) ii = 2 * (t - 1) - ii;
          idx = ii;
          v = y[static_cast<size_t>(b) * t + ii];
        }
      }
      xin[r * kXPitch + j] = v;
      xidx[i] = idx;
    }
    __syncthreads();
    if (dw && rh < rgroups) {
      // [4 channels] x [4 columns] outer products per staged row: 6 shared-memory loads feed 16 FMAs
      for (int r = rh; r < kFirstTile; r += rgroups) {
        const uint32_t* dr = reinterpret_cast<const uint32_t*>(dp + r * pitch) + cg * 2;
        const float2 d01 = hg::unpack_bf16x2(dr[0]), d23 = hg::unpack_bf16x2(dr[1]);
        const float4 xv = *reinterpret_cast<const float4*>(xin + r * kXPitch + jg * 4);
        const float dv[4] = {d01.x, d01.y, d23.x, d23.y};
        const float xc[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int c = 0; c < 4; ++c) acc[a][c] += dv[a] * xc[c];
      }
    }
    if (dy) {
      // phase A: per output position, G[j] = sum_co dpre[co] * w[co][j] (two threads per position, half of the
      // channels each); phase B: every INPUT row of the tile gathers its taps from G -> one atomic per input row
      const int r = tid & (kFirstTile - 1), half = tid >> 7;
      float gy[kFirstK];
#pragma unroll
      for (int j = 0; j < kFirstK; ++j) gy[j] = 0.f;
      if (q0 + r < p1) {
        const int c0 = half * (cout / 2), c1 = c0 + cout / 2;
        const __nv_bfloat16* drow = dp + r * pitch;
#pragma unroll 2
        for (int co = c0; co < c1; ++co) {
          const float d = __bfloat162float(drow[co]);
          const float* wc = ws + co;
#pragma unroll
          for (int j = 0; j < kFirstK; ++j) gy[j] += d * wc[j * cout];   // taps >= k hold zero weights: no predicate
        }
      }
#pragma unroll
      for (int j = 0; j < kFirstK; ++j) gsm[(half * kFirstTile + r) * kFirstK + j] = gy[j];
      __syncthreads();
      const int n_in = (kFirstTile - 1) * stride + k;
      for (int e = tid; e < n_in; e += 256) {
        const int hh = q0 * stride - pad + e;
        if (hh < 0 || hh >= h_in) continue;
        float a = 0.f;
        for (int j = 0; j < k; ++j) {
          const int num = hh + pad - j;
          if (num < 0 || num % stride) continue;
          const int ho = num / stride;
          if (ho < q0 || ho >= p1 || ho >= q0 + kFirstTile) continue;
          a += gsm[(ho - q0) * kFirstK + j] + gsm[(kFirstTile + ho - q0) * kFirstK + j];
        }
        int ii = hh * period + wcol;
        if (ii >= t) ii = 2 * (t - 1) - ii;
        atomicAdd(dy + static_cast<size_t>(b) * t + ii, a);
      }
    }
  }
  if (dw) {
    // the row groups of the block meet in shared memory (the staging buffers are free now): one atomic per
    // (channel, tap | bias) per block instead of one per row group — the atomics were the cost of this kernel
    __syncthreads();
    float* red = reinterpret_cast<float*>(smb);                 // [rgroups][cout][kFirstK]
    if (rh < rgroups) {
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) red[(rh * cout + cg * 4 + a) * kFirstK + jg * 4 + c] = acc[a][c];
    }
    __syncthreads();
    for (int i = tid; i < cout * kFirstK; i += 256) {
      const int co = i / kFirstK, j = i % kFirstK;
      if (j > k) continue;
      float v = 0.f;
      for (int g = 0; g < rgroups; ++g) v += red[g * cout * kFirstK + i];
      if (j < k) atomicAdd(dw + co * k + j, v);
      else atomicAdd(db + co, v);
    }
  }
}

// AvgPool1d(4,2,2) backward: din[b][i] += 0.25 * sum_{o: 2o-2+j = i} dout[b][o]
__global__ void avgpool_bwd_kernel(const float* __restrict__ dout, int t, int t_out, float* __restrict__ din) {
  const int b = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= t) return;
  float a = 0.f;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int e = i + 2 - j;
    if (e >= 0 && (e & 1) == 0 && (e >> 1) < t_out) a += dout[static_cast<size_t>(b) * t_out + (e >> 1)];
  }
  din[static_cast<size_t>(b) * t + i] += 0.25f * a;
}

// mode 0: out = coef * sgn(a - b); mode 1: out = coef * (a - c); mode 2: out = coef * (a - c) + coef2 * sgn(a - b)
// scale_dev (optional): a device scalar both coefficients are multiplied with (the incoming gradient of a mean)
__global__ void loss_grad_kernel(const float* __restrict__ a, const float* __restrict__ b, long long n, int mode,
                                 float c, float coef, float coef2, const float* __restrict__ scale_dev,
                                 float* __restrict__ out) {
  if (scale_dev) { const float sc = *scale_dev; coef *= sc; coef2 *= sc; }
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += 256LL * gridDim.x) {
    const float av = a[i];
    float g;
    if (mode == 0) g = coef * sgn(av - b[i]);
    else if (mode == 1) g = coef * (av - c);
    else g = coef * (av - c) + coef2 * sgn(av - b[i]);
    out[i] = g;
  }
}

// torch.optim.AdamW step on one flat fp32 tensor.  kGuard: the clip_grad_norm_ / non-finite-skip flavour — nothing
// is written when *skip is set, otherwise the gradient scale is multiplied by *clip_coef (hg_grad_norm_finalize).
// The guard arguments come last so the unguarded instantiation keeps its parameter offsets.
template <bool kGuard>
__global__ void adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                             float* __restrict__ v, long long n, float lr, float b1, float b2, float eps, float wd,
                             float bc1, float bc2_sqrt, float gscale, const int* __restrict__ dev_step,
                             const float* __restrict__ dev_lr, const float* __restrict__ clip_coef,
                             const int* __restrict__ skip) {
  if constexpr (kGuard) {
    if (*skip) return;
    gscale = gscale * *clip_coef;
  }
  if (dev_step) {   // step counter kept on the device so a captured CUDA graph advances it
    const float st = static_cast<float>(*dev_step);
    bc1 = 1.f - powf(b1, st);
    bc2_sqrt = sqrtf(1.f - powf(b2, st));
  }
  if (dev_lr) lr = *dev_lr;   // learning-rate schedule without re-capturing the graph
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += 256LL * gridDim.x) {
    const float gi = g[i] * gscale;
    float pi = p[i] * (1.f - lr * wd);
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    pi -= (lr / bc1) * mi / (sqrtf(vi) / bc2_sqrt + eps);
    p[i] = pi;
  }
}

// dgrad (polyphase) pack: fp32 [cout][cin_g][k] -> bf16 [m][rho * cin + ci][cc], cc = dy channel inside the
// (merged) group tile of ci;  j = rho + pad - stride * (m + shift_min)
// One thread per output element; used when a layer's shape does not tile (HG_JOB_DISC_DGRAD_TILE covers the others).
struct DiscPackArgs {
  int cin_g, k, merge, cout_g, cin, stride, pad, nshift, shift_min, cout_tile;
};
__global__ void pack_disc_dgrad_kernel(const float* __restrict__ w, const DiscPackArgs a, __nv_bfloat16* __restrict__ out) {
  const long long n = static_cast<long long>(a.nshift) * a.stride * a.cin * a.cout_tile;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += 256LL * gridDim.x) {
    const int cc = static_cast<int>(i % a.cout_tile);
    long long r = i / a.cout_tile;
    const int ci = static_cast<int>(r % a.cin); r /= a.cin;
    const int rho = static_cast<int>(r % a.stride);
    const int m = static_cast<int>(r / a.stride);
    const int g = ci / a.cin_g;
    const int co = (g / a.merge) * a.cout_tile + cc;
    const int j = rho + a.pad - a.stride * (m + a.shift_min);
    float v = 0.f;
    if (co / a.cout_g == g && j >= 0 && j < a.k) v = w[(static_cast<size_t>(co) * a.cin_g + (ci - g * a.cin_g)) * a.k + j];
    out[i] = __float2bfloat16(v);
  }
}
// ---- spectral norm (torch.nn.utils.spectral_norm, dim 0, one power iteration, eps 1e-12; src/models.py:194) ----
// K1: t[j] += sum_{i in row chunk} W[i][j] * u[i]            (W^T u, rows split over blockIdx.y, t zeroed before)
__global__ void __launch_bounds__(256)
sn_wtu_kernel(const float* __restrict__ w, const float* __restrict__ u, int rows, int cols, int rows_per_block,
              float* __restrict__ t) {
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= cols) return;
  const int r0 = blockIdx.y * rows_per_block, r1 = min(rows, r0 + rows_per_block);
  float a = 0.f;
  for (int i = r0; i < r1; ++i) a += w[static_cast<size_t>(i) * cols + j] * u[i];
  atomicAdd(t + j, a);
}
// K2: v = normalize(t) (or the stored v when !iterate);  s[i] = sum_j W[i][j] * v[j]   (one warp per row)
__global__ void __launch_bounds__(256)
sn_wv_kernel(const float* __restrict__ w, const float* __restrict__ t, float* __restrict__ v, float* __restrict__ v_copy,
             int rows, int cols, int iterate, float eps, float* __restrict__ s) {
  __shared__ float red[32];
  float inv = 1.f;
  if (iterate) {
    float ss = 0.f;
    for (int j = threadIdx.x; j < cols; j += 256) ss += t[j] * t[j];
    ss = hg::block_sum(ss, red);
    inv = 1.f / fmaxf(sqrtf(ss), eps);
  }
  const float* src = iterate ? t : v;
  if (blockIdx.x == 0) {
    for (int j = threadIdx.x; j < cols; j += 256) {
      const float val = src[j] * inv;
      if (v_copy) v_copy[j] = val;
      if (iterate) v[j] = val;     // in-place buffer update, as torch does in train mode
    }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = blockIdx.x * 8 + warp; i < rows; i += gridDim.x * 8) {
    const float* wr = w + static_cast<size_t>(i) * cols;
    float a = 0.f;
    for (int j = lane; j < cols; j += 32) a += wr[j] * src[j];
    a = warp_sum(a) * inv;
    if (lane == 0) s[i] = a;
  }
}
// K3: u = normalize(s) (or the stored u), sigma = u . s, w_eff = W / sigma
__global__ void __launch_bounds__(256)
sn_scale_kernel(const float* __restrict__ w, const float* __restrict__ s, float* __restrict__ u,
                float* __restrict__ u_copy, int rows, long long n, int iterate, float eps, float* __restrict__ w_eff,
                float* __restrict__ sigma_out) {
  __shared__ float red[32];
  float sigma;
  if (iterate) {
    float ss = 0.f;
    for (int i = threadIdx.x; i < rows; i += 256) ss += s[i] * s[i];
    ss = hg::block_sum(ss, red);
    const float inv = 1.f / fmaxf(sqrtf(ss), eps);
    sigma = ss * inv;
    if (blockIdx.x == 0)
      for (int i = threadIdx.x; i < rows; i += 256) {
        const float val = s[i] * inv;
        u[i] = val;
        if (u_copy) u_copy[i] = val;
      }
  } else {
    float d = 0.f;
    for (int i = threadIdx.x; i < rows; i += 256) d += u[i] * s[i];
    sigma = hg::block_sum(d, red);
    if (blockIdx.x == 0 && u_copy)
      for (int i = threadIdx.x; i < rows; i += 256) u_copy[i] = u[i];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && sigma_out) *sigma_out = sigma;
  const float inv_sigma = 1.f / sigma;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += 256LL * gridDim.x) w_eff[i] = w[i] * inv_sigma;
}
// backward: dot = <dw_eff, w_eff>;  dW[i][j] (+)= (dw_eff[i][j] - dot * u[i] * v[j]) / sigma
__global__ void __launch_bounds__(256)
sn_bwd_dot_kernel(const float* __restrict__ d, const float* __restrict__ w_eff, long long n, float* __restrict__ dot) {
  __shared__ float red[32];
  float a = 0.f;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += 256LL * gridDim.x) a += d[i] * w_eff[i];
  a = hg::block_sum(a, red);
  if (threadIdx.x == 0) atomicAdd(dot, a);
}
__global__ void __launch_bounds__(256)
sn_bwd_apply_kernel(const float* __restrict__ d, const float* __restrict__ u, const float* __restrict__ v,
                    const float* __restrict__ sigma, const float* __restrict__ dot, int cols, long long n,
                    int accumulate, float* __restrict__ out) {
  const float inv = 1.f / *sigma, dt = *dot;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += 256LL * gridDim.x) {
    const int r = static_cast<int>(i / cols), c = static_cast<int>(i - static_cast<long long>(r) * cols);
    const float val = (d[i] - dt * u[r] * v[c]) * inv;
    out[i] = accumulate ? out[i] + val : val;
  }
}

// ---- gradient norm (torch.nn.utils.clip_grad_norm_) -------------------------------------------------------------
// Deterministic: the grid and every thread's share depend on n alone, the sums run in a fixed order, and no
// floating-point atomics are used, so the same gradient bits give the same norm bits on any stream or lane order.
constexpr int kNormSlot = 1024;         // per-block partials of one hg_grad_sumsq call = max blocks
constexpr int kNormPerBlock = 4096;     // at least 16 elements (4 groups) per thread before another block is added

__device__ __forceinline__ double warp_sum_d(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// 256 threads: the fixed-order block sum of one double per thread (valid in thread 0)
__device__ __forceinline__ double block_sum_d(double v, double* red) {
  v = warp_sum_d(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int i = 0; i < 8; ++i) s += red[i];
  return s;
}

inline int norm_blocks(long long n) {
  const long long b = (n + kNormPerBlock - 1) / kNormPerBlock;
  return static_cast<int>(b < 1 ? 1 : (b > kNormSlot ? kNormSlot : b));
}

// partial[b] = sum of x^2 over the 4-element groups j = b*256 + tid (+ k * grid * 256) of block b, the squares of
// one group summed in fp32, the groups of a thread in fp64.  16-byte loads when x is 16-byte aligned; otherwise the
// same groups are read element by element, so the result does not depend on the alignment.  Blocks past the grid
// write zeros into the rest of the slot (the finalize sums the whole slot).
__global__ void __launch_bounds__(256)
grad_sumsq_kernel(const float* __restrict__ x, long long n, double* __restrict__ partial) {
  __shared__ double red[8];
  const long long groups = (n + 3) >> 2, full = n >> 2;
  const long long stride = 256LL * gridDim.x;
  const bool vec = (reinterpret_cast<uintptr_t>(x) & 15) == 0;
  double acc = 0.0;
  for (long long j = blockIdx.x * 256LL + threadIdx.x; j < groups; j += stride) {
    float4 q;
    if (vec && j < full) {
      q = __ldg(reinterpret_cast<const float4*>(x) + j);
    } else {
      const long long e = 4 * j;
      q.x = x[e];
      q.y = e + 1 < n ? x[e + 1] : 0.f;
      q.z = e + 2 < n ? x[e + 2] : 0.f;
      q.w = e + 3 < n ? x[e + 3] : 0.f;
    }
    acc += static_cast<double>(fmaf(q.w, q.w, fmaf(q.z, q.z, fmaf(q.y, q.y, q.x * q.x))));
  }
  const double s = block_sum_d(acc, red);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
  if (blockIdx.x == 0)
    for (int i = gridDim.x + threadIdx.x; i < kNormSlot; i += 256) partial[i] = 0.0;
}

// One block: norm = sqrt(sum of every partial of `nslots` slots) * grad_scale, then torch's coefficient and the
// skip decision; the step counter advances only for a step that will be applied.
__global__ void __launch_bounds__(256)
grad_norm_finalize_kernel(const double* __restrict__ partial, int nslots, float max_norm, float grad_scale,
                          float* __restrict__ norm_out, float* __restrict__ coef_out, int* __restrict__ skip_out,
                          int* __restrict__ dev_step, int* __restrict__ skipped) {
  __shared__ double red[8];
  double acc = 0.0;
  const int total = nslots * kNormSlot;
  for (int i = threadIdx.x; i < total; i += 256) acc += partial[i];
  const double s = block_sum_d(acc, red);
  if (threadIdx.x != 0) return;
  const float norm = static_cast<float>(sqrt(s) * static_cast<double>(grad_scale));
  const bool finite = isfinite(norm);
  *norm_out = norm;
  *coef_out = fminf(max_norm / (norm + 1e-6f), 1.f);    // clip_grad_norm_: clamp(max_norm / (total + 1e-6), max=1)
  *skip_out = finite ? 0 : 1;
  if (finite) {
    if (dev_step) *dev_step += 1;
  } else if (skipped) {
    *skipped += 1;
  }
}

// HG_JOB_FINISH_ROW mode 0 for a conv's packed gradient [k][rows_p][cin_tile]; tab[packed position] = original tap
hg_prep_job finish_conv_job(const float* dw_packed, int cout, int cin_g, int k, int rows_p, int cin_tile, int cout_g,
                            int merge, const int* host_tap_order, const float* v, const float* g, int accumulate,
                            float* dv, float* dg) {
  hg_prep_job j{};
  j.kind = HG_JOB_FINISH_ROW;
  j.src0 = dw_packed; j.src1 = g; j.src2 = v; j.dst0 = dv; j.dst1 = dg;
  const int ints[] = {0, cout, cin_g, k, rows_p, cin_tile, cout_g, merge};
  for (int q = 0; q < 8; ++q) j.i[q] = ints[q];
  j.i[12] = accumulate;
  for (int q = 0; q < k; ++q) j.tab[host_tap_order ? host_tap_order[q] : q] = q;
  return j;
}

int blocks_for(long long n, int per = 256) {
  long long b = (n + per - 1) / per;
  if (b > 148 * 16) b = 148 * 16;
  return b < 1 ? 1 : static_cast<int>(b);
}

}  // namespace

extern "C" int hg_pack_dgrad_weight(const void* w_packed, int ktaps, int n, int c, void* out, void* stream) {
  HG_REQUIRE(w_packed && out && ktaps > 0 && n > 0 && c > 0 && ktaps <= 65535, "hg_pack_dgrad_weight: bad arguments");
  hg_prep_job j{};
  j.kind = HG_JOB_TRANSPOSE_TILE;
  j.src0 = w_packed; j.dst0 = out;
  const int tiles_c = (c + 31) / 32, tiles_n = (n + 31) / 32;
  const int ints[] = {ktaps, n, c, tiles_c, tiles_n};
  for (int q = 0; q < 5; ++q) j.i[q] = ints[q];
  return hg_prep_launch_one(j, ktaps * tiles_c * tiles_n, 32 * 34 * 2, stream);
}

extern "C" int hg_colsum_bf16(const void* x, int batch, int t_valid, int t_rows, int c, int accumulate, float* out,
                              void* stream) {
  HG_REQUIRE(x && out && batch > 0 && batch <= 65535 && t_valid > 0 && t_rows >= t_valid, "hg_colsum_bf16: bad sizes");
  HG_REQUIRE(c % 8 == 0 && c / 8 <= 256, "hg_colsum_bf16: c must be a multiple of 8, at most 2048");
  if (!accumulate) HG_CHECK_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * c, S(stream)));
  // enough blocks to fill the machine, few enough that the per-channel atomics stay cheap
  int rows_per_block = static_cast<int>((static_cast<long long>(batch) * t_valid + 591) / 592);
  if (rows_per_block < 64) rows_per_block = 64;
  dim3 grid((t_valid + rows_per_block - 1) / rows_per_block, batch);
  const size_t smem = static_cast<size_t>(256 / (c / 8)) * c * sizeof(float);
  colsum_kernel<<<grid, 256, smem, S(stream)>>>(static_cast<const __nv_bfloat16*>(x), t_valid, t_rows, c, rows_per_block,
                                              out);
  HG_CHECK_CUDA(cudaGetLastError());
  count();
  return HG_OK;
}

extern "C" int hg_conv_post_tanh_bwd(const void* x, const float* w, const float* y, const float* dy, int batch, int t,
                                     int c, int k, float in_slope, float dx_scale, void* dx, float* dpre_ws, float* dw,
                                     float* db, float* bias_grad0, float* bias_grad1, float* bias_grad2, void* stream) {
  HG_REQUIRE(x && w && y && dy && dx && dpre_ws, "hg_conv_post_tanh_bwd: null pointer");
  HG_REQUIRE(batch > 0 && batch <= 65535 && t > 0 && c % 8 == 0 && (k & 1) && k <= 15, "hg_conv_post_tanh_bwd: bad shape");
  HG_REQUIRE(bias_grad0 || (!bias_grad1 && !bias_grad2), "hg_conv_post_tanh_bwd: fill bias_grad slots from 0");
  dim3 grid((t + 255) / 256, batch);
  const size_t smem = (static_cast<size_t>(c) * k + 256 + k + c) * sizeof(float);
  conv_post_bwd_dx_kernel<<<grid, 256, smem, S(stream)>>>(static_cast<const __nv_bfloat16*>(x), w, y, dy, t, c, k,
                                                          in_slope, dx_scale, static_cast<__nv_bfloat16*>(dx), dpre_ws,
                                                          bias_grad0, bias_grad1, bias_grad2);
  HG_CHECK_CUDA(cudaGetLastError());
  count();
  if (dw) {
    const int tile = 1024;
    dim3 g2((t + tile - 1) / tile, batch);
    conv_post_bwd_dw_kernel<<<g2, 256, tile * sizeof(float), S(stream)>>>(static_cast<const __nv_bfloat16*>(x),
                                                                          dpre_ws, t, c, k, tile, dw, db);
    HG_CHECK_CUDA(cudaGetLastError());
    count();
  }
  return HG_OK;
}

extern "C" int hg_disc_last_conv_bwd(const void* x, const float* w, const float* dlogit, int nseq, int h, int h_rows,
                                     int c, int k, float slope, const void* fm_r, float fm_coef, const void* pre_add,
                                     void* dx, float* dw, float* db, float* bias_grad_in, void* stream) {
  HG_REQUIRE(x && w && dlogit, "hg_disc_last_conv_bwd: null pointer");
  HG_REQUIRE(nseq > 0 && nseq <= 65535 && h > 0 && h_rows >= h && k <= 7 && (k & 1), "hg_disc_last_conv_bwd: bad shape");
  HG_REQUIRE(dx || !bias_grad_in, "hg_disc_last_conv_bwd: bias_grad_in needs dx");
  if (dx) {
    dim3 grid((h + kLastRows - 1) / kLastRows, nseq);
    disc_last_bwd_dx_kernel<<<grid, 256, 0, S(stream)>>>(static_cast<const __nv_bfloat16*>(x), w, dlogit, h, h_rows, c,
                                                         k, slope, static_cast<const __nv_bfloat16*>(fm_r), fm_coef,
                                                         static_cast<const __nv_bfloat16*>(pre_add),
                                                         static_cast<__nv_bfloat16*>(dx), bias_grad_in);
    HG_CHECK_CUDA(cudaGetLastError());
    count();
  }
  if (dw) {
    HG_REQUIRE(c % 2 == 0, "hg_disc_last_conv_bwd: channel count must be even");
    const int total = nseq * h;
    int chunks = (total + 31) / 32;          // ~16 positions per thread
    if (chunks > 256) chunks = 256;
    dim3 grid((c + 255) / 256, chunks < 1 ? 1 : chunks);
    disc_last_bwd_dw_kernel<<<grid, 256, 0, S(stream)>>>(static_cast<const __nv_bfloat16*>(x), dlogit, nseq, h, h_rows,
                                                         c, k, dw, db);
    HG_CHECK_CUDA(cudaGetLastError());
    count();
  }
  return HG_OK;
}

extern "C" int hg_disc_first_conv_bwd(const float* y, const float* w, const void* dpre, int batch, int t, int period,
                                      int k, int stride, int pad, int cout, int h_rows, float* dw, float* db,
                                      float* dy, void* stream) {
  HG_REQUIRE(y && w && dpre && (dw || dy), "hg_disc_first_conv_bwd: null pointer");
  HG_REQUIRE(!dw || db, "hg_disc_first_conv_bwd: dw needs db");
  HG_REQUIRE(batch > 0 && t > 1 && period >= 1 && k >= 1 && k <= kFirstK && stride >= 1 && cout > 0 && cout % 2 == 0,
             "hg_disc_first_conv_bwd: bad shape");
  HG_REQUIRE(cout % 4 == 0 && 256 % cout == 0 && cout >= 4, "hg_disc_first_conv_bwd: cout must divide 256 (got %d)", cout);
  const int t_pad = (t + period - 1) / period * period;
  const int h_in = t_pad / period;
  const int h_out = (h_in + 2 * pad - k) / stride + 1;
  HG_REQUIRE(h_out > 0 && h_rows >= h_out && batch * period <= 65535, "hg_disc_first_conv_bwd: bad geometry");
  dim3 grid((h_out + kFirstChunk - 1) / kFirstChunk, batch * period);
  const size_t smem = static_cast<size_t>(kFirstK) * cout * 4 + kFirstTile * kXPitch * 4 + kFirstTile * kFirstK * 4 +
                      2 * kFirstTile * kFirstK * 4 + static_cast<size_t>(kFirstTile) * (cout + 2) * 2;
  static hg::PerDeviceOnce once;
  if (once.need())
    HG_CHECK_CUDA(cudaFuncSetAttribute(disc_first_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
  HG_REQUIRE(smem <= 96 * 1024, "hg_disc_first_conv_bwd: tile does not fit shared memory");
  disc_first_bwd_kernel<<<grid, 256, smem, S(stream)>>>(y, w, static_cast<const __nv_bfloat16*>(dpre), t, period, h_in,
                                                        h_out, h_rows, k, stride, pad, cout, dw, db, dy);
  HG_CHECK_CUDA(cudaGetLastError());
  count();
  return HG_OK;
}

extern "C" int hg_avgpool_4_2_2_bwd(const float* dout, int batch, int t, float* din, void* stream) {
  HG_REQUIRE(dout && din && batch > 0 && batch <= 65535 && t > 0, "hg_avgpool_4_2_2_bwd: bad arguments");
  dim3 grid((t + 255) / 256, batch);
  avgpool_bwd_kernel<<<grid, 256, 0, S(stream)>>>(dout, t, t / 2 + 1, din);
  HG_CHECK_CUDA(cudaGetLastError());
  count();
  return HG_OK;
}

extern "C" int hg_loss_grad(const float* a, const float* b, long long n, int mode, float c, float coef, float coef2,
                            const float* scale_dev, float* out, void* stream) {
  HG_REQUIRE(a && out && n > 0 && mode >= 0 && mode <= 2 && (mode == 1 || b), "hg_loss_grad: bad arguments");
  loss_grad_kernel<<<blocks_for(n), 256, 0, S(stream)>>>(a, b, n, mode, c, coef, coef2, scale_dev, out);
  HG_CHECK_CUDA(cudaGetLastError());
  count();
  return HG_OK;
}

extern "C" int hg_unpack_wgrad_conv(const float* dw_packed, int cout, int cin_g, int k, int rows_p, int cin_tile,
                                    int cout_g, int merge, const int* host_tap_order, float* dw, void* stream) {
  HG_REQUIRE(dw_packed && dw && k > 0 && k <= 64 && cout > 0 && cin_g > 0 && merge >= 1 && cout_g >= 1,
             "hg_unpack_wgrad_conv: bad arguments");
  HG_REQUIRE(static_cast<size_t>(cin_g) * k * 4 <= kPrepMaxSmem, "hg_unpack_wgrad_conv: row of %d values does not fit",
             cin_g * k);
  const hg_prep_job j = finish_conv_job(dw_packed, cout, cin_g, k, rows_p, cin_tile, cout_g, merge, host_tap_order,
                                        nullptr, nullptr, 0, dw, nullptr);
  return hg_prep_launch_one(j, cout, cin_g * k * 4, stream);
}

extern "C" int hg_weight_norm_bwd(const float* dw, const float* v, const float* g, int dim0, int rest, int accumulate,
                                  float* dv, float* dg, void* stream) {
  HG_REQUIRE(dw && v && g && dv && dg && dim0 > 0 && rest > 0, "hg_weight_norm_bwd: bad arguments");
  hg_prep_job j{};
  j.kind = HG_JOB_FINISH_ROW;
  j.src0 = dw; j.src1 = g; j.src2 = v; j.dst0 = dv; j.dst1 = dg;
  j.i[0] = 2; j.i[1] = dim0; j.i[2] = rest; j.i[3] = 1; j.i[12] = accumulate;
  return hg_prep_launch_one(j, dim0, 0, stream);
}

extern "C" int hg_adamw_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                             float beta2, float eps, float weight_decay, int step, const int* dev_step,
                             const float* dev_lr, float grad_scale, void* stream) {
  HG_REQUIRE(p && g && m && v && n > 0 && (step >= 1 || dev_step), "hg_adamw_step: bad arguments");
  if (step < 1) step = 1;
  const float bc1 = 1.f - powf(beta1, static_cast<float>(step));
  const float bc2 = 1.f - powf(beta2, static_cast<float>(step));
  adamw_kernel<false><<<blocks_for(n, 1024), 256, 0, S(stream)>>>(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay,
                                                                  bc1, sqrtf(bc2), grad_scale, dev_step, dev_lr,
                                                                  nullptr, nullptr);
  HG_CHECK_CUDA(cudaGetLastError());
  count();
  return HG_OK;
}

extern "C" int hg_adamw_step_guarded(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                                     float beta2, float eps, float weight_decay, const int* dev_step,
                                     const float* dev_lr, float grad_scale, const float* clip_coef, const int* skip,
                                     void* stream) {
  HG_REQUIRE(p && g && m && v && n > 0 && dev_step && clip_coef && skip, "hg_adamw_step_guarded: bad arguments");
  adamw_kernel<true><<<blocks_for(n, 1024), 256, 0, S(stream)>>>(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay,
                                                                 1.f, 1.f, grad_scale, dev_step, dev_lr, clip_coef,
                                                                 skip);
  HG_CHECK_CUDA(cudaGetLastError());
  count();
  return HG_OK;
}

extern "C" int hg_grad_norm_slot_size(void) { return kNormSlot; }

extern "C" int hg_grad_sumsq(const float* x, long long n, double* partials, void* stream) {
  HG_REQUIRE(x && partials && n > 0 && (reinterpret_cast<uintptr_t>(x) & 3) == 0, "hg_grad_sumsq: bad arguments");
  grad_sumsq_kernel<<<norm_blocks(n), 256, 0, S(stream)>>>(x, n, partials);
  HG_CHECK_CUDA(cudaGetLastError());
  count();
  return HG_OK;
}

extern "C" int hg_grad_norm_finalize(const double* partials, int nslots, float max_norm, float grad_scale,
                                     float* norm, float* clip_coef, int* skip, int* dev_step, int* skipped,
                                     void* stream) {
  HG_REQUIRE(partials && nslots > 0 && nslots <= 64 && norm && clip_coef && skip && max_norm > 0.f,
             "hg_grad_norm_finalize: bad arguments");
  grad_norm_finalize_kernel<<<1, 256, 0, S(stream)>>>(partials, nslots, max_norm, grad_scale, norm, clip_coef, skip,
                                                      dev_step, skipped);
  HG_CHECK_CUDA(cudaGetLastError());
  count();
  return HG_OK;
}

extern "C" int hg_pack_disc_weight(const float* w_eff, int cout, int cin, int groups, int merge, int k, int stride,
                                   int pad, void* w_fwd, void* w_dgrad, void* stream) {
  HG_REQUIRE(w_eff && (w_fwd || w_dgrad), "hg_pack_disc_weight: null pointer");
  HG_REQUIRE(cout > 0 && cin > 0 && groups >= 1 && merge >= 1 && groups % merge == 0 && k >= 1 && k <= 64 && stride >= 1,
             "hg_pack_disc_weight: bad arguments");
  DiscPackArgs a{};
  a.cin = cin; a.merge = merge; a.k = k; a.stride = stride; a.pad = pad;
  a.cin_g = cin / groups; a.cout_g = cout / groups;
  a.cout_tile = a.cout_g * merge;
  const int cin_tile = a.cin_g * merge;
  hg_prep_job j{};
  int rc = hg_conv1d_tap_order(k, stride, pad, j.tab);
  if (rc) return rc;
  rc = hg_convtr1d_geometry(k, stride, pad, &a.nshift, &a.shift_min);
  if (rc) return rc;
  if (w_fwd) {
    const size_t smem = static_cast<size_t>(a.cin_g) * k * sizeof(float);
    HG_REQUIRE(smem <= 48 * 1024 && cin_tile % 2 == 0, "hg_pack_disc_weight: filter row does not fit (cin/groups * k = %d)",
               a.cin_g * k);
    j.kind = HG_JOB_DISC_ROW;
    j.src0 = w_eff; j.dst1 = w_fwd;                  // src1 (g) NULL: w_eff is the weight, scaled by 1
    const int ints[] = {cout, a.cin_g, k, merge, a.cout_g, cin_tile};
    for (int q = 0; q < 6; ++q) j.i[q] = ints[q];
    rc = hg_prep_launch_one(j, cout, static_cast<int>(smem), stream);
    if (rc) return rc;
  }
  if (w_dgrad) {
    int tci = k <= 10 ? 32 : 8;
    while (tci > 2 && (a.cin_g % tci || cin % tci)) tci >>= 1;
    const size_t smem = 32 * (static_cast<size_t>(tci) * k + 1) * sizeof(float);
    if (a.cin_g % tci == 0 && cin % tci == 0 && a.cout_tile % 32 == 0 && smem <= 48 * 1024) {
      hg_prep_job d{};
      d.kind = HG_JOB_DISC_DGRAD_TILE;
      d.src0 = w_eff; d.dst0 = w_dgrad;
      const int ints[] = {cout, a.cin_g, k, merge, a.cout_g, cin, stride, pad, a.nshift, a.shift_min, a.cout_tile,
                          tci, cin / tci};
      for (int q = 0; q < 13; ++q) d.i[q] = ints[q];
      return hg_prep_launch_one(d, (cin / tci) * (a.cout_tile / 32), static_cast<int>(smem), stream);
    }
    pack_disc_dgrad_kernel<<<blocks_for(static_cast<long long>(a.nshift) * stride * cin * a.cout_tile), 256, 0,
                             S(stream)>>>(w_eff, a, static_cast<__nv_bfloat16*>(w_dgrad));
    HG_CHECK_CUDA(cudaGetLastError());
    count();
  }
  return HG_OK;
}

extern "C" int hg_spectral_norm_fwd(const float* w, float* u, float* v, int rows, int cols, int iterate, float* w_eff,
                                    float* sigma_out, float* u_copy, float* v_copy, float* ws, void* stream) {
  HG_REQUIRE(w && u && v && w_eff && ws && rows > 0 && cols > 0, "hg_spectral_norm_fwd: bad arguments");
  float* t = ws;            // [cols]
  float* sv = ws + cols;    // [rows]
  const float eps = 1e-12f;
  if (iterate) {
    HG_CHECK_CUDA(cudaMemsetAsync(t, 0, sizeof(float) * cols, S(stream)));
    const int rpb = 64;
    dim3 g1((cols + 255) / 256, (rows + rpb - 1) / rpb);
    sn_wtu_kernel<<<g1, 256, 0, S(stream)>>>(w, u, rows, cols, rpb, t);
    HG_CHECK_CUDA(cudaGetLastError());
    count();
  }
  const int g2 = (rows + 7) / 8 < 592 ? (rows + 7) / 8 : 592;
  sn_wv_kernel<<<g2, 256, 0, S(stream)>>>(w, t, v, v_copy, rows, cols, iterate, eps, sv);
  HG_CHECK_CUDA(cudaGetLastError());
  count();
  const long long n = static_cast<long long>(rows) * cols;
  sn_scale_kernel<<<blocks_for(n, 1024), 256, 0, S(stream)>>>(w, sv, u, u_copy, rows, n, iterate, eps, w_eff, sigma_out);
  HG_CHECK_CUDA(cudaGetLastError());
  count();
  return HG_OK;
}

extern "C" int hg_spectral_norm_bwd(const float* dw_eff, const float* w_eff, const float* u, const float* v,
                                    const float* sigma, int rows, int cols, int accumulate, float* dw_orig, float* ws,
                                    void* stream) {
  HG_REQUIRE(dw_eff && w_eff && u && v && sigma && dw_orig && ws && rows > 0 && cols > 0,
             "hg_spectral_norm_bwd: bad arguments");
  const long long n = static_cast<long long>(rows) * cols;
  HG_CHECK_CUDA(cudaMemsetAsync(ws, 0, sizeof(float), S(stream)));
  sn_bwd_dot_kernel<<<blocks_for(n, 2048), 256, 0, S(stream)>>>(dw_eff, w_eff, n, ws);
  HG_CHECK_CUDA(cudaGetLastError());
  count();
  sn_bwd_apply_kernel<<<blocks_for(n, 1024), 256, 0, S(stream)>>>(dw_eff, u, v, sigma, ws, cols, n, accumulate, dw_orig);
  HG_CHECK_CUDA(cudaGetLastError());
  count();
  return HG_OK;
}

// hg_wgrad_finish_conv: the packed-gradient unpack + hg_weight_norm_bwd fused (one launch per layer).  v, g: the
// module's weight_v / weight_g (g == NULL: plain `weight`, dv receives the unpacked gradient).
extern "C" int hg_wgrad_finish_conv(const float* dw_packed, int cout, int cin_g, int k, int rows_p, int cin_tile,
                                    int cout_g, int merge, const int* host_tap_order, const float* v, const float* g,
                                    int accumulate, float* dv, float* dg, void* stream) {
  HG_REQUIRE(dw_packed && v && dv && (!g || dg) && k > 0 && k <= 64 && cout > 0 && cin_g > 0 && merge >= 1 && cout_g >= 1,
             "hg_wgrad_finish_conv: bad arguments");
  HG_REQUIRE(static_cast<size_t>(cin_g) * k * 4 <= 48 * 1024, "hg_wgrad_finish_conv: row of %d values does not fit", cin_g * k);
  const hg_prep_job j = finish_conv_job(dw_packed, cout, cin_g, k, rows_p, cin_tile, cout_g, merge, host_tap_order,
                                        v, g, accumulate, dv, dg);
  return hg_prep_launch_one(j, cout, cin_g * k * 4, stream);
}
