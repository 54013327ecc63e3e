// hg_prep.cu — bandwidth-bound helpers around the implicit-GEMM conv:
//   * weight_norm fold + GEMM-ready bf16 packing (Conv1d and polyphase ConvTranspose1d)
//   * [B][C][T] fp32 <-> [B][T][C] bf16 layout edges
//   * conv_post + tanh (src/models.py:113-114)
#include "hg_common.cuh"

#include <atomic>

#include "../../include/hifigan_b200.h"

extern std::atomic<int64_t> g_hg_launches;

namespace {

__device__ __forceinline__ float block_sum(float v, float* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
  if (l == 0) red[w] = v;
  __syncthreads();
  float s = 0.f;
  for (int i = 0; i < nw; ++i) s += red[i];
  __syncthreads();
  return s;
}

// one block per output channel: w[co] = g[co] * v[co] / ||v[co]||  ->  out[j][co][ci]
__global__ void pack_conv1d_weight_kernel(const float* __restrict__ v, const float* __restrict__ g,
                                          int cout, int cin, int k, int cin_pad,
                                          __nv_bfloat16* __restrict__ out) {
  __shared__ float red[32];
  const int co = blockIdx.x;
  const float* vc = v + static_cast<size_t>(co) * cin * k;
  float scale = 1.f;
  if (g) {
    float ss = 0.f;
    for (int i = threadIdx.x; i < cin * k; i += blockDim.x) ss += vc[i] * vc[i];
    ss = block_sum(ss, red);
    scale = ss > 0.f ? g[co] / sqrtf(ss) : 0.f;  // all-zero rows only exist as channel padding
  }
  for (int j = 0; j < k; ++j) {
    __nv_bfloat16* o = out + (static_cast<size_t>(j) * cout + co) * cin_pad;
    for (int ci = threadIdx.x; ci < cin_pad; ci += blockDim.x)
      o[ci] = __float2bfloat16(ci < cin ? vc[ci * k + j] * scale : 0.f);
  }
}

// one block per input channel (weight_norm dim 0 of ConvTranspose1d): polyphase scatter
__global__ void pack_convtr1d_weight_kernel(const float* __restrict__ v, const float* __restrict__ g,
                                            int cin, int cout, int k, int stride, int padding,
                                            int nshift, int shift_min,
                                            __nv_bfloat16* __restrict__ out) {
  __shared__ float red[32];
  const int ci = blockIdx.x;
  const float* vc = v + static_cast<size_t>(ci) * cout * k;
  float scale = 1.f;
  if (g) {
    float ss = 0.f;
    for (int i = threadIdx.x; i < cout * k; i += blockDim.x) ss += vc[i] * vc[i];
    ss = block_sum(ss, red);
    scale = ss > 0.f ? g[ci] / sqrtf(ss) : 0.f;
  }
  const int n_total = stride * cout;
  for (int idx = threadIdx.x; idx < nshift * n_total; idx += blockDim.x) {
    const int s = idx / n_total;
    const int n = idx % n_total;
    const int p = n / cout, co = n % cout;
    const int j = p + padding - (shift_min + s) * stride;
    const float w = (j >= 0 && j < k) ? vc[co * k + j] * scale : 0.f;
    out[(static_cast<size_t>(s) * n_total + n) * cin + ci] = __float2bfloat16(w);
  }
}

// fp32 [B][C][T] -> bf16 [B][T][c_pad]; 32x32 smem transpose tiles
__global__ void ncl_to_nlc_kernel(const float* __restrict__ x, int c, int t, int c_pad,
                                  __nv_bfloat16* __restrict__ out, __nv_bfloat16* __restrict__ out_act,
                                  float slope) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int cc = c0 + i, tt = t0 + tx;
    tile[i][tx] = (cc < c && tt < t) ? x[(static_cast<size_t>(b) * c + cc) * t + tt] : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int tt = t0 + i, cc = c0 + tx;
    if (tt < t && cc < c_pad) {
      const size_t o = (static_cast<size_t>(b) * t + tt) * c_pad + cc;
      const float v = tile[tx][i];
      if (out) out[o] = __float2bfloat16(v);
      if (out_act) out_act[o] = __float2bfloat16(hg::lrelu(v, slope));
    }
  }
}

// bf16 [B][T][C] -> fp32 [B][C][T]
__global__ void nlc_to_ncl_kernel(const __nv_bfloat16* __restrict__ x, int t, int c,
                                  float* __restrict__ out) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int c0 = blockIdx.x * 32, t0 = blockIdx.y * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;
  for (int i = ty; i < 32; i += 8) {
    const int tt = t0 + i, cc = c0 + tx;
    tile[i][tx] = (tt < t && cc < c) ? __bfloat162float(x[(static_cast<size_t>(b) * t + tt) * c + cc]) : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int cc = c0 + i, tt = t0 + tx;
    if (cc < c && tt < t) out[(static_cast<size_t>(b) * c + cc) * t + tt] = tile[tx][i];
  }
}

// conv_post + tanh: y[b,t] = tanh(bias + sum_{j,c} x[b, t + j - k/2, c] * w[c][j]).
// Each thread produces kPostPer consecutive samples so that one shared-memory read of a weight vector feeds
// kPostPer FMAs (one-output-per-thread was bound by the LDS issue rate, 0.76 ms at config 2).  The
// (tile + k - 1) x C input window is staged in shared memory with a 16-byte row pad so the 128-bit row reads of
// a quarter-warp hit distinct banks.
constexpr int kPostThreads = 128;
constexpr int kPostPer = 4;
constexpr int kPostTile = kPostThreads * kPostPer;

__global__ void __launch_bounds__(kPostThreads)
conv_post_tanh_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w,
                      const float* __restrict__ bias, int t, int c, int k, float* __restrict__ y) {
  extern __shared__ __align__(16) uint8_t sm[];
  const int pitch = c * 2 + 16;                 // bytes per staged row
  const int rows = kPostTile + k - 1;
  float* ws = reinterpret_cast<float*>(sm);     // [k][c]
  uint8_t* xs = sm + ((k * c * 4 + 15) & ~15);  // [rows][pitch]
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * kPostTile;
  const int half = k / 2;
  for (int i = threadIdx.x; i < k * c; i += blockDim.x) {
    const int j = i / c, cc = i % c;
    ws[i] = w[cc * k + j];
  }
  const int vec_per_row = c / 8;  // uint4 = 8 bf16
  const __nv_bfloat16* xb = x + static_cast<size_t>(b) * t * c;
  for (int i = threadIdx.x; i < rows * vec_per_row; i += blockDim.x) {
    const int r = i / vec_per_row, vq = i % vec_per_row;
    const int tt = t0 + r - half;
    uint4 val = make_uint4(0, 0, 0, 0);
    if (tt >= 0 && tt < t) val = *reinterpret_cast<const uint4*>(xb + static_cast<size_t>(tt) * c + vq * 8);
    *reinterpret_cast<uint4*>(xs + r * pitch + vq * 16) = val;
  }
  __syncthreads();
  // thread owns outputs tid, tid + 128, tid + 256, tid + 384 of the tile: lanes of a warp read adjacent staged
  // rows (conflict-free with the 16-byte pad) and every weight vector read from shared memory feeds 4 outputs
  float acc[kPostPer];
#pragma unroll
  for (int o = 0; o < kPostPer; ++o) acc[o] = bias ? bias[0] : 0.f;
  for (int j = 0; j < k; ++j) {
    for (int vq = 0; vq < vec_per_row; ++vq) {
      const float4 w0 = *reinterpret_cast<const float4*>(ws + j * c + vq * 8);
      const float4 w1 = *reinterpret_cast<const float4*>(ws + j * c + vq * 8 + 4);
#pragma unroll
      for (int o = 0; o < kPostPer; ++o) {
        const uint4 rv = *reinterpret_cast<const uint4*>(xs + (threadIdx.x + o * kPostThreads + j) * pitch + vq * 16);
        const float2 a0 = hg::unpack_bf16x2(rv.x), a1 = hg::unpack_bf16x2(rv.y), a2 = hg::unpack_bf16x2(rv.z),
                     a3 = hg::unpack_bf16x2(rv.w);
        acc[o] += a0.x * w0.x + a0.y * w0.y + a1.x * w0.z + a1.y * w0.w + a2.x * w1.x + a2.y * w1.y +
                  a3.x * w1.z + a3.y * w1.w;
      }
    }
  }
#pragma unroll
  for (int o = 0; o < kPostPer; ++o) {
    const int tt = t0 + threadIdx.x + o * kPostThreads;
    if (tt < t) y[static_cast<size_t>(b) * t + tt] = tanhf(acc[o]);
  }
}

// conv_post + tanh, register-window version for the shapes the configs use (C = 32 channels, k = 7).  The kernel
// above re-reads every staged input row from shared memory once per tap and converts it again (ncu, round 2: 29
// warp-instructions per output sample, 0.78 ms per 16.8 M samples, 18 % of the HBM rate).  Here a thread owns
// kPost2R CONSECUTIVE outputs and walks the channels in slabs of 4: the kPost2R + K - 1 rows of a slab are read and
// converted once into registers and feed all K taps of all kPost2R outputs (224 FMAs per output, ~50 other
// instructions instead of ~700).  kPost2R is odd and the staged row pitch is C*2 + 8 bytes, so the 8-byte row reads of
// a half-warp (thread stride 9 x 72 B = 81 x 8 B) fall on distinct bank pairs.  Outputs leave through shared memory
// so the global stores stay coalesced.  Measured: 0.781 -> 0.486 ms per 64 x 262 144 samples.
constexpr int kPost2R = 9;
template <int C, int K, int kPost2Threads>
__global__ void __launch_bounds__(kPost2Threads)
conv_post_tanh_kernel2(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w,
                       const float* __restrict__ bias, int t, float* __restrict__ y) {
  extern __shared__ __align__(16) uint8_t sm[];
  constexpr int kPost2Tile = kPost2R * kPost2Threads;
  constexpr int kPitch = C * 2 + 8;
  constexpr int kRows = kPost2Tile + K - 1;
  constexpr int kWin = kPost2R + K - 1;
  float* ws = reinterpret_cast<float*>(sm);              // [K][C]
  uint8_t* xs = sm + ((K * C * 4 + 15) & ~15);           // [kRows][kPitch]
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * kPost2Tile;
  for (int i = threadIdx.x; i < K * C; i += kPost2Threads) ws[i] = w[(i % C) * K + i / C];
  constexpr int kVec = C / 8;                             // 16-byte global loads per row
  const __nv_bfloat16* xb = x + static_cast<size_t>(b) * t * C;
  for (int i = threadIdx.x; i < kRows * kVec; i += kPost2Threads) {
    const int r = i / kVec, vq = i % kVec;
    const int tt = t0 + r - K / 2;
    uint4 val = make_uint4(0, 0, 0, 0);
    if (tt >= 0 && tt < t) val = *reinterpret_cast<const uint4*>(xb + static_cast<size_t>(tt) * C + vq * 8);
    uint2* dst = reinterpret_cast<uint2*>(xs + r * kPitch + vq * 16);     // rows are 8-byte aligned only
    dst[0] = make_uint2(val.x, val.y);
    dst[1] = make_uint2(val.z, val.w);
  }
  __syncthreads();
  float acc[kPost2R];
  const float b0 = bias ? bias[0] : 0.f;
#pragma unroll
  for (int o = 0; o < kPost2R; ++o) acc[o] = b0;
  const uint8_t* base = xs + static_cast<size_t>(threadIdx.x) * kPost2R * kPitch;
#pragma unroll 1
  for (int q = 0; q < C / 4; ++q) {
    float xr[kWin][4];
#pragma unroll
    for (int r = 0; r < kWin; ++r) {
      const uint2 v = *reinterpret_cast<const uint2*>(base + r * kPitch + q * 8);
      const float2 lo = hg::unpack_bf16x2(v.x), hi = hg::unpack_bf16x2(v.y);
      xr[r][0] = lo.x; xr[r][1] = lo.y; xr[r][2] = hi.x; xr[r][3] = hi.y;
    }
#pragma unroll
    for (int j = 0; j < K; ++j) {
      const float4 wv = *reinterpret_cast<const float4*>(ws + j * C + q * 4);
#pragma unroll
      for (int o = 0; o < kPost2R; ++o)
        acc[o] += xr[o + j][0] * wv.x + xr[o + j][1] * wv.y + xr[o + j][2] * wv.z + xr[o + j][3] * wv.w;
    }
  }
  __syncthreads();                                        // everyone is done reading the staged rows
  float* ys = reinterpret_cast<float*>(xs);
#pragma unroll
  for (int o = 0; o < kPost2R; ++o) ys[threadIdx.x * kPost2R + o] = tanhf(acc[o]);
  __syncthreads();
  for (int i = threadIdx.x; i < kPost2Tile; i += kPost2Threads)
    if (t0 + i < t) y[static_cast<size_t>(b) * t + t0 + i] = ys[i];
}

// out[b][i] = i < valid[b] ? pool[start[b] + i] : 0   (MelDataset crop / right zero-pad, meldataset.py:141-150)
__global__ void segment_gather_kernel(const float* __restrict__ pool, const long long* __restrict__ start,
                                      const int* __restrict__ valid, int seg, float* __restrict__ out) {
  const int b = blockIdx.y;
  const long long s0 = start[b];
  const int nv = valid[b];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < seg; i += gridDim.x * blockDim.x)
    out[static_cast<size_t>(b) * seg + i] = i < nv ? pool[s0 + i] : 0.f;
}

// One int16 sample -> the fp32 value the host pipeline gives it: q / 32768 (read_wav) / 32768 (MAX_WAV_VALUE, both
// divisions exact), then the utterance's normalisation.  peak: (q / m) * 0.95f with m = max|q| over the utterance;
// the two 2^-15 scales cancel exactly in the IEEE quotient.
__device__ __forceinline__ float stage_sample(int q, int m, int mode) {
  if (mode == HG_STAGE_PEAK) return m > 0 ? __fmul_rn(__fdiv_rn(static_cast<float>(q), static_cast<float>(m)), 0.95f) : 0.f;
  if (mode == HG_STAGE_FORK) return q > 0 ? 0.95f : (q < 0 ? -0.95f : 0.f);
  return __fmul_rn(static_cast<float>(q), 0x1p-30f);
}

// out[b][i] = i < valid[b] ? stage_sample(staged[b][i], peak[b]) : 0; kVec: 8 samples per thread in 16-byte accesses
template <bool kVec>
__global__ void __launch_bounds__(256)
segment_stage_i16_kernel(const int16_t* __restrict__ staged, const int* __restrict__ peak,
                         const int* __restrict__ valid, int seg, int mode, float* __restrict__ out) {
  const int b = blockIdx.y;
  const int i0 = (blockIdx.x * 256 + threadIdx.x) * 8;
  if (i0 >= seg) return;
  const int nv = valid[b], m = peak[b];
  const int16_t* src = staged + static_cast<size_t>(b) * seg + i0;
  float* dst = out + static_cast<size_t>(b) * seg + i0;
  if (kVec) {
    const int4 raw = *reinterpret_cast<const int4*>(src);
    const int w[4] = {raw.x, raw.y, raw.z, raw.w};
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int q = static_cast<int16_t>(static_cast<uint32_t>(w[j >> 1]) >> ((j & 1) * 16));
      v[j] = i0 + j < nv ? stage_sample(q, m, mode) : 0.f;
    }
    reinterpret_cast<float4*>(dst)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4*>(dst)[1] = make_float4(v[4], v[5], v[6], v[7]);
  } else {
    for (int j = 0; j < 8 && i0 + j < seg; ++j) dst[j] = i0 + j < nv ? stage_sample(src[j], m, mode) : 0.f;
  }
}

// staged fp32 [B][fps][num_mels] -> out [B][num_mels][fps], frames >= valid_frames[b] zero; 32x32 smem transpose tiles
__global__ void segment_stage_mel_kernel(const float* __restrict__ staged, const int* __restrict__ valid_frames,
                                         int fps, int num_mels, float* __restrict__ out) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int f0 = blockIdx.x * 32, m0 = blockIdx.y * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
  const int nv = valid_frames[b];
  const float* src = staged + static_cast<size_t>(b) * fps * num_mels;
  for (int i = ty; i < 32; i += 8) {
    const int f = f0 + i, m = m0 + tx;
    tile[i][tx] = (f < nv && f < fps && m < num_mels) ? src[static_cast<size_t>(f) * num_mels + m] : 0.f;
  }
  __syncthreads();
  float* dst = out + static_cast<size_t>(b) * num_mels * fps;
  for (int i = ty; i < 32; i += 8) {
    const int m = m0 + i, f = f0 + tx;
    if (m < num_mels && f < fps) dst[static_cast<size_t>(m) * fps + f] = tile[tx][i];
  }
}

// mode 0: sum |a - b|     (feature_loss / mel L1, src/models.py:251-257)
// mode 1: sum (c - a)^2   (LSGAN terms, src/models.py:260-282; c = 1 for "real", 0 for "generated")
__global__ void __launch_bounds__(256)
loss_sum_kernel(const float* __restrict__ a, const float* __restrict__ b, long long n, int mode, float c,
                float* __restrict__ out) {
  __shared__ float red[32];
  float acc = 0.f;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += 256LL * gridDim.x) {
    const float d = mode == 0 ? a[i] - b[i] : c - a[i];
    acc += mode == 0 ? fabsf(d) : d * d;
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) atomicAdd(out, acc);
}

// out[i] = (int16) trunc(x[i] * scale): the `audio * MAX_WAV_VALUE -> astype('int16')` of the reference's drivers
// (src/inference.py:57-58, src/inference_e2e.py:51-52) on the device, so the D2H copy moves 2 bytes per sample
__global__ void float_to_int16_kernel(const float* __restrict__ x, long long n, float scale, int16_t* __restrict__ out) {
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += 256LL * gridDim.x)
    out[i] = static_cast<int16_t>(static_cast<int>(x[i] * scale));
}

}  // namespace

extern "C" int hg_float_to_int16(const float* x, long long n, float scale, int16_t* out, void* stream) {
  HG_REQUIRE(x && out && n > 0, "hg_float_to_int16: bad arguments");
  long long blocks = (n + 256 * 4 - 1) / (256 * 4);
  if (blocks > 148 * 16) blocks = 148 * 16;
  float_to_int16_kernel<<<static_cast<int>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, n, scale, out);
  HG_CHECK_CUDA(cudaGetLastError());
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

extern "C" int hg_loss_sum(const float* a, const float* b, long long n, int mode, float c, float* out_acc,
                           void* stream) {
  HG_REQUIRE(a && out_acc && n > 0 && (mode == 0 ? b != nullptr : mode == 1), "hg_loss_sum: bad arguments");
  long long blocks = (n + 256 * 8 - 1) / (256 * 8);
  if (blocks > 148 * 8) blocks = 148 * 8;
  loss_sum_kernel<<<static_cast<int>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(a, b, n, mode, c,
                                                                                              out_acc);
  HG_CHECK_CUDA(cudaGetLastError());
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

extern "C" int hg_segment_gather(const float* pool, const long long* start, const int* valid, int batch,
                                 int seg, float* out, void* stream) {
  HG_REQUIRE(pool && start && valid && out && batch > 0 && batch <= 65535 && seg > 0,
             "hg_segment_gather: bad arguments");
  dim3 grid((seg + 1023) / 1024 < 64 ? (seg + 1023) / 1024 : 64, batch);
  segment_gather_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(pool, start, valid, seg, out);
  HG_CHECK_CUDA(cudaGetLastError());
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

extern "C" int hg_segment_stage_i16(const int16_t* staged, const int* peak, const int* valid, int batch, int seg,
                                    int mode, float* out, void* stream) {
  HG_REQUIRE(staged && peak && valid && out && batch > 0 && batch <= 65535 && seg > 0 &&
             (mode == HG_STAGE_PEAK || mode == HG_STAGE_FORK || mode == HG_STAGE_NONE),
             "hg_segment_stage_i16: bad arguments");
  dim3 grid((seg + 256 * 8 - 1) / (256 * 8), batch);
  const bool vec = seg % 8 == 0 && reinterpret_cast<uintptr_t>(staged) % 16 == 0 &&
                   reinterpret_cast<uintptr_t>(out) % 16 == 0;
  if (vec)
    segment_stage_i16_kernel<true><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(staged, peak, valid, seg,
                                                                                        mode, out);
  else
    segment_stage_i16_kernel<false><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(staged, peak, valid, seg,
                                                                                         mode, out);
  HG_CHECK_CUDA(cudaGetLastError());
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

extern "C" int hg_segment_stage_mel(const float* staged, const int* valid_frames, int batch, int fps, int num_mels,
                                    float* out, void* stream) {
  HG_REQUIRE(staged && valid_frames && out && batch > 0 && batch <= 65535 && fps > 0 && num_mels > 0 &&
             (num_mels + 31) / 32 <= 65535, "hg_segment_stage_mel: bad arguments");
  dim3 grid((fps + 31) / 32, (num_mels + 31) / 32, batch), block(32, 8);
  segment_stage_mel_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(staged, valid_frames, fps,
                                                                                  num_mels, out);
  HG_CHECK_CUDA(cudaGetLastError());
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

extern "C" int hg_pack_conv1d_weight(const float* v, const float* g, int cout, int cin, int k,
                                     int cin_pad, void* w_packed, void* stream) {
  HG_REQUIRE(v && w_packed, "hg_pack_conv1d_weight: null pointer");
  HG_REQUIRE(cout > 0 && cin > 0 && k > 0 && cin_pad >= cin, "hg_pack_conv1d_weight: bad shape");
  pack_conv1d_weight_kernel<<<cout, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      v, g, cout, cin, k, cin_pad, static_cast<__nv_bfloat16*>(w_packed));
  HG_CHECK_CUDA(cudaGetLastError());
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

extern "C" int hg_convtr1d_geometry(int k, int stride, int padding, int* host_nshift,
                                    int* host_shift_min) {
  HG_REQUIRE(k > 0 && stride > 0 && padding >= 0, "hg_convtr1d_geometry: bad arguments");
  // shift s = (p + padding - j) / stride for phases p in [0,stride), taps j in [0,k)
  auto floordiv = [](int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); };
  const int s_max = floordiv(stride - 1 + padding, stride);
  const int s_min = -floordiv(k - 1 - padding, stride);  // ceil((padding-(k-1))/stride)
  if (host_nshift) *host_nshift = s_max - s_min + 1;
  if (host_shift_min) *host_shift_min = s_min;
  return HG_OK;
}

extern "C" int hg_pack_convtr1d_weight(const float* v, const float* g, int cin, int cout, int k,
                                       int stride, int padding, void* w_packed, void* stream) {
  HG_REQUIRE(v && w_packed, "hg_pack_convtr1d_weight: null pointer");
  int nshift = 0, shift_min = 0;
  int rc = hg_convtr1d_geometry(k, stride, padding, &nshift, &shift_min);
  if (rc) return rc;
  pack_convtr1d_weight_kernel<<<cin, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      v, g, cin, cout, k, stride, padding, nshift, shift_min,
      static_cast<__nv_bfloat16*>(w_packed));
  HG_CHECK_CUDA(cudaGetLastError());
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

extern "C" int hg_ncl_to_nlc(const float* x, int batch, int c, int t, int c_pad, void* out,
                             void* out_act, float act_slope, void* stream) {
  HG_REQUIRE(x && (out || out_act), "hg_ncl_to_nlc: null pointer");
  HG_REQUIRE(batch > 0 && c > 0 && t > 0 && c_pad >= c, "hg_ncl_to_nlc: bad shape");
  HG_REQUIRE(batch <= 65535, "hg_ncl_to_nlc: batch too large");
  dim3 grid((t + 31) / 32, (c_pad + 31) / 32, batch), block(32, 8);
  ncl_to_nlc_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(
      x, c, t, c_pad, static_cast<__nv_bfloat16*>(out), static_cast<__nv_bfloat16*>(out_act),
      act_slope);
  HG_CHECK_CUDA(cudaGetLastError());
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

extern "C" int hg_nlc_to_ncl(const void* x, int batch, int t, int c, float* out, void* stream) {
  HG_REQUIRE(x && out, "hg_nlc_to_ncl: null pointer");
  HG_REQUIRE(batch > 0 && c > 0 && t > 0, "hg_nlc_to_ncl: bad shape");
  HG_REQUIRE(batch <= 65535 && (t + 31) / 32 <= 65535, "hg_nlc_to_ncl: grid too large");
  dim3 grid((c + 31) / 32, (t + 31) / 32, batch), block(32, 8);
  nlc_to_ncl_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(x), t, c, out);
  HG_CHECK_CUDA(cudaGetLastError());
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

template <int TH>
static int launch_post2(const __nv_bfloat16* x, const float* w, const float* bias, int batch, int t, float* y,
                        cudaStream_t st) {
  constexpr int tile = kPost2R * TH;
  constexpr size_t smem = ((7 * 32 * 4 + 15) & ~15) + static_cast<size_t>(tile + 7 - 1) * (32 * 2 + 8);
  static hg::PerDeviceOnce once;
  if (once.need())
    HG_CHECK_CUDA(cudaFuncSetAttribute(conv_post_tanh_kernel2<32, 7, TH>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
  dim3 grid((t + tile - 1) / tile, batch);
  conv_post_tanh_kernel2<32, 7, TH><<<grid, TH, smem, st>>>(x, w, bias, t, y);
  HG_CHECK_CUDA(cudaGetLastError());
  return HG_OK;
}

extern "C" int hg_conv_post_tanh_fwd(const void* x, const float* w, const float* bias, int batch,
                                     int t, int c, int k, float* y, void* stream) {
  HG_REQUIRE(x && w && y, "hg_conv_post_tanh_fwd: null pointer");
  HG_REQUIRE(batch > 0 && t > 0 && c > 0 && c % 8 == 0 && k > 0 && (k & 1) && k <= 15,
             "hg_conv_post_tanh_fwd: bad shape (c %% 8 == 0, odd k <= 15 required)");
  HG_REQUIRE(batch <= 65535, "hg_conv_post_tanh_fwd: batch too large");
  if (c == 32 && k == 7) {  // every shipped config (conv_post: 32 -> 1, k = 7)
    // 64 threads x 9 outputs per block (42 KB of staged rows, 5 blocks per SM): 0.486 ms per 16.8 M samples against
    // 0.609 ms with 128 threads and 0.781 ms for the kernel above (profiles/r02_summary.md section 4)
    const int rc = launch_post2<64>(static_cast<const __nv_bfloat16*>(x), w, bias, batch, t, y,
                                    static_cast<cudaStream_t>(stream));
    if (rc) return rc;
    g_hg_launches.fetch_add(1, std::memory_order_relaxed);
    return HG_OK;
  }
  const size_t smem = ((k * c * 4 + 15) & ~15) + static_cast<size_t>(kPostTile + k - 1) * (c * 2 + 16);
  HG_REQUIRE(smem <= 200 * 1024, "hg_conv_post_tanh_fwd: window does not fit shared memory");
  dim3 grid((t + kPostTile - 1) / kPostTile, batch);
  if (smem > 48 * 1024)
    HG_CHECK_CUDA(cudaFuncSetAttribute(conv_post_tanh_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
  conv_post_tanh_kernel<<<grid, kPostThreads, smem, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(x), w, bias, t, c, k, y);
  HG_CHECK_CUDA(cudaGetLastError());
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}
