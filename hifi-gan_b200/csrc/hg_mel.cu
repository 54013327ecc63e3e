// hg_mel.cu — mel_spectrogram (src/meldataset.py:56-85) as ONE fused kernel:
//   reflect-pad -> frame x periodic Hann -> rFFT(n_fft) -> |X|^2 -> HTK mel (sparse) -> log(clamp(.,1e-5))
// The reference goes through torchaudio.transforms.MelSpectrogram (meldataset.py:59-71): >= 6 library
// launches and three HBM round trips of the [B,513,F] spectrum.  n_fft in {256, 512, 1024, 2048} runs mel_kernel2<N2>
// (one warp per 32 / N2 frames, the FFT in registers), any other n_fft the direct-DFT mel_dft_kernel.  The backward
// mel_bwd_kernel<N> (one thread group per frame running an N = n_fft / 2 point complex Stockham FFT, radix 8 x 8 then
// 2, 4, 8 or 8 x 2, on the even/odd packed samples) takes the same four sizes.
//
// The per-thread phases are __host__ __device__ so tests can run the exact same arithmetic on the CPU
// (hg_mel_emulate_host, hg_mel_bwd_emulate_host below) — there is no GPU in the development container.
#include "hg_common.cuh"

#include <atomic>
#include <cmath>
#include <vector>

#include "../../include/hifigan_b200.h"

extern std::atomic<int64_t> g_hg_launches;

struct hg_mel_plan {
  int n_fft, num_mels, sampling_rate, hop, win, pad;
  double fmin, fmax;
  int nnz;
  // device tables
  float* window;     // [n_fft]
  float2* tw_half;   // [n_fft/2]    exp(-2*pi*i*m/(n_fft/2)): the FFT sizes only (null otherwise)
  float2* tw_full;   // [n_fft/2+1]  exp(-2*pi*i*k/n_fft): the FFT sizes only (null otherwise)
  float2* tw_n;      // [n_fft] (cos, sin)(2*pi*n/n_fft): the direct-DFT path of every other n_fft
  int* mel_start;    // [num_mels] first rFFT bin with a non-zero weight
  int* mel_off;      // [num_mels+1] CSR offsets into mel_w
  float* mel_w;      // [nnz]
  // host copies (CPU emulation for tests, and geometry queries)
  std::vector<float> h_window;
  std::vector<float2> h_tw_half, h_tw_full, h_tw_n;
  std::vector<int> h_mel_start, h_mel_off;
  std::vector<float> h_mel_w;
};

namespace {

// the transform sizes with an FFT path, forward and backward: n_fft = 256, 512, 1024, 2048
__host__ __device__ constexpr bool is_fft_size(int n_fft) {
  return n_fft == 256 || n_fft == 512 || n_fft == 1024 || n_fft == 2048;
}

__host__ __device__ __forceinline__ int padi(int i) { return i + (i >> 4); }
// complex entries of an N-point buffer addressed through padi: padi(N - 1) + 1, rounded up
__host__ __device__ constexpr int pad_len(int n) { return n + n / 16; }

struct cpx {
  float x, y;
};
__host__ __device__ __forceinline__ cpx cadd(cpx a, cpx b) { return {a.x + b.x, a.y + b.y}; }
__host__ __device__ __forceinline__ cpx csub(cpx a, cpx b) { return {a.x - b.x, a.y - b.y}; }
__host__ __device__ __forceinline__ cpx cmul(cpx a, cpx b) {
  return {a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x};
}
__host__ __device__ __forceinline__ cpx mul_negi(cpx a) { return {a.y, -a.x}; }  // a * (-i)

__host__ __device__ __forceinline__ void fft4(cpx& x0, cpx& x1, cpx& x2, cpx& x3) {
  const cpx b0 = cadd(x0, x2), b2 = csub(x0, x2), b1 = cadd(x1, x3), b3 = mul_negi(csub(x1, x3));
  x0 = cadd(b0, b1);
  x2 = csub(b0, b1);
  x1 = cadd(b2, b3);
  x3 = csub(b2, b3);
}

// in-place 8-point DFT (forward, e^{-i...}), natural order out
__host__ __device__ __forceinline__ void fft8(cpx (&v)[8]) {
  const float h = 0.70710678118654752440f;
  cpx a0 = cadd(v[0], v[4]), a4 = csub(v[0], v[4]);
  cpx a1 = cadd(v[1], v[5]), a5 = csub(v[1], v[5]);
  cpx a2 = cadd(v[2], v[6]), a6 = csub(v[2], v[6]);
  cpx a3 = cadd(v[3], v[7]), a7 = csub(v[3], v[7]);
  a5 = cpx{(a5.x + a5.y) * h, (a5.y - a5.x) * h};    // * (1 - i)/sqrt2
  a6 = mul_negi(a6);                                 // * (-i)
  a7 = cpx{(a7.y - a7.x) * h, -(a7.x + a7.y) * h};   // * (-1 - i)/sqrt2
  fft4(a0, a1, a2, a3);
  fft4(a4, a5, a6, a7);
  v[0] = a0; v[2] = a1; v[4] = a2; v[6] = a3;
  v[1] = a4; v[3] = a5; v[5] = a6; v[7] = a7;
}

__host__ __device__ __forceinline__ void fft_radix(cpx (&v)[2]) {
  const cpx a = cadd(v[0], v[1]);
  v[1] = csub(v[0], v[1]);
  v[0] = a;
}
__host__ __device__ __forceinline__ void fft_radix(cpx (&v)[4]) { fft4(v[0], v[1], v[2], v[3]); }
__host__ __device__ __forceinline__ void fft_radix(cpx (&v)[8]) { fft8(v); }

// One Stockham radix-R pass of an N-point FFT for butterfly j in [0, N / R); tw holds W_N^m, m in [0, N).
//   FIRST: inputs come from the staged real samples (even/odd packing + window), Ns = 1.
template <int R, int N, bool FIRST>
__host__ __device__ __forceinline__ void fft_pass(int j, int ns, const cpx* __restrict__ in,
                                                  cpx* __restrict__ out,
                                                  const float* __restrict__ samples,
                                                  const float* __restrict__ window,
                                                  const float2* __restrict__ tw) {
  constexpr int kStride = N / R;
  cpx v[R];
  const int k = j & (ns - 1);
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int n = j + r * kStride;
    if (FIRST) {
      v[r] = cpx{samples[2 * n] * window[2 * n], samples[2 * n + 1] * window[2 * n + 1]};
    } else {
      v[r] = in[padi(n)];
      if (r) {
        const float2 w = tw[r * k * (kStride / ns)];
        v[r] = cmul(v[r], cpx{w.x, w.y});
      }
    }
  }
  fft_radix(v);
  const int j0 = (j / ns) * ns * R + k;
#pragma unroll
  for (int r = 0; r < R; ++r) out[padi(j0 + r * ns)] = v[r];
}
// the pass for thread j of a G-thread group: N / R butterflies, a whole number of them per thread, or (N = 128, radix
// 8: 16 butterflies over 32 threads) one each for the first N / R threads
template <int R, int N, int G, bool FIRST>
__host__ __device__ __forceinline__ void fft_pass_group(int j, int ns, const cpx* __restrict__ in,
                                                        cpx* __restrict__ out, const float* __restrict__ samples,
                                                        const float* __restrict__ window,
                                                        const float2* __restrict__ tw) {
  constexpr int kBfly = N / R;
  if constexpr (kBfly < G) {
    if (j < kBfly) fft_pass<R, N, FIRST>(j, ns, in, out, samples, window, tw);
  } else {
    static_assert(kBfly % G == 0, "butterflies must split evenly over the group");
#pragma unroll
    for (int i = 0; i < kBfly / G; ++i) fft_pass<R, N, FIRST>(j + i * G, ns, in, out, samples, window, tw);
  }
}
// N = 8 x 8 x R3 (x 2 at N = 1024): the radix of the third pass
__host__ __device__ constexpr int third_radix(int n) { return n >= 512 ? 8 : n / 64; }

__host__ __device__ __forceinline__ int reflect_index(int i, int t) {
  if (i < 0) i = -i;
  if (i >= t) i = 2 * (t - 1) - i;
  return i;
}

__device__ __forceinline__ void atomic_min_f32(float* addr, float v) {
  if (v >= 0.f) atomicMin(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMax(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_f32(float* addr, float v) {
  if (v >= 0.f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

// asynchronous global -> shared copies (LDGSTS): every copy of the block prologue is in flight at once, so the
// prologue costs one memory round trip instead of one per dependent load / store pair (ncu source view of the
// round-1 forward kernel: the staging stores waiting on their loads, and the barrier behind them, were ~25 % of its
// stall samples)
__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(hg::smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(void* dst_smem, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(hg::smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
// nbytes (a multiple of 4) from a 16-byte aligned global table into a 16-byte aligned shared region
__device__ __forceinline__ void cp_async_table(void* dst_smem, const void* src, int nbytes, int tid, int nthreads) {
  const int n16 = nbytes >> 4;
  for (int i = tid; i < n16; i += nthreads)
    cp_async16(static_cast<uint8_t*>(dst_smem) + 16 * i, static_cast<const uint8_t*>(src) + 16 * i);
  for (int i = n16 * 4 + tid; i < (nbytes >> 2); i += nthreads)
    cp_async4(static_cast<uint8_t*>(dst_smem) + 4 * i, static_cast<const uint8_t*>(src) + 4 * i);
}
// the G threads (whole warps) of a frame group meet on their own named barrier: groups drift apart freely
template <int G>
__device__ __forceinline__ void group_sync(int g) {
  asm volatile("bar.sync %0, %1;" ::"r"(g + 1), "n"(G) : "memory");
}

// ---------------------------------------------------------------------------------------------
// mel_kernel2 — the forward kernel of round 2: ONE WARP PER TWO FRAMES, the FFT held in registers.
//
// The N-point complex FFT (N = n_fft / 2 = 32 N2, N2 in {4, 8, 16, 32}) of a frame's even/odd packed samples is split
// N = 32 x N2 (n = N2 n1 + n2, k = k1 + 32 k2):
//   Z[k1 + 32 k2] = sum_n2 W_N2^(n2 k2) [ W_N^(n2 k1) sum_n1 z[N2 n1 + n2] W32^(n1 k1) ]
// A warp serves 32 / N2 frames (n_fft 256 / 512 / 1024 / 2048: 8 / 4 / 2 / 1).
//   phase 1  lane = (frame, n2): 32 windowed complex samples straight from global memory (64-bit coalesced loads,
//            reflect padding by index arithmetic), a 32-point DFT in registers (4 x 8, compile-time twiddles), the
//            W_N twiddles from a padded shared table, results to the warp's exchange buffer (conflict-free pitch 33)
//   phase 2  lane = k1: the N2 values of each frame from the exchange buffer, an N2-point DFT in registers,
//            Z to shared memory in natural order
//   phase 3  lane = k mod 32: real-FFT un-pack of its N2 (+1) bins from Z[k], Z[N - k], |X|^2 (only up to the last
//            bin any mel filter reads), written over the frame's own Z region
//   phase 4  lane = mel bin mod 32: the CSR triangle sums + log(clamp), staged for 64-byte output runs
// Warps never meet (__syncwarp between phases); a block is 8 warps = 8 x 32 / N2 consecutive frames and loops over
// frame groups, so the constant tables are loaded once per block.  At n_fft 1024 ~2.4x fewer warp-instructions per
// frame than the round-1 radix-8 x 8 x 8 shared-memory kernel (whose FFT passes, fft_pass above, the backward kernel
// still runs), and no block-wide or named barriers on the frame path.  Every size holds 32 complex values per lane in
// phases 1 and 2, and uses the same exchange buffer.
// The lane phases are __host__ __device__ (hg_mel_emulate_host runs them lane by lane on the CPU).
constexpr int kExPitch = 33;                              // complex per (frame, n2) row of the exchange buffer
constexpr int kWarpScratch = 32 * kExPitch;               // complex per warp (8448 B) >= (32 / N2) x N (the Z / power view)
constexpr int kMel2Warps = 8;
constexpr int kMel2Threads = kMel2Warps * 32;
template <int N2>
struct Mel2Size {
  static constexpr int kN = 32 * N2;                      // complex FFT points; n_fft = 2 kN
  static constexpr int kNfft = 2 * kN;
  static constexpr int kFramesPerWarp = 32 / N2;
  static constexpr int kFramesPerBlock = kMel2Warps * kFramesPerWarp;
  static constexpr int kTwPad = pad_len(kN);              // padi(kN - 1) + 1, rounded up
  static_assert(kFramesPerWarp * kN <= kWarpScratch, "the Z view must fit the exchange buffer");
};

// e^{-2 pi i j / 32}, j a compile-time constant after unrolling
__host__ __device__ __forceinline__ cpx w32(int j) {
  constexpr float c[9] = {1.f, 0.98078528040323044913f, 0.92387953251128675613f, 0.83146961230254523708f,
                          0.70710678118654752440f, 0.55557023301960222474f, 0.38268343236508977173f,
                          0.19509032201612826785f, 0.f};
  // cos(2 pi j / 32) for j in [0, 32) by symmetry around the quarter turns; sin likewise
  const int q = j & 31;
  const int r = q & 7, quad = q >> 3;
  const float cr = c[r], sr = c[8 - r];                   // cos, sin of the first-quadrant remainder
  switch (quad) {
    case 0: return cpx{cr, -sr};
    case 1: return cpx{-sr, -cr};
    case 2: return cpx{-cr, sr};
    default: return cpx{sr, cr};
  }
}

// 32-point DFT (forward), v in natural order -> natural order
__host__ __device__ __forceinline__ void fft32(cpx (&v)[32]) {
#pragma unroll
  for (int b = 0; b < 8; ++b) fft4(v[b], v[8 + b], v[16 + b], v[24 + b]);       // over a (n = 8a + b): v[8 ka + b]
#pragma unroll
  for (int ka = 1; ka < 4; ++ka)
#pragma unroll
    for (int b = 1; b < 8; ++b) v[8 * ka + b] = cmul(v[8 * ka + b], w32(b * ka));
  cpx o[32];
#pragma unroll
  for (int ka = 0; ka < 4; ++ka) {
    cpx t[8];
#pragma unroll
    for (int b = 0; b < 8; ++b) t[b] = v[8 * ka + b];
    fft8(t);
#pragma unroll
    for (int kb = 0; kb < 8; ++kb) o[ka + 4 * kb] = t[kb];
  }
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = o[i];
}

// 16-point DFT (forward), natural order in and out
__host__ __device__ __forceinline__ void fft16(cpx (&v)[16]) {
#pragma unroll
  for (int b = 0; b < 4; ++b) fft4(v[b], v[4 + b], v[8 + b], v[12 + b]);        // n = 4a + b -> v[4 ka + b]
#pragma unroll
  for (int ka = 1; ka < 4; ++ka)
#pragma unroll
    for (int b = 1; b < 4; ++b) v[4 * ka + b] = cmul(v[4 * ka + b], w32(2 * b * ka));
  cpx o[16];
#pragma unroll
  for (int ka = 0; ka < 4; ++ka) {
    cpx t0 = v[4 * ka], t1 = v[4 * ka + 1], t2 = v[4 * ka + 2], t3 = v[4 * ka + 3];
    fft4(t0, t1, t2, t3);
    o[ka] = t0; o[ka + 4] = t1; o[ka + 8] = t2; o[ka + 12] = t3;
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = o[i];
}

// the N2-point DFT of the second factor (phase 2 of mel_kernel2<N2>)
__host__ __device__ __forceinline__ void fft_n2(cpx (&v)[4]) { fft4(v[0], v[1], v[2], v[3]); }
__host__ __device__ __forceinline__ void fft_n2(cpx (&v)[8]) { fft8(v); }
__host__ __device__ __forceinline__ void fft_n2(cpx (&v)[16]) { fft16(v); }
__host__ __device__ __forceinline__ void fft_n2(cpx (&v)[32]) { fft32(v); }

struct Mel2Args {
  const float* y;
  float* out;
  float* minmax;
  int batch, t, frames, hop, pad, num_mels;
  const float* window;
  const float2* tw_half;  // W_N^m, m < N
  const float2* tw_full;  // W_2N^k, k <= N
  const int* mel_start;
  const int* mel_off;
  const float* mel_w;
  int nnz, max_bin;       // max_bin: the last rFFT bin any mel filter reads
  int groups_per_item;    // ceil(frames / kFramesPerBlock)
  int total_groups;       // batch * groups_per_item
};

// phase 1 (lane = N2 * frame + n2): frame samples -> window -> DFT-32 -> W_N twiddle -> exchange buffer.
// `yb` is the batch item, `start` the (possibly negative) first sample of this lane's frame, `vec` whether the
// frame is interior and 8-byte aligned (plain 64-bit loads).  Returns the lane's sample extrema through lo / hi.
template <int N2>
__host__ __device__ __forceinline__ void mel2_phase1(int lane, const float* __restrict__ yb, int start, int t, bool vec,
                                                     const float* __restrict__ window, const float2* __restrict__ twp,
                                                     cpx* __restrict__ ex, float& lo, float& hi) {
  const int n2 = lane & (N2 - 1);
  cpx v[32];
#pragma unroll
  for (int n1 = 0; n1 < 32; ++n1) {
    const int s = 2 * N2 * n1 + 2 * n2;
    float x0, x1;
    if (vec) {
      const float2 xv = *reinterpret_cast<const float2*>(yb + start + s);
      x0 = xv.x; x1 = xv.y;
    } else {
      x0 = yb[reflect_index(start + s, t)];
      x1 = yb[reflect_index(start + s + 1, t)];
    }
    lo = fminf(lo, fminf(x0, x1));
    hi = fmaxf(hi, fmaxf(x0, x1));
    const float2 w = *reinterpret_cast<const float2*>(window + s);
    v[n1] = cpx{x0 * w.x, x1 * w.y};
  }
  fft32(v);
  cpx* row = ex + lane * kExPitch;          // (frame * N2 + n2) * pitch
  row[0] = v[0];
#pragma unroll
  for (int k1 = 1; k1 < 32; ++k1) {
    const float2 w = twp[padi(n2 * k1)];
    row[k1] = cmul(v[k1], cpx{w.x, w.y});
  }
}
// phase 2a (lane = k1): gather the N2 n2 values of each of the warp's frames; 2b: DFT-N2, Z in natural order over the
// same buffer (frame h's Z at z + h N)
template <int N2>
__host__ __device__ __forceinline__ void mel2_phase2_read(int lane, const cpx* __restrict__ ex,
                                                          cpx (&a)[32 / N2][N2]) {
#pragma unroll
  for (int n2 = 0; n2 < N2; ++n2)
#pragma unroll
    for (int h = 0; h < 32 / N2; ++h) a[h][n2] = ex[(h * N2 + n2) * kExPitch + lane];
}
template <int N2>
__host__ __device__ __forceinline__ void mel2_phase2_write(int lane, cpx (&a)[32 / N2][N2], cpx* __restrict__ z) {
#pragma unroll
  for (int h = 0; h < 32 / N2; ++h) fft_n2(a[h]);
#pragma unroll
  for (int k2 = 0; k2 < N2; ++k2)
#pragma unroll
    for (int h = 0; h < 32 / N2; ++h) z[h * Mel2Size<N2>::kN + lane + 32 * k2] = a[h][k2];
}
// phase 3a (lane = k mod 32): |X[k]|^2 of the lane's bins k = lane + 32 k2 (k <= max_bin) of one frame's Z;
// pw[N2] is bin N (lane 0).  3b: the powers go over the frame's own Z region (as floats).
template <int N2>
__host__ __device__ __forceinline__ void mel2_phase3_compute(int lane, const cpx* __restrict__ z, int max_bin,
                                                             const float2* __restrict__ tw_full, float (&pw)[N2 + 1]) {
  constexpr int kN = Mel2Size<N2>::kN;
#pragma unroll
  for (int k2 = 0; k2 < N2; ++k2) {
    const int k = lane + 32 * k2;
    float p = 0.f;
    if (k <= max_bin) {
      const cpx zk = z[k];
      cpx zc = z[(kN - k) & (kN - 1)];
      zc.y = -zc.y;
      const cpx e = cpx{0.5f * (zk.x + zc.x), 0.5f * (zk.y + zc.y)};
      const cpx d = csub(zk, zc);
      const cpx o = cpx{0.5f * d.y, -0.5f * d.x};  // (zk - zc) / (2i)
      const float2 w = tw_full[k];
      const cpx x = cadd(e, cmul(o, cpx{w.x, w.y}));
      p = x.x * x.x + x.y * x.y;
    }
    pw[k2] = p;
  }
  pw[N2] = 0.f;
  if (lane == 0 && kN <= max_bin) {
    const cpx z0 = z[0];                           // X[N] = Re Z[0] - Im Z[0]
    pw[N2] = (z0.x - z0.y) * (z0.x - z0.y);
  }
}
template <int N2>
__host__ __device__ __forceinline__ void mel2_phase3_write(int lane, const float (&pw)[N2 + 1], float* __restrict__ power) {
#pragma unroll
  for (int k2 = 0; k2 < N2; ++k2) power[lane + 32 * k2] = pw[k2];
  if (lane == 0) power[Mel2Size<N2>::kN] = pw[N2];
}
// phase 4 (lane = m mod 32): CSR triangle sums + log(clamp(., 1e-5)) of one frame -> out_col[m * out_stride]
__host__ __device__ __forceinline__ void mel2_phase4(int lane, int num_mels, const float* __restrict__ power,
                                                     const int* __restrict__ mel_start, const int* __restrict__ mel_off,
                                                     const float* __restrict__ mel_w, float* __restrict__ out_col,
                                                     int out_stride) {
  for (int m = lane; m < num_mels; m += 32) {
    const int s = mel_start[m], o = mel_off[m], n = mel_off[m + 1] - o;
    float acc = 0.f;
    for (int i = 0; i < n; ++i) acc += mel_w[o + i] * power[s + i];
    out_col[m * out_stride] = logf(fmaxf(acc, 1e-5f));
  }
}

struct Mel2Smem {
  uint32_t win, tw_half, tw_full, melw, melidx, meloff, scratch, outs, total;
};
template <int N2>
__host__ __device__ inline Mel2Smem mel2_smem_layout(int num_mels, int nnz) {
  using S = Mel2Size<N2>;
  auto up = [](uint32_t v) { return (v + 15u) & ~15u; };
  Mel2Smem l;
  uint32_t o = 0;
  l.win = o;      o += S::kNfft * 4u;
  l.tw_half = o;  o += up(S::kTwPad * 8u);
  l.tw_full = o;  o += up((S::kN + 1) * 8u);
  l.melw = o;     o += up(static_cast<uint32_t>(nnz > 0 ? nnz : 1) * 4u);
  l.melidx = o;   o += up(static_cast<uint32_t>(num_mels) * 4u);
  l.meloff = o;   o += up(static_cast<uint32_t>(num_mels + 1) * 4u);
  l.scratch = o;  o += kMel2Warps * kWarpScratch * 8u;
  l.outs = o;     o += static_cast<uint32_t>(num_mels) * S::kFramesPerBlock * 4u;
  l.total = o;
  return l;
}

template <int N2>
__global__ void __launch_bounds__(kMel2Threads, 2) mel_kernel2(const Mel2Args a) {
  using S = Mel2Size<N2>;
  constexpr int kN = S::kN, kFPW = S::kFramesPerWarp, kFPB = S::kFramesPerBlock;
  extern __shared__ __align__(16) uint8_t sm[];
  constexpr int kThreads2 = kMel2Threads;
  const Mel2Smem L = mel2_smem_layout<N2>(a.num_mels, a.nnz);
  float* s_win = reinterpret_cast<float*>(sm + L.win);
  float2* s_twp = reinterpret_cast<float2*>(sm + L.tw_half);                   // padded: entry i at padi(i)
  float2* s_twf = reinterpret_cast<float2*>(sm + L.tw_full);
  float* s_melw = reinterpret_cast<float*>(sm + L.melw);
  int* s_start = reinterpret_cast<int*>(sm + L.melidx);
  int* s_off = reinterpret_cast<int*>(sm + L.meloff);
  float* outs = reinterpret_cast<float*>(sm + L.outs);                         // [num_mels][kFPB]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  cpx* scratch = reinterpret_cast<cpx*>(sm + L.scratch) + warp * kWarpScratch;

  cp_async_table(s_win, a.window, S::kNfft * 4, tid, kThreads2);
  cp_async_table(s_twf, a.tw_full, (kN + 1) * 8, tid, kThreads2);
  cp_async_table(s_melw, a.mel_w, a.nnz * 4, tid, kThreads2);
  cp_async_table(s_start, a.mel_start, a.num_mels * 4, tid, kThreads2);
  cp_async_table(s_off, a.mel_off, (a.num_mels + 1) * 4, tid, kThreads2);
  for (int i = tid; i < kN; i += kThreads2) s_twp[padi(i)] = a.tw_half[i];
  cp_async_wait_all();
  __syncthreads();

  float vmin = INFINITY, vmax = -INFINITY;
  for (int grp = blockIdx.x; grp < a.total_groups; grp += gridDim.x) {
    const int b = grp / a.groups_per_item;
    const int f0 = (grp - b * a.groups_per_item) * kFPB;
    const float* yb = a.y + static_cast<size_t>(b) * a.t;
    const int fl0 = kFPW * warp;                        // this warp's frames within the group
    const int f = f0 + fl0 + lane / N2;
    const bool live = f < a.frames;                     // uniform over the lane's N2-lane frame
    if (f0 + fl0 < a.frames) {                          // warp-uniform: at least the first frame exists
      const int start = (live ? f : a.frames - 1) * a.hop - a.pad;
      const bool vec = start >= 0 && start + S::kNfft <= a.t &&
                       ((reinterpret_cast<uintptr_t>(yb + start) & 7) == 0);
      float lo = INFINITY, hi = -INFINITY;
      mel2_phase1<N2>(lane, yb, start, a.t, vec, s_win, s_twp, scratch, lo, hi);
      if (live) { vmin = fminf(vmin, lo); vmax = fmaxf(vmax, hi); }
      __syncwarp();
      cpx za[kFPW][N2];
      mel2_phase2_read<N2>(lane, scratch, za);
      __syncwarp();
      mel2_phase2_write<N2>(lane, za, scratch);
      __syncwarp();
#pragma unroll
      for (int h = 0; h < kFPW; ++h) {
        float pw[N2 + 1];
        mel2_phase3_compute<N2>(lane, scratch + h * kN, a.max_bin, s_twf, pw);
        __syncwarp();
        float* power = reinterpret_cast<float*>(scratch + h * kN);
        mel2_phase3_write<N2>(lane, pw, power);
        __syncwarp();
        if (f0 + fl0 + h < a.frames)
          mel2_phase4(lane, a.num_mels, power, s_start, s_off, s_melw, outs + fl0 + h, kFPB);
      }
    }
    __syncthreads();
    // outs[m][fl] -> out[b][m][f0 + fl]
    float* ob = a.out + static_cast<size_t>(b) * a.num_mels * a.frames;
    for (int i = tid; i < a.num_mels * kFPB; i += kThreads2) {
      const int m = i / kFPB, fl = i % kFPB;
      if (f0 + fl < a.frames) ob[static_cast<size_t>(m) * a.frames + f0 + fl] = outs[i];
    }
    __syncthreads();
  }
  if (a.minmax) {
    for (int o = 16; o > 0; o >>= 1) {
      vmin = fminf(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
      vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    }
    if (lane == 0) {
      if (vmin < *reinterpret_cast<volatile float*>(a.minmax)) atomic_min_f32(a.minmax, vmin);
      if (vmax > *reinterpret_cast<volatile float*>(a.minmax + 1)) atomic_max_f32(a.minmax + 1, vmax);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Every n_fft without an FFT path (not a power of two, or outside 256..2048: the reference's other callers pass n_fft =
// a layer's kernel size at sr 16000, src/speech_distillation/lightning_model.py:513-522, custom_layers.py:138-161):
// one block per frame, direct DFT
// over a shared-memory twiddle table.  O(n_fft^2 / 2) per frame — a general-purpose path, not the tuned one.
// Per-bin and per-mel phases are __host__ __device__ so hg_mel_emulate_host runs the same arithmetic.
__host__ __device__ inline float dft_bin_power(int k, int n_fft, const float* xw, const float2* tw) {
  float ar = 0.f, ai = 0.f;
  int idx = 0;                                  // (k * n) mod n_fft, advanced incrementally
  for (int n = 0; n < n_fft; ++n) {
    const float2 c = tw[idx];
    ar += xw[n] * c.x;
    ai -= xw[n] * c.y;
    idx += k;
    if (idx >= n_fft) idx -= n_fft;
  }
  return ar * ar + ai * ai;
}
__host__ __device__ inline float mel_bin_log(int m, const float* power, const int* mel_start, const int* mel_off,
                                             const float* mel_w) {
  const int k0 = mel_start[m], o0 = mel_off[m], cnt = mel_off[m + 1] - o0;
  float acc = 0.f;
  for (int i = 0; i < cnt; ++i) acc += mel_w[o0 + i] * power[k0 + i];
  return logf(fmaxf(acc, 1e-5f));
}

__global__ void __launch_bounds__(256)
mel_dft_kernel(const float* __restrict__ y, int t, int frames, int n_fft, int hop, int pad, int num_mels,
               const float* __restrict__ window, const float2* __restrict__ twiddle, const int* __restrict__ mel_start,
               const int* __restrict__ mel_off, const float* __restrict__ mel_w, float* __restrict__ out,
               float* __restrict__ minmax) {
  extern __shared__ __align__(16) uint8_t smg[];
  float2* tw = reinterpret_cast<float2*>(smg);                  // [n_fft]
  float* xw = reinterpret_cast<float*>(tw + n_fft);             // [n_fft]
  float* power = xw + n_fft;                                    // [n_fft / 2 + 1]
  const int f = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const float* yb = y + static_cast<size_t>(b) * t;
  float vmin = INFINITY, vmax = -INFINITY;
  for (int n = tid; n < n_fft; n += 256) {
    const float v = yb[reflect_index(f * hop + n - pad, t)];
    vmin = fminf(vmin, v);
    vmax = fmaxf(vmax, v);
    xw[n] = v * window[n];
    tw[n] = twiddle[n];
  }
  if (minmax) {
    for (int o = 16; o > 0; o >>= 1) {
      vmin = fminf(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
      vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    }
    if ((tid & 31) == 0) {
      if (vmin < *reinterpret_cast<volatile float*>(minmax)) atomic_min_f32(minmax, vmin);
      if (vmax > *reinterpret_cast<volatile float*>(minmax + 1)) atomic_max_f32(minmax + 1, vmax);
    }
  }
  __syncthreads();
  const int nbins = n_fft / 2 + 1;
  for (int k = tid; k < nbins; k += 256) power[k] = dft_bin_power(k, n_fft, xw, tw);
  __syncthreads();
  for (int m = tid; m < num_mels; m += 256)
    out[(static_cast<size_t>(b) * num_mels + m) * frames + f] = mel_bin_log(m, power, mel_start, mel_off, mel_w);
}

double hz_to_mel_htk(double f) { return 2595.0 * std::log10(1.0 + f / 700.0); }
double mel_to_hz_htk(double m) { return 700.0 * (std::pow(10.0, m / 2595.0) - 1.0); }

}  // namespace

extern "C" int hg_mel_num_frames(const hg_mel_plan* plan, int t) {
  if (!plan || t <= 0) return 0;
  const int padded = t + 2 * plan->pad;
  if (padded < plan->n_fft) return 0;
  return 1 + (padded - plan->n_fft) / plan->hop;
}

extern "C" int hg_mel_plan_create(hg_mel_plan** out_plan, int n_fft, int num_mels, int sampling_rate,
                                  int hop_size, int win_size, double fmin, double fmax,
                                  void* stream) {
  HG_REQUIRE(out_plan, "hg_mel_plan_create: null out_plan");
  HG_REQUIRE(n_fft >= 16 && n_fft <= 4096 && n_fft % 2 == 0,
             "hg_mel_plan_create: n_fft must be even and within [16, 4096] (got %d)", n_fft);
  HG_REQUIRE(num_mels > 0 && num_mels <= 128, "hg_mel_plan_create: num_mels out of range");
  HG_REQUIRE(win_size > 0 && win_size <= n_fft, "hg_mel_plan_create: win_size must be <= n_fft");
  HG_REQUIRE(hop_size > 0 && hop_size <= n_fft, "hg_mel_plan_create: bad hop_size");
  hg_mel_plan* p = new hg_mel_plan();
  p->n_fft = n_fft; p->num_mels = num_mels; p->sampling_rate = sampling_rate;
  p->hop = hop_size; p->win = win_size; p->pad = (n_fft - hop_size) / 2;
  p->fmin = fmin;
  p->fmax = fmax < 0 ? static_cast<double>(sampling_rate / 2) : fmax;  // torchaudio: sr // 2

  // periodic Hann of win_size, centred inside n_fft like torch.stft does
  p->h_window.assign(n_fft, 0.f);
  const int left = (n_fft - win_size) / 2;
  const double two_pi = 6.283185307179586476925286766559;
  for (int i = 0; i < win_size; ++i)
    p->h_window[left + i] = static_cast<float>(0.5 - 0.5 * std::cos(two_pi * i / win_size));
  if (is_fft_size(n_fft)) {
    const int half = n_fft / 2;
    p->h_tw_half.resize(half);
    for (int m = 0; m < half; ++m)
      p->h_tw_half[m] = make_float2(static_cast<float>(std::cos(two_pi * m / half)),
                                    static_cast<float>(-std::sin(two_pi * m / half)));
    p->h_tw_full.resize(half + 1);
    for (int k = 0; k <= half; ++k)
      p->h_tw_full[k] = make_float2(static_cast<float>(std::cos(two_pi * k / n_fft)),
                                    static_cast<float>(-std::sin(two_pi * k / n_fft)));
  } else {
    p->h_tw_n.resize(n_fft);
    for (int n = 0; n < n_fft; ++n)
      p->h_tw_n[n] = make_float2(static_cast<float>(std::cos(two_pi * n / n_fft)),
                                 static_cast<float>(std::sin(two_pi * n / n_fft)));
  }

  // HTK triangles, norm=None (torchaudio.functional.melscale_fbanks), as CSR per mel bin
  const int n_freqs = n_fft / 2 + 1;
  const double nyq = static_cast<double>(sampling_rate / 2);
  const double m_min = hz_to_mel_htk(p->fmin), m_max = hz_to_mel_htk(p->fmax);
  std::vector<double> f_pts(num_mels + 2);
  for (int i = 0; i < num_mels + 2; ++i)
    f_pts[i] = mel_to_hz_htk(m_min + (m_max - m_min) * i / (num_mels + 1));
  p->h_mel_start.assign(num_mels, 0);
  p->h_mel_off.assign(num_mels + 1, 0);
  for (int m = 0; m < num_mels; ++m) {
    const double lo = f_pts[m], ce = f_pts[m + 1], hi = f_pts[m + 2];
    int first = -1, last = -2;
    std::vector<float> wts(n_freqs, 0.f);
    for (int k = 0; k < n_freqs; ++k) {
      const double f = nyq * k / (n_freqs - 1);
      const double down = (f - lo) / (ce - lo), up = (hi - f) / (hi - ce);
      const double w = std::fmax(0.0, std::fmin(down, up));
      const float wf = static_cast<float>(w);
      if (wf > 0.f) {
        if (first < 0) first = k;
        last = k;
        wts[k] = wf;
      }
    }
    if (first < 0) { first = 0; last = -1; }
    p->h_mel_start[m] = first;
    for (int k = first; k <= last; ++k) p->h_mel_w.push_back(wts[k]);
    p->h_mel_off[m + 1] = static_cast<int>(p->h_mel_w.size());
  }
  p->nnz = static_cast<int>(p->h_mel_w.size());
  if (p->h_mel_w.empty()) p->h_mel_w.push_back(0.f);

  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    // host-only plan (CPU emulation in tests); device tables stay null
    (void)cudaGetLastError();
    p->window = nullptr; p->tw_half = nullptr; p->tw_full = nullptr; p->tw_n = nullptr;
    p->mel_start = nullptr; p->mel_off = nullptr; p->mel_w = nullptr;
    *out_plan = p;
    return HG_OK;
  }
#define HG_UP(dst, src, type)                                                               \
  HG_CHECK_CUDA(cudaMalloc(&p->dst, p->src.size() * sizeof(type)));                         \
  HG_CHECK_CUDA(cudaMemcpyAsync(p->dst, p->src.data(), p->src.size() * sizeof(type),        \
                                cudaMemcpyHostToDevice, st));
  HG_UP(window, h_window, float)
  p->tw_half = nullptr; p->tw_full = nullptr; p->tw_n = nullptr;
  if (!p->h_tw_half.empty()) { HG_UP(tw_half, h_tw_half, float2) HG_UP(tw_full, h_tw_full, float2) }
  if (!p->h_tw_n.empty()) { HG_UP(tw_n, h_tw_n, float2) }
  HG_UP(mel_start, h_mel_start, int)
  HG_UP(mel_off, h_mel_off, int)
  HG_UP(mel_w, h_mel_w, float)
#undef HG_UP
  HG_CHECK_CUDA(cudaStreamSynchronize(st));
  *out_plan = p;
  return HG_OK;
}

extern "C" int hg_mel_plan_destroy(hg_mel_plan* p) {
  if (!p) return HG_OK;
  if (p->window) cudaFree(p->window);
  if (p->tw_half) cudaFree(p->tw_half);
  if (p->tw_full) cudaFree(p->tw_full);
  if (p->tw_n) cudaFree(p->tw_n);
  if (p->mel_start) cudaFree(p->mel_start);
  if (p->mel_off) cudaFree(p->mel_off);
  if (p->mel_w) cudaFree(p->mel_w);
  delete p;
  return HG_OK;
}

namespace {

// the last rFFT bin any mel filter reads: the forward un-packs and squares bins up to here only
int mel_max_bin(const hg_mel_plan* plan) {
  int max_bin = 0;
  for (int m = 0; m < plan->num_mels; ++m) {
    const int last = plan->h_mel_start[m] + (plan->h_mel_off[m + 1] - plan->h_mel_off[m]) - 1;
    if (last > max_bin) max_bin = last;
  }
  return max_bin;
}

template <int N2>
int launch_mel_kernel2(const hg_mel_plan* plan, const float* y, int batch, int t, int frames, float* out,
                       float* minmax, cudaStream_t st) {
  constexpr int kFPB = Mel2Size<N2>::kFramesPerBlock;
  Mel2Args a{};
  a.y = y; a.out = out; a.minmax = minmax;
  a.batch = batch; a.t = t; a.frames = frames; a.hop = plan->hop; a.pad = plan->pad;
  a.num_mels = plan->num_mels;
  a.window = plan->window; a.tw_half = plan->tw_half; a.tw_full = plan->tw_full;
  a.mel_start = plan->mel_start; a.mel_off = plan->mel_off; a.mel_w = plan->mel_w;
  a.nnz = plan->nnz;
  a.max_bin = mel_max_bin(plan);
  a.groups_per_item = (frames + kFPB - 1) / kFPB;
  a.total_groups = batch * a.groups_per_item;
  const size_t smem = mel2_smem_layout<N2>(plan->num_mels, plan->nnz).total;
  // two resident blocks per SM (the launch bounds and the grid below assume it)
  HG_REQUIRE(smem <= 113 * 1024, "hg_mel_fwd: %zu bytes of shared memory per block", smem);
  static hg::PerDeviceOnce once;                          // per instantiation
  if (once.need(smem))
    HG_CHECK_CUDA(cudaFuncSetAttribute(mel_kernel2<N2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int grid = a.total_groups < 2 * sms ? a.total_groups : 2 * sms;   // two resident blocks per SM, looping
  mel_kernel2<N2><<<grid, kMel2Threads, smem, st>>>(a);
  HG_CHECK_CUDA(cudaGetLastError());
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

}  // namespace

extern "C" int hg_mel_fwd(const hg_mel_plan* plan, const float* y, int batch, int t, float* out,
                          float* minmax, void* stream) {
  HG_REQUIRE(plan && y && out, "hg_mel_fwd: null pointer");
  HG_REQUIRE(plan->window, "hg_mel_fwd: plan has no device tables (created without a GPU)");
  HG_REQUIRE(batch > 0 && batch <= 65535, "hg_mel_fwd: bad batch %d", batch);
  HG_REQUIRE(t > plan->pad, "hg_mel_fwd: reflect padding %d needs more than %d samples", plan->pad, t);
  const int frames = hg_mel_num_frames(plan, t);
  HG_REQUIRE(frames > 0, "hg_mel_fwd: input too short for one frame");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (plan->n_fft) {
    case 256: return launch_mel_kernel2<4>(plan, y, batch, t, frames, out, minmax, st);
    case 512: return launch_mel_kernel2<8>(plan, y, batch, t, frames, out, minmax, st);
    case 1024: return launch_mel_kernel2<16>(plan, y, batch, t, frames, out, minmax, st);
    case 2048: return launch_mel_kernel2<32>(plan, y, batch, t, frames, out, minmax, st);
    default: break;
  }
  const size_t smem = static_cast<size_t>(plan->n_fft) * (sizeof(float2) + sizeof(float)) +
                      (plan->n_fft / 2 + 1) * sizeof(float);
  static hg::PerDeviceOnce once;
  if (once.need())
    HG_CHECK_CUDA(cudaFuncSetAttribute(mel_dft_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
  dim3 grid(frames, batch);
  mel_dft_kernel<<<grid, 256, smem, st>>>(
      y, t, frames, plan->n_fft, plan->hop, plan->pad, plan->num_mels, plan->window, plan->tw_n, plan->mel_start,
      plan->mel_off, plan->mel_w, out, minmax);
  HG_CHECK_CUDA(cudaGetLastError());
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

// ---------------------------------------------------------------------------------------------
// mel_spectrogram backward (the generated-mel L1 term of the generator loss, UPSTREAM train.py: F.l1_loss(y_mel,
// y_g_hat_mel) * 45 through src/meldataset.py:78-83).  One G-thread group per frame (G = max(32, N / 8), N = n_fft / 2),
// the Stockham FFT of fft_pass (N = 8 x 8 x R3, and x 2 at N = 1024):
//   recompute Z = FFT_N(packed windowed frame), un-pack X[0..N] (kept complex) and |X|^2, the CSR mel sums;
//   dmel = g / mel above the 1e-5 clamp (0 below), dP[k] = sum_m fb[m][k] dmel[m], G[k] = 2 dP[k] X[k];
//   the gradient at the windowed samples is S[n] = Re sum_{k=0..N} G[k] e^{+2 pi i k n / 2N}: the real inverse
//   transform of the Hermitian spectrum H (H[k] = G[k] / 2, H[0] = Re G[0], H[N] = Re G[N]), taken as ONE
//   N-point complex transform of Zc[k] = (H[k] + conj H[N-k]) + i e^{+2 pi i k / 2N} (H[k] - conj H[N-k])
//   (S[2m] + i S[2m+1] = sum_k Zc[k] e^{+2 pi i m k / N}), run through the same forward passes on conj(Zc);
//   then the window, and a scatter-add into dy with the reflect padding folded back.
// The phases are __host__ __device__ (hg_mel_bwd_emulate_host runs them with the threads serialised).
namespace {

// un-pack the real spectrum, keeping X complex: bins k = tid, tid + G, ... (0..N)
template <int N, int G>
__host__ __device__ __forceinline__ void unpack_spectrum(int tid, const cpx* __restrict__ z, cpx* __restrict__ X,
                                                         float* __restrict__ power,
                                                         const float2* __restrict__ tw_full) {
  for (int k = tid; k <= N; k += G) {
    const cpx zk = z[padi(k & (N - 1))];
    cpx zc = z[padi((N - k) & (N - 1))];
    zc.y = -zc.y;
    const cpx e = cpx{0.5f * (zk.x + zc.x), 0.5f * (zk.y + zc.y)};
    const cpx d = csub(zk, zc);
    const cpx o = cpx{0.5f * d.y, -0.5f * d.x};  // (zk - zc) / (2i)
    const float2 w = tw_full[k];
    const cpx x = cadd(e, cmul(o, cpx{w.x, w.y}));
    X[k] = x;
    power[k] = x.x * x.x + x.y * x.y;
  }
}
// dm[m] = g[m] / mel[m] above the clamp, else 0 (m = tid, tid + G, ...); also clears dP for the scatter
template <int N, int G>
__host__ __device__ __forceinline__ void mel_grad(int tid, int num_mels, const float* __restrict__ power,
                                                  const int* __restrict__ mel_start, const int* __restrict__ mel_off,
                                                  const float* __restrict__ mel_w, const float* __restrict__ g_col,
                                                  int g_stride, float* __restrict__ dm, float* __restrict__ dp) {
  for (int k = tid; k <= N; k += G) dp[k] = 0.f;
  for (int m = tid; m < num_mels; m += G) {
    const int s = mel_start[m], o = mel_off[m], n = mel_off[m + 1] - o;
    float acc = 0.f;
    for (int i = 0; i < n; ++i) acc += mel_w[o + i] * power[s + i];
    dm[m] = acc > 1e-5f ? g_col[static_cast<size_t>(m) * g_stride] / acc : 0.f;   // clamp(min=1e-5): no gradient below
  }
}
// dP[k] += fb[m][k] * dm[m]
template <int G>
__host__ __device__ __forceinline__ void mel_scatter(int tid, int num_mels, const int* __restrict__ mel_start,
                                                     const int* __restrict__ mel_off, const float* __restrict__ mel_w,
                                                     const float* __restrict__ dm, float* __restrict__ dp) {
  for (int m = tid; m < num_mels; m += G) {
    const int s = mel_start[m], o = mel_off[m], n = mel_off[m + 1] - o;
    const float d = dm[m];
    for (int i = 0; i < n; ++i) {
#ifdef __CUDA_ARCH__
      atomicAdd(dp + s + i, mel_w[o + i] * d);
#else
      dp[s + i] += mel_w[o + i] * d;
#endif
    }
  }
}
// conj(Zc)[k] for k = tid, tid + G, ... (0..N-1) into the padded FFT buffer
template <int N, int G>
__host__ __device__ __forceinline__ void build_adjoint_input(int tid, const cpx* __restrict__ X,
                                                             const float* __restrict__ dp, cpx* __restrict__ out,
                                                             const float2* __restrict__ tw_full) {
  auto hk = [&](int k) -> cpx {
    const float d = dp[k];
    if (k == 0 || k == N) return cpx{2.f * d * X[k].x, 0.f};
    return cpx{d * X[k].x, d * X[k].y};
  };
  for (int k = tid; k < N; k += G) {
    const cpx a = hk(k);
    cpx b = hk(N - k);
    b.y = -b.y;
    const cpx sum = cadd(a, b), dif = csub(a, b);
    const float2 w = tw_full[k];                      // e^{-2 pi i k / 2N}; its conjugate is needed
    const cpx rot = cmul(dif, cpx{w.x, -w.y});        // e^{+2 pi i k / 2N} (a - b)
    const cpx zc = cpx{sum.x - rot.y, sum.y + rot.x};  // sum + i * rot
    out[padi(k)] = cpx{zc.x, -zc.y};
  }
}
// samples 2m, 2m+1 of the frame's gradient from R = FFT_N(conj Zc): S[2m] = R[m].x, S[2m+1] = -R[m].y
template <int N, int G>
__host__ __device__ __forceinline__ void scatter_frame(int tid, const cpx* __restrict__ r, const float* __restrict__ window,
                                                       int frame_start, int t, float* __restrict__ dy_row) {
  for (int m = tid; m < N; m += G) {
    const cpx v = r[padi(m)];
    const float s0 = v.x * window[2 * m], s1 = -v.y * window[2 * m + 1];
    const int i0 = reflect_index(frame_start + 2 * m, t), i1 = reflect_index(frame_start + 2 * m + 1, t);
#ifdef __CUDA_ARCH__
    atomicAdd(dy_row + i0, s0);
    atomicAdd(dy_row + i1, s1);
#else
    dy_row[i0] += s0;
    dy_row[i1] += s1;
#endif
  }
}

// geometry of mel_bwd_kernel<N>: G threads per frame group (whole warps for bar.sync, at least one butterfly per
// thread in a radix-8 pass from N = 256 up), 128 threads a block; the static shared memory stays under 40 KB
// (N = 128 / 256 / 512 / 1024: 4 / 4 / 2 / 1 frames a block, 21 / 40 / 39 / 38 KB)
template <int N>
struct BwdSize {
  static constexpr int kG = N / 8 < 32 ? 32 : N / 8;
  static constexpr int kGroups = 128 / kG;
  static constexpr int kPasses = N == 1024 ? 4 : 3;
};

// the N-point transform of a frame group, ping-ponging from `in` (unused when FIRST: pass 0 reads the staged samples)
// through `other`; returns the buffer that holds the result (`other` after an odd number of passes, else `in`)
template <int N, int G, bool FIRST>
__device__ __forceinline__ cpx* group_fft(int j, int g, cpx* in, cpx* other, const float* __restrict__ samples,
                                          const float* __restrict__ window, const float2* __restrict__ tw) {
  fft_pass_group<8, N, G, FIRST>(j, 1, in, other, samples, window, tw);
  group_sync<G>(g);
  fft_pass_group<8, N, G, false>(j, 8, other, in, nullptr, nullptr, tw);
  group_sync<G>(g);
  fft_pass_group<third_radix(N), N, G, false>(j, 64, in, other, nullptr, nullptr, tw);
  group_sync<G>(g);
  if constexpr (BwdSize<N>::kPasses == 4) {
    fft_pass_group<2, N, G, false>(j, 512, other, in, nullptr, nullptr, tw);
    group_sync<G>(g);
    return in;
  }
  return other;
}
// the same passes with the G threads serialised (hg_mel_bwd_emulate_host)
template <int N, int G, bool FIRST>
cpx* host_fft(cpx* in, cpx* other, const float* samples, const float* window, const float2* tw) {
  for (int j = 0; j < G; ++j) fft_pass_group<8, N, G, FIRST>(j, 1, in, other, samples, window, tw);
  for (int j = 0; j < G; ++j) fft_pass_group<8, N, G, false>(j, 8, other, in, nullptr, nullptr, tw);
  for (int j = 0; j < G; ++j) fft_pass_group<third_radix(N), N, G, false>(j, 64, in, other, nullptr, nullptr, tw);
  if constexpr (BwdSize<N>::kPasses == 4) {
    for (int j = 0; j < G; ++j) fft_pass_group<2, N, G, false>(j, 512, other, in, nullptr, nullptr, tw);
    return in;
  }
  return other;
}

template <int N>
__global__ void __launch_bounds__(BwdSize<N>::kGroups * BwdSize<N>::kG)
mel_bwd_kernel(const float* __restrict__ y, const float* __restrict__ dmel, int t, int frames, int hop, int pad,
               int num_mels, const float* __restrict__ window, const float2* __restrict__ tw_half,
               const float2* __restrict__ tw_full, const int* __restrict__ mel_start, const int* __restrict__ mel_off,
               const float* __restrict__ mel_w, float* __restrict__ dy) {
  constexpr int G = BwdSize<N>::kG, kGroups = BwdSize<N>::kGroups;
  constexpr bool kOdd = BwdSize<N>::kPasses & 1;
  __shared__ float smp[kGroups][2 * N];
  __shared__ cpx zbuf[kGroups][2][pad_len(N)];
  __shared__ cpx xs[kGroups][N + 1];
  __shared__ float dps[kGroups][N + 1];
  __shared__ float dms[kGroups][128];
  const int g = threadIdx.x / G, j = threadIdx.x % G;
  const int f = blockIdx.x * kGroups + g, b = blockIdx.y;
  if (f >= frames) return;                          // group-uniform; the groups only meet on their own barriers
  const float* yb = y + static_cast<size_t>(b) * t;
  const int start = f * hop - pad;
  for (int n = j; n < 2 * N; n += G) smp[g][n] = yb[reflect_index(start + n, t)];
  group_sync<G>(g);
  cpx* z0 = zbuf[g][0];
  cpx* z1 = zbuf[g][1];
  cpx* zr = kOdd ? z0 : z1;                         // where the recomputed spectrum lands
  cpx* zo = kOdd ? z1 : z0;
  group_fft<N, G, true>(j, g, z1, z0, smp[g], window, tw_half);
  float* power = reinterpret_cast<float*>(zo);
  unpack_spectrum<N, G>(j, zr, xs[g], power, tw_full);
  group_sync<G>(g);
  mel_grad<N, G>(j, num_mels, power, mel_start, mel_off, mel_w,
                 dmel + static_cast<size_t>(b) * num_mels * frames + f, frames, dms[g], dps[g]);
  group_sync<G>(g);
  mel_scatter<G>(j, num_mels, mel_start, mel_off, mel_w, dms[g], dps[g]);
  group_sync<G>(g);
  build_adjoint_input<N, G>(j, xs[g], dps[g], zo, tw_full);
  group_sync<G>(g);
  const cpx* r = group_fft<N, G, false>(j, g, zo, zr, nullptr, nullptr, tw_half);
  scatter_frame<N, G>(j, r, window, start, t, dy + static_cast<size_t>(b) * t);
}

template <int N>
int launch_mel_bwd(const hg_mel_plan* plan, const float* y, const float* dmel, int batch, int t, int frames, float* dy,
                   cudaStream_t st) {
  constexpr int kGroups = BwdSize<N>::kGroups;
  dim3 grid((frames + kGroups - 1) / kGroups, batch);
  mel_bwd_kernel<N><<<grid, kGroups * BwdSize<N>::kG, 0, st>>>(
      y, dmel, t, frames, plan->hop, plan->pad, plan->num_mels, plan->window, plan->tw_half, plan->tw_full,
      plan->mel_start, plan->mel_off, plan->mel_w, dy);
  HG_CHECK_CUDA(cudaGetLastError());
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

template <int N>
void mel_bwd_emulate(const hg_mel_plan* plan, const float* host_y, const float* host_dmel, int batch, int t,
                     int frames, float* host_dy) {
  constexpr int G = BwdSize<N>::kG;
  std::vector<float> smp(2 * N), dp(N + 1), dm(128);
  std::vector<cpx> z0(pad_len(N)), z1(pad_len(N)), X(N + 1);
  const float* win = plan->h_window.data();
  const float2 *twh = plan->h_tw_half.data(), *twf = plan->h_tw_full.data();
  const int *ms = plan->h_mel_start.data(), *mo = plan->h_mel_off.data();
  const float* mw = plan->h_mel_w.data();
  for (int b = 0; b < batch; ++b)
    for (int f = 0; f < frames; ++f) {
      const int start = f * plan->hop - plan->pad;
      for (int n = 0; n < 2 * N; ++n) smp[n] = host_y[static_cast<size_t>(b) * t + reflect_index(start + n, t)];
      cpx* zr = host_fft<N, G, true>(z1.data(), z0.data(), smp.data(), win, twh);
      cpx* zo = zr == z0.data() ? z1.data() : z0.data();
      float* power = reinterpret_cast<float*>(zo);
      for (int j = 0; j < G; ++j) unpack_spectrum<N, G>(j, zr, X.data(), power, twf);
      for (int j = 0; j < G; ++j)
        mel_grad<N, G>(j, plan->num_mels, power, ms, mo, mw,
                       host_dmel + static_cast<size_t>(b) * plan->num_mels * frames + f, frames, dm.data(), dp.data());
      for (int j = 0; j < G; ++j) mel_scatter<G>(j, plan->num_mels, ms, mo, mw, dm.data(), dp.data());
      for (int j = 0; j < G; ++j) build_adjoint_input<N, G>(j, X.data(), dp.data(), zo, twf);
      const cpx* r = host_fft<N, G, false>(zo, zr, nullptr, nullptr, twh);
      for (int j = 0; j < G; ++j) scatter_frame<N, G>(j, r, win, start, t, host_dy + static_cast<size_t>(b) * t);
    }
}

// mel_kernel2<N2>'s lane phases, the 32 lanes of a warp serialised, 32 / N2 frames at a time
template <int N2>
void mel_emulate(const hg_mel_plan* plan, const float* host_y, int batch, int t, int frames, float* host_out) {
  using S = Mel2Size<N2>;
  constexpr int kFPW = S::kFramesPerWarp;
  std::vector<cpx> scratch(kWarpScratch);
  std::vector<float2> twp(S::kTwPad);
  for (int i = 0; i < S::kN; ++i) twp[padi(i)] = plan->h_tw_half[i];
  const int max_bin = mel_max_bin(plan);
  std::vector<cpx> regs(32 * 32);                  // each lane's 32 phase-2 registers
  std::vector<float> pws(32 * (N2 + 1));
  for (int b = 0; b < batch; ++b)
    for (int f0 = 0; f0 < frames; f0 += kFPW) {
      const float* yb = host_y + static_cast<size_t>(b) * t;
      for (int lane = 0; lane < 32; ++lane) {
        const int f = f0 + lane / N2;
        const int start = (f < frames ? f : frames - 1) * plan->hop - plan->pad;
        float lo = 0.f, hi = 0.f;
        mel2_phase1<N2>(lane, yb, start, t, false, plan->h_window.data(), twp.data(), scratch.data(), lo, hi);
      }
      for (int lane = 0; lane < 32; ++lane)
        mel2_phase2_read<N2>(lane, scratch.data(), *reinterpret_cast<cpx(*)[kFPW][N2]>(&regs[lane * 32]));
      for (int lane = 0; lane < 32; ++lane)
        mel2_phase2_write<N2>(lane, *reinterpret_cast<cpx(*)[kFPW][N2]>(&regs[lane * 32]), scratch.data());
      for (int h = 0; h < kFPW && f0 + h < frames; ++h) {
        for (int lane = 0; lane < 32; ++lane)
          mel2_phase3_compute<N2>(lane, scratch.data() + h * S::kN, max_bin, plan->h_tw_full.data(),
                                  *reinterpret_cast<float(*)[N2 + 1]>(&pws[lane * (N2 + 1)]));
        float* power = reinterpret_cast<float*>(scratch.data() + h * S::kN);
        for (int lane = 0; lane < 32; ++lane)
          mel2_phase3_write<N2>(lane, *reinterpret_cast<float(*)[N2 + 1]>(&pws[lane * (N2 + 1)]), power);
        float* col = host_out + static_cast<size_t>(b) * plan->num_mels * frames + f0 + h;
        for (int lane = 0; lane < 32; ++lane)
          mel2_phase4(lane, plan->num_mels, power, plan->h_mel_start.data(), plan->h_mel_off.data(),
                      plan->h_mel_w.data(), col, frames);
      }
    }
}

}  // namespace

extern "C" int hg_mel_bwd(const hg_mel_plan* plan, const float* y, const float* dmel, int batch, int t, float* dy,
                          void* stream) {
  HG_REQUIRE(plan && y && dmel && dy, "hg_mel_bwd: null pointer");
  HG_REQUIRE(plan->window, "hg_mel_bwd: plan has no device tables");
  HG_REQUIRE(is_fft_size(plan->n_fft), "hg_mel_bwd: n_fft must be 256, 512, 1024 or 2048 (got %d)", plan->n_fft);
  HG_REQUIRE(batch > 0 && batch <= 65535 && t > plan->pad && plan->num_mels <= 128, "hg_mel_bwd: bad arguments");
  const int frames = hg_mel_num_frames(plan, t);
  HG_REQUIRE(frames > 0, "hg_mel_bwd: input too short for one frame");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (plan->n_fft) {
    case 256: return launch_mel_bwd<128>(plan, y, dmel, batch, t, frames, dy, st);
    case 512: return launch_mel_bwd<256>(plan, y, dmel, batch, t, frames, dy, st);
    case 1024: return launch_mel_bwd<512>(plan, y, dmel, batch, t, frames, dy, st);
    default: return launch_mel_bwd<1024>(plan, y, dmel, batch, t, frames, dy, st);
  }
}

// Test hook: the backward kernel's phase functions on the HOST (threads serialised).  host_y fp32 [B][T],
// host_dmel fp32 [B][num_mels][frames], host_dy fp32 [B][T] is ADDED to.
extern "C" int hg_mel_bwd_emulate_host(const hg_mel_plan* plan, const float* host_y, const float* host_dmel,
                                       int batch, int t, float* host_dy) {
  HG_REQUIRE(plan && host_y && host_dmel && host_dy, "hg_mel_bwd_emulate_host: null pointer");
  HG_REQUIRE(is_fft_size(plan->n_fft), "hg_mel_bwd_emulate_host: n_fft must be 256, 512, 1024 or 2048 (got %d)",
             plan->n_fft);
  const int frames = hg_mel_num_frames(plan, t);
  HG_REQUIRE(frames > 0 && t > plan->pad, "hg_mel_bwd_emulate_host: input too short");
  switch (plan->n_fft) {
    case 256: mel_bwd_emulate<128>(plan, host_y, host_dmel, batch, t, frames, host_dy); break;
    case 512: mel_bwd_emulate<256>(plan, host_y, host_dmel, batch, t, frames, host_dy); break;
    case 1024: mel_bwd_emulate<512>(plan, host_y, host_dmel, batch, t, frames, host_dy); break;
    default: mel_bwd_emulate<1024>(plan, host_y, host_dmel, batch, t, frames, host_dy); break;
  }
  return HG_OK;
}

// ---------------------------------------------------------------------------------------------
// CPU emulation of the kernel's arithmetic (same phase functions, threads serialised).  Test-only
// entry point: lets the CPU test-suite pin the FFT / un-pack / CSR-mel logic without a GPU.
// y, out are HOST pointers here.
extern "C" int hg_mel_emulate_host(const hg_mel_plan* plan, const float* host_y, int batch, int t,
                                   float* host_out) {
  HG_REQUIRE(plan && host_y && host_out, "hg_mel_emulate_host: null pointer");
  const int frames = hg_mel_num_frames(plan, t);
  HG_REQUIRE(frames > 0 && t > plan->pad, "hg_mel_emulate_host: input too short");
  switch (plan->n_fft) {
    case 256: mel_emulate<4>(plan, host_y, batch, t, frames, host_out); return HG_OK;
    case 512: mel_emulate<8>(plan, host_y, batch, t, frames, host_out); return HG_OK;
    case 1024: mel_emulate<16>(plan, host_y, batch, t, frames, host_out); return HG_OK;
    case 2048: mel_emulate<32>(plan, host_y, batch, t, frames, host_out); return HG_OK;
    default: break;
  }
  const int n_fft = plan->n_fft, nbins = n_fft / 2 + 1;
  std::vector<float> xw(n_fft), pw(nbins);
  for (int b = 0; b < batch; ++b)
    for (int f = 0; f < frames; ++f) {
      for (int n = 0; n < n_fft; ++n)
        xw[n] = host_y[static_cast<size_t>(b) * t + reflect_index(f * plan->hop - plan->pad + n, t)] *
                plan->h_window[n];
      for (int k = 0; k < nbins; ++k) pw[k] = dft_bin_power(k, n_fft, xw.data(), plan->h_tw_n.data());
      for (int m = 0; m < plan->num_mels; ++m)
        host_out[(static_cast<size_t>(b) * plan->num_mels + m) * frames + f] =
            mel_bin_log(m, pw.data(), plan->h_mel_start.data(), plan->h_mel_off.data(), plan->h_mel_w.data());
    }
  return HG_OK;
}
