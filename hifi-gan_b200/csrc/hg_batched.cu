// hg_batched.cu — weight preparation and weight-gradient finishing, for one layer or for MANY layers in one launch.
//
// The training step re-derives every GEMM-ready filter bank after each optimizer update (weight_norm fold — the
// reference's hook recomputes w = g * v / ||v|| on every forward, src/models.py:16-31,56-59,81,86-88,96,132-140,196-204 —
// plus the bf16 packs the tcgen05 kernels read) and maps every packed weight gradient back to the parameters.  Per
// layer those are 3-4 tiny launches; a V1 step has ~80 generator convs and ~55 discriminator convs, so they were 650
// of its 1 300 launches and a fifth of its SM-time.  Here a launch covers a whole network: the host describes each
// layer once in a device-resident job table (hg_prep_job), a second table maps every block of the grid to
// (job, block-within-job), and one generic kernel dispatches on the job kind.  The job bodies below are the only
// implementation of these folds, packs and finishes: the single-layer entry points (hg_pack_conv1d_weight,
// hg_pack_disc_weight, hg_wgrad_finish_conv, ...) fill one job and launch it on its own (hg_prep_launch_one).
#include "hg_common.cuh"

#include <atomic>

#include "../../include/hifigan_b200.h"

extern std::atomic<int64_t> g_hg_launches;

namespace {

// ---- HG_JOB_GEN_CONV: one block per (padded) output channel --------------------------------------------------
// v fp32 [cout][cin][k] (+ g [cout]) -> w bf16 [k][cout_p][cin_p]; bias_out[co] = bias[co] (0 for padding rows)
__device__ void job_gen_conv(const hg_prep_job& j, int co, float* red) {
  const int cout = j.i[0], cin = j.i[1], k = j.i[2], cout_p = j.i[3], cin_p = j.i[4];
  const float* v = static_cast<const float*>(j.src0);
  const float* g = static_cast<const float*>(j.src1);
  __nv_bfloat16* out = static_cast<__nv_bfloat16*>(j.dst0);
  const bool real = co < cout;
  const float* vc = v + static_cast<size_t>(real ? co : 0) * cin * k;
  float scale = real ? 1.f : 0.f;
  if (g && real) {                                   // block-uniform branch
    float ss = 0.f;
    for (int i = threadIdx.x; i < cin * k; i += 256) ss += vc[i] * vc[i];
    ss = hg::block_sum(ss, red);
    scale = ss > 0.f ? g[co] / sqrtf(ss) : 0.f;
  }
  for (int idx = threadIdx.x; idx < k * cin_p; idx += 256) {
    const int t = idx / cin_p, ci = idx - t * cin_p;
    out[(static_cast<size_t>(t) * cout_p + co) * cin_p + ci] =
        __float2bfloat16((real && ci < cin) ? vc[ci * k + t] * scale : 0.f);
  }
  if (threadIdx.x == 0 && j.dst1) {
    const float* b = static_cast<const float*>(j.src2);
    static_cast<float*>(j.dst1)[co] = (real && b) ? b[co] : 0.f;
  }
}

// ---- HG_JOB_GEN_CONVTR: one block per (padded) input channel; polyphase scatter -----------------------------
// v fp32 [cin][cout][k] (+ g [cin]) -> w bf16 [nshift][stride*cout_p][cin_p]; bias_out[p*cout_p + co] = bias[co]
__device__ void job_gen_convtr(const hg_prep_job& j, int ci, float* red) {
  const int cin = j.i[0], cout = j.i[1], k = j.i[2], cin_p = j.i[3], cout_p = j.i[4];
  const int stride = j.i[5], padding = j.i[6], nshift = j.i[7], shift_min = j.i[8];
  const float* v = static_cast<const float*>(j.src0);
  const float* g = static_cast<const float*>(j.src1);
  __nv_bfloat16* out = static_cast<__nv_bfloat16*>(j.dst0);
  const bool real = ci < cin;
  const float* vc = v + static_cast<size_t>(real ? ci : 0) * cout * k;
  float scale = real ? 1.f : 0.f;
  if (g && real) {
    float ss = 0.f;
    for (int i = threadIdx.x; i < cout * k; i += 256) ss += vc[i] * vc[i];
    ss = hg::block_sum(ss, red);
    scale = ss > 0.f ? g[ci] / sqrtf(ss) : 0.f;
  }
  const int n_total = stride * cout_p;
  for (int idx = threadIdx.x; idx < nshift * n_total; idx += 256) {
    const int s = idx / n_total, n = idx - s * n_total;
    const int p = n / cout_p, co = n - p * cout_p;
    const int t = p + padding - (shift_min + s) * stride;
    const float w = (real && co < cout && t >= 0 && t < k) ? vc[co * k + t] * scale : 0.f;
    out[(static_cast<size_t>(s) * n_total + n) * cin_p + ci] = __float2bfloat16(w);
  }
  if (ci == 0 && j.dst1) {
    const float* b = static_cast<const float*>(j.src2);
    float* bo = static_cast<float*>(j.dst1);
    for (int n = threadIdx.x; n < n_total; n += 256) {
      const int co = n % cout_p;
      bo[n] = (b && co < cout) ? b[co] : 0.f;
    }
  }
}

// ---- HG_JOB_GEN_POST: conv_post (one output channel) folded to fp32 [cin_p][k], one block ---------------------
__device__ void job_gen_post(const hg_prep_job& j, float* red) {
  const int cin = j.i[0], k = j.i[1], cin_p = j.i[2];
  const float* v = static_cast<const float*>(j.src0);
  const float* g = static_cast<const float*>(j.src1);
  float scale = 1.f;
  if (g) {
    float ss = 0.f;
    for (int i = threadIdx.x; i < cin * k; i += 256) ss += v[i] * v[i];
    ss = hg::block_sum(ss, red);
    scale = ss > 0.f ? g[0] / sqrtf(ss) : 0.f;
  }
  float* out = static_cast<float*>(j.dst0);
  for (int i = threadIdx.x; i < cin_p * k; i += 256) out[i] = i < cin * k ? v[i] * scale : 0.f;
  if (threadIdx.x == 0 && j.dst1) static_cast<float*>(j.dst1)[0] = j.src2 ? static_cast<const float*>(j.src2)[0] : 0.f;
}

// ---- HG_JOB_DISC_ROW: one block per output channel of a discriminator conv -------------------------------
// v fp32 [cout][cin_g][k] (+ g: weight_norm fold; g == NULL: v is already the effective weight) -> eff fp32 (optional)
// and the forward bank bf16 [q][cout][cin_tile] (taps in kernel order tab[q], narrow groups merged block-diagonally)
__device__ void job_disc_row(const hg_prep_job& j, int co, float* red, float* row) {
  const int cin_g = j.i[1], k = j.i[2], merge = j.i[3], cout_g = j.i[4], cin_tile = j.i[5], cout = j.i[0];
  const int n = cin_g * k;
  const float* vr = static_cast<const float*>(j.src0) + static_cast<size_t>(co) * n;
  const float* g = static_cast<const float*>(j.src1);
  float scale = 1.f;
  if (g) {
    float ss = 0.f;
    for (int i = threadIdx.x; i < n; i += 256) ss += vr[i] * vr[i];
    ss = hg::block_sum(ss, red);
    scale = ss > 0.f ? g[co] / sqrtf(ss) : 0.f;
  }
  float* eff = static_cast<float*>(j.dst0);
  __nv_bfloat16* wf = static_cast<__nv_bfloat16*>(j.dst1);
  for (int i = threadIdx.x; i < n; i += 256) {
    const float w = vr[i] * scale;
    if (eff) eff[static_cast<size_t>(co) * n + i] = w;
    if (wf) row[i] = w;
  }
  if (!wf) return;                                   // block-uniform
  __syncthreads();
  const int lo = ((co / cout_g) % merge) * cin_g;    // this channel's slot inside the merged group tile
  const int half = cin_tile >> 1;
  for (int idx = threadIdx.x; idx < k * half; idx += 256) {
    const int q = idx / half, ct = (idx - q * half) * 2;
    const int cl = ct - lo, tap = j.tab[q];
    const float v0 = (cl >= 0 && cl < cin_g) ? row[cl * k + tap] : 0.f;
    const float v1 = (cl + 1 >= 0 && cl + 1 < cin_g) ? row[(cl + 1) * k + tap] : 0.f;
    *reinterpret_cast<uint32_t*>(wf + (static_cast<size_t>(q) * cout + co) * cin_tile + ct) = hg::pack_bf16x2(v0, v1);
  }
}

// ---- HG_JOB_TRANSPOSE_TILE: bf16 [k][n][c] -> bf16 [k][c][n], taps reversed (stride-1 data-gradient bank) ------
__device__ void job_transpose_tile(const hg_prep_job& j, int lb, float* smem) {
  const int k = j.i[0], n = j.i[1], c = j.i[2], tiles_c = j.i[3], tiles_n = j.i[4];
  const __nv_bfloat16* w = static_cast<const __nv_bfloat16*>(j.src0);
  __nv_bfloat16* out = static_cast<__nv_bfloat16*>(j.dst0);
  __nv_bfloat16(*tile)[34] = reinterpret_cast<__nv_bfloat16(*)[34]>(smem);
  const int per_tap = tiles_c * tiles_n;
  const int t = lb / per_tap, r = lb - t * per_tap;
  const int n0 = (r / tiles_c) * 32, c0 = (r % tiles_c) * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int i = ty; i < 32; i += 8)
    if (n0 + i < n && c0 + tx < c) tile[i][tx] = w[(static_cast<size_t>(t) * n + n0 + i) * c + c0 + tx];
  __syncthreads();
  for (int i = ty; i < 32; i += 8)
    if (c0 + i < c && n0 + tx < n) out[(static_cast<size_t>(k - 1 - t) * c + c0 + i) * n + n0 + tx] = tile[tx][i];
}

// ---- HG_JOB_DISC_DGRAD_TILE: effective weight fp32 [cout][cin_g][k] -> polyphase data-gradient bank
// bf16 [m][rho * cin + ci][cc]; a block owns [tci input channels of one group] x [32 dy channels] -------------
__device__ void job_disc_dgrad_tile(const hg_prep_job& j, int lb, float* sm) {
  const int cin_g = j.i[1], k = j.i[2], merge = j.i[3], cout_g = j.i[4], cin = j.i[5], stride = j.i[6], pad = j.i[7];
  const int nshift = j.i[8], shift_min = j.i[9], cout_tile = j.i[10], tci = j.i[11], grid_x = j.i[12];
  const float* w = static_cast<const float*>(j.src0);
  __nv_bfloat16* out = static_cast<__nv_bfloat16*>(j.dst0);
  const int bx = lb % grid_x, by = lb / grid_x;
  const int ci0 = bx * tci, cc0 = by * 32;
  const int g = ci0 / cin_g, cil0 = ci0 - g * cin_g;
  const int co_base = (g / merge) * cout_tile + cc0;
  const int run = tci * k, pitch = run + 1;
  for (int idx = threadIdx.x; idx < 32 * run; idx += 256) {
    const int ccl = idx / run, r = idx - ccl * run;
    const int co = co_base + ccl;
    sm[ccl * pitch + r] = (co / cout_g == g) ? w[(static_cast<size_t>(co) * cin_g + cil0) * k + r] : 0.f;
  }
  __syncthreads();
  const int planes = nshift * stride;
  for (int idx = threadIdx.x; idx < planes * tci * 16; idx += 256) {
    const int cc2 = (idx & 15) * 2;
    const int t = idx >> 4;
    const int ms = t / tci, cil = t - ms * tci;
    const int m = ms / stride, rho = ms - m * stride;
    const int tap = rho + pad - stride * (m + shift_min);
    float v0 = 0.f, v1 = 0.f;
    if (tap >= 0 && tap < k) {
      v0 = sm[cc2 * pitch + cil * k + tap];
      v1 = sm[(cc2 + 1) * pitch + cil * k + tap];
    }
    *reinterpret_cast<uint32_t*>(out + (static_cast<size_t>(ms) * cin + ci0 + cil) * cout_tile + cc0 + cc2) =
        hg::pack_bf16x2(v0, v1);
  }
}

// ---- HG_JOB_FINISH_ROW: weight gradient -> parameter gradients (unpack + weight_norm backward), one block per
// dim-0 index of the parameter.  Modes 0 / 1 gather the row from the packed layout of a conv / polyphase convtr into
// shared memory tap plane by tap plane (a conv's plane is contiguous along d1, so the reads coalesce; the transposing
// writes go to shared memory); mode 2 reads a dense [d0][d1 * k] gradient in place.  weight_norm backward (dim 0):
// dg = <dw, v> / ||v||, dv = g / ||v|| * (dw - v * <dw, v> / ||v||^2); g == NULL: plain weight, dv (+)= dw ---------
__device__ __forceinline__ float gather_packed(const float* __restrict__ p, const hg_prep_job& j, int i0, int i1, int t) {
  const int mode = j.i[0], d1 = j.i[2], rows_p = j.i[4], cin_tile = j.i[5];
  if (mode == 0) {
    const int cout_g = j.i[6], merge = j.i[7];
    const int slot = (i0 / cout_g) % merge;
    return p[(static_cast<size_t>(j.tab[t]) * rows_p + i0) * cin_tile + slot * d1 + i1];
  }
  const int stride = j.i[8], padding = j.i[9], shift_min = j.i[10], cout_p = j.i[11];
  const int ph = (((t - padding) % stride) + stride) % stride;
  const int s = (ph + padding - t) / stride - shift_min;
  return p[(static_cast<size_t>(s) * rows_p + ph * cout_p + i1) * cin_tile + i0];
}

__device__ void job_finish_row(const hg_prep_job& j, int r, float* red, float* sdw) {
  const int mode = j.i[0], d1 = j.i[2], k = j.i[3], accumulate = j.i[12];
  const int rest = d1 * k;
  const float* p = static_cast<const float*>(j.src0);
  const float* g = static_cast<const float*>(j.src1);
  const float* vr = static_cast<const float*>(j.src2) + static_cast<size_t>(r) * rest;
  float* o = static_cast<float*>(j.dst0) + static_cast<size_t>(r) * rest;
  float* dg = static_cast<float*>(j.dst1);
  const float* dw = sdw;                             // this row's gradient in parameter order [d1][k]
  if (mode == 2) {                                   // block-uniform
    dw = p + static_cast<size_t>(r) * rest;
  } else {
    for (int idx = threadIdx.x; idx < rest; idx += 256) {
      const int t = idx / d1, i1 = idx - t * d1;
      sdw[i1 * k + t] = gather_packed(p, j, r, i1, t);
    }
    __syncthreads();
  }
  if (!g) {
    for (int i = threadIdx.x; i < rest; i += 256) o[i] = accumulate ? o[i] + dw[i] : dw[i];
    return;
  }
  float ss = 0.f, dot = 0.f;
  for (int i = threadIdx.x; i < rest; i += 256) {
    const float vv = vr[i];
    ss += vv * vv;
    dot += vv * dw[i];
  }
  ss = hg::block_sum(ss, red);
  dot = hg::block_sum(dot, red);
  const float nrm = sqrtf(ss);
  const float inv = nrm > 0.f ? 1.f / nrm : 0.f;
  const float gg = g[r];
  // accumulate: rounded explicitly (the product is never fused into the add, the dg update always is), so the
  // batched and the single-job kernel, which inline this body in different contexts, give the same bits
  for (int i = threadIdx.x; i < rest; i += 256) {
    const float val = gg * inv * (dw[i] - vr[i] * dot * inv * inv);
    o[i] = accumulate ? __fadd_rn(o[i], val) : val;
  }
  if (threadIdx.x == 0) dg[r] = accumulate ? fmaf(dot, inv, dg[r]) : dot * inv;
}

// ---- HG_JOB_LOSS_SUM: one block per chunk of a reduction; *dst0 += partial sum (fp32 atomic) ------------------
// mode 0: sum |a - b| (fp32), 1: sum (c - a)^2 (fp32), 2: sum |a - b| over bf16 arrays (8 elements per 16-byte load)
__device__ void job_loss_sum(const hg_prep_job& j, int lb, float* red) {
  const int mode = j.i[0], chunk = j.i[3];
  const long long n = (static_cast<long long>(j.i[2]) << 32) | static_cast<unsigned int>(j.i[1]);
  const float c = __int_as_float(j.i[4]);
  const long long lo = static_cast<long long>(lb) * chunk;
  const long long hi = lo + chunk < n ? lo + chunk : n;
  float acc = 0.f;
  if (mode == 2) {
    const uint4* a = static_cast<const uint4*>(j.src0);
    const uint4* b = static_cast<const uint4*>(j.src1);
    for (long long i = lo + threadIdx.x; i < hi; i += 256) {
      const uint4 av = a[i], bv = b[i];
      const uint32_t aw[4] = {av.x, av.y, av.z, av.w}, bw[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        const float2 x = hg::unpack_bf16x2(aw[h]), y = hg::unpack_bf16x2(bw[h]);
        acc += fabsf(x.x - y.x) + fabsf(x.y - y.y);
      }
    }
  } else {
    const float* a = static_cast<const float*>(j.src0);
    const float* b = static_cast<const float*>(j.src1);
    for (long long i = lo + threadIdx.x; i < hi; i += 256) {
      const float d = mode == 0 ? a[i] - b[i] : c - a[i];
      acc += mode == 0 ? fabsf(d) : d * d;
    }
  }
  acc = hg::block_sum(acc, red);
  if (threadIdx.x == 0) atomicAdd(static_cast<float*>(j.dst0), acc);
}

// kKind >= 0: the kind is known at compile time and only that body is compiled in
template <int kKind = -1>
__device__ __forceinline__ void run_job(const hg_prep_job& j, int lb, float* red, float* dyn) {
  switch (kKind < 0 ? j.kind : kKind) {              // block-uniform
    case HG_JOB_GEN_CONV: job_gen_conv(j, lb, red); break;
    case HG_JOB_GEN_CONVTR: job_gen_convtr(j, lb, red); break;
    case HG_JOB_GEN_POST: job_gen_post(j, red); break;
    case HG_JOB_DISC_ROW: job_disc_row(j, lb, red, dyn); break;
    case HG_JOB_TRANSPOSE_TILE: job_transpose_tile(j, lb, dyn); break;
    case HG_JOB_DISC_DGRAD_TILE: job_disc_dgrad_tile(j, lb, dyn); break;
    case HG_JOB_FINISH_ROW: job_finish_row(j, lb, red, dyn); break;
    case HG_JOB_LOSS_SUM: job_loss_sum(j, lb, red); break;
    default: break;
  }
}

__global__ void __launch_bounds__(256)
prep_batched_kernel(const hg_prep_job* __restrict__ jobs, const int2* __restrict__ block_job) {
  extern __shared__ __align__(16) float dyn[];
  __shared__ float red[8];
  const int2 bj = block_job[blockIdx.x];
  run_job(jobs[bj.x], bj.y, red, dyn);
}

// One job of kind kKind, block b = block b of the job.  __grid_constant__: the job is read from the parameter space in
// place; a by-value parameter bound to the job bodies' const reference would be copied into a local-memory frame per
// thread.  One instantiation per kind: with every body inlined the kernel needs 40 registers (6 blocks of 256 threads
// per SM), with one body 32 (8 blocks), so a 1 024-row discriminator finish runs as one wave on 148 SMs.
template <int kKind>
__global__ void __launch_bounds__(256) prep_one_kernel(const __grid_constant__ hg_prep_job j) {
  extern __shared__ __align__(16) float dyn[];
  __shared__ float red[8];
  run_job<kKind>(j, blockIdx.x, red, dyn);
}

template <int kKind>
int launch_one(const hg_prep_job& job, int nblocks, int smem_bytes, void* stream) {
  static hg::PerDeviceOnce once;
  if (smem_bytes > 48 * 1024 && once.need(static_cast<size_t>(smem_bytes)))
    HG_CHECK_CUDA(cudaFuncSetAttribute(prep_one_kernel<kKind>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       kPrepMaxSmem));
  prep_one_kernel<kKind><<<nblocks, 256, smem_bytes, static_cast<cudaStream_t>(stream)>>>(job);
  HG_CHECK_CUDA(cudaGetLastError());
  return HG_OK;
}

}  // namespace

extern "C" int hg_prep_job_size(void) { return static_cast<int>(sizeof(hg_prep_job)); }

extern "C" int hg_prep_batched(const hg_prep_job* jobs, const int* block_job, int first_block, int nblocks,
                               int smem_bytes, void* stream) {
  HG_REQUIRE(jobs && block_job && first_block >= 0 && nblocks > 0 && smem_bytes >= 0 && smem_bytes <= kPrepMaxSmem,
             "hg_prep_batched: bad arguments");
  static hg::PerDeviceOnce once;
  if (smem_bytes > 48 * 1024 && once.need(static_cast<size_t>(smem_bytes)))
    HG_CHECK_CUDA(cudaFuncSetAttribute(prep_batched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPrepMaxSmem));
  prep_batched_kernel<<<nblocks, 256, smem_bytes, static_cast<cudaStream_t>(stream)>>>(
      jobs, reinterpret_cast<const int2*>(block_job) + first_block);
  HG_CHECK_CUDA(cudaGetLastError());
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

int hg_prep_launch_one(const hg_prep_job& job, int nblocks, int smem_bytes, void* stream) {
  int rc;
  switch (job.kind) {
    case HG_JOB_GEN_CONV: rc = launch_one<HG_JOB_GEN_CONV>(job, nblocks, smem_bytes, stream); break;
    case HG_JOB_GEN_CONVTR: rc = launch_one<HG_JOB_GEN_CONVTR>(job, nblocks, smem_bytes, stream); break;
    case HG_JOB_DISC_ROW: rc = launch_one<HG_JOB_DISC_ROW>(job, nblocks, smem_bytes, stream); break;
    case HG_JOB_TRANSPOSE_TILE: rc = launch_one<HG_JOB_TRANSPOSE_TILE>(job, nblocks, smem_bytes, stream); break;
    case HG_JOB_DISC_DGRAD_TILE: rc = launch_one<HG_JOB_DISC_DGRAD_TILE>(job, nblocks, smem_bytes, stream); break;
    case HG_JOB_FINISH_ROW: rc = launch_one<HG_JOB_FINISH_ROW>(job, nblocks, smem_bytes, stream); break;
    default: HG_REQUIRE(false, "hg_prep_launch_one: no single-job kernel for job kind %d", job.kind);
  }
  if (rc) return rc;
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}
