// hg_resblock_pair.cu — one fused ResBlock1 step on tcgen05/TMEM/TMA (sm_100a):
//
//     y = conv2(leaky_relu(conv1(leaky_relu(x)) + b1)) + b2 + x          (src/models.py:36-41)
//
// for the narrow stages (C = 32 or 64), where the two convolutions run back to back inside one
// persistent CTA and the intermediate never leaves the SM.  HBM traffic per step drops from six
// activation-sized transfers (conv1: read act, write act; conv2: read act + residual, write raw + act)
// to two (read x, write y); both leaky_relus are applied on chip.
//
// Per tile of R = 129 - k output steps (conv2, dilation 1, needs (k-1)/2 halo rows of t1 on each side,
// so conv1 produces exactly 128 rows):
//   producer warp   TMA box of 128 + (k-1)*d1 raw rows of x           -> X[slot]          (x_full)
//   transform warps in-place leaky_relu on the box (generic proxy), fence.proxy.async      (x_ready)
//                   (kActIn: x arrives already leaky_relu'd, the box is left as it is)
//   MMA thread      acc1 = sum_j X[slot][r + j*d1] * W1_j   (row-shifted descriptors)      (acc1_full)
//   E1 warps (8)    t1 = leaky_relu(acc1 + b1), zero outside [0,T), bf16 -> T1[i&1] in the swizzled
//                   K-major layout UMMA expects, fence.proxy.async                         (t1_full)
//   MMA thread      acc2 = sum_j T1[i&1][r + j] * W2_j                                     (acc2_full)
//   E2 warps (8)    y = (acc2 + b2 + x + res1 + res2) * scale -> raw / leaky_relu'd bf16 outputs
//                   (kActIn: x is rebuilt from its activated copy, hg::add_bf16x16_unlrelu)
// The MMA thread issues conv1 of tile i+1 before conv2 of tile i, and the two epilogue groups work on
// different tiles concurrently, so the tensor pipe stays busy while an intermediate is being written.  Both filter banks stay
// resident in shared memory for the whole kernel.  The residual x is re-read from global memory
// (L2-hot: the same CTA has just pulled those rows in through TMA).
#include "hg_common.cuh"

#include <atomic>

#include "../../include/hifigan_b200.h"

extern std::atomic<int64_t> g_hg_launches;

namespace {

constexpr int kM = 128;
constexpr int kXformWarps = 4;
// epilogue fan-out per role (E1 = intermediate writers, E2 = output writers): C = 64 -> 8 + 8 warps (two per
// TMEM lane quarter, half the columns each), C = 32 -> 4 + 4 (measured best, profiles/r01_pair_trace.md)
__host__ __device__ constexpr int epi_halves(int c) { return c == 64 ? 2 : 1; }
__host__ __device__ constexpr int pair_threads(int c) { return 64 + (kXformWarps + 8 * epi_halves(c)) * 32; }
constexpr int kMaxXSlots = 4;

struct PairArgs {
  int batch, t, c;
  int ktaps, dil1;
  int single;           // 1: ResBlock2 step — ONE conv: y = conv1(lrelu(x)) + b1 + x (no conv2 / intermediate)
  int subs;             // 128-row sub-tiles per pipeline item (1, 2 or 4): one barrier hand-off covers all
  int r_out;            // output rows per item = subs*128 - (k-1)
  int pad1, pad2;       // (k-1)*d1/2, (k-1)/2
  int a_rows;           // rows of x an item needs: subs*128 + (k-1)*d1
  int x_boxes, x_box_rows;  // the item's x rows arrive as x_boxes TMA boxes of x_box_rows (<= 256) rows
  int tiles_t, num_tiles;
  int x_slots;
  uint32_t x_slot_bytes, t1_slot_bytes, w_bytes;  // w_bytes: one filter bank
  const __nv_bfloat16* x;
  const float* b1;
  const float* b2;
  const __nv_bfloat16* res1;
  const __nv_bfloat16* res2;
  float scale, in_slope, out_slope;
  __nv_bfloat16* out_raw;
  __nv_bfloat16* out_act;
  // ragged batches: item b is item_len[b] * item_mul rows long; the intermediate is zero beyond that (it is conv2's
  // zero padding when the item runs alone) and the output rows up to t are stored as zeros.  NULL: all items t rows.
  const int* item_len;
  int item_mul;
  float x_inv;          // kActIn: 1 / in_slope, undoes the activation of the re-read residual
};

struct PairBarriers {
  uint64_t x_full[kMaxXSlots], x_ready[kMaxXSlots], x_empty[kMaxXSlots];
  uint64_t w_full;
  uint64_t acc1_full[2], acc1_empty[2], t1_full[2], t1_empty[2], acc2_full[2], acc2_empty[2];
  uint32_t tmem_base;
  uint32_t pad;
  __align__(16) float b1[64];
  __align__(16) float b2[64];   // biases, read back as shared-memory broadcasts by the epilogue warps
};

__device__ __forceinline__ uint32_t lrelu_bf16x2(uint32_t w, __nv_bfloat162 slope2) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&w);
  v = __hmax2(v, __hmul2(v, slope2));  // slope < 1: max(x, slope*x) == leaky_relu(x)
  return *reinterpret_cast<uint32_t*>(&v);
}

// C = channels = UMMA N = K-chunk width: 64 -> SWIZZLE_128B rows of 128 B, 32 -> SWIZZLE_64B rows of 64 B.
// kMrf = true: the general instantiation (MRF-final launches: two extra addends, scale, activated output; ragged
// batches).  kMrf = false: the plain step "one residual in, raw out, every item t rows long, scale 1" — 15 of the 18
// pair launches of a V1 forward.  The output role is the kernel's bottleneck at C = 32: compiled without the other
// paths it takes 0.86 -> 0.76 ms (k = 3) and 0.89 -> 0.75 ms (k = 7) per launch at 64 x 1024 frames.
// kActIn = true: x holds leaky_relu(x, in_slope), the only copy a stage input that also feeds unfused convs is
// stored as; false: x is raw.
template <int C, bool kSingle, bool kMrf, bool kActIn>
__global__ void __launch_bounds__(pair_threads(C), 1)
resblock_pair_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_w1,
                     const __grid_constant__ CUtensorMap tm_w2, const PairArgs p) {
  constexpr uint32_t kRowBytes = C * 2;
  constexpr uint32_t kLayout = (C == 64) ? 2u : 4u;
  constexpr uint32_t kSbo = 8 * kRowBytes;
  constexpr uint32_t kTapBytes = C * kRowBytes;
  constexpr int kChunksPerRow = kRowBytes / 16;
  constexpr int kHalves = epi_halves(C);
  constexpr int kRoleWarps = 4 * kHalves;      // warps per epilogue role
  constexpr int kThreads = pair_threads(C);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* x_buf = smem;
  uint8_t* t1_buf = x_buf + p.x_slots * p.x_slot_bytes;
  uint8_t* w1_buf = t1_buf + 2 * p.t1_slot_bytes;
  uint8_t* w2_buf = w1_buf + p.w_bytes;
  PairBarriers* bars = reinterpret_cast<PairBarriers*>(w1_buf + (kSingle ? 1 : 2) * p.w_bytes);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int S = p.subs;
  const uint32_t acc_cols = static_cast<uint32_t>(S) * C;          // one accumulator set (all sub-tiles)
  const uint32_t tmem_cols = 4 * acc_cols <= 128 ? 128u : 4 * acc_cols <= 256 ? 256u : 512u;  // acc1[2] + acc2[2]

  if (warp == 0 && lane == 0) {
    hg::tma_prefetch_desc(&tm_x);
    hg::tma_prefetch_desc(&tm_w1);
    hg::tma_prefetch_desc(&tm_w2);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int i = 0; i < kMaxXSlots; ++i) {
        hg::mbar_init(&bars->x_full[i], 1);
        hg::mbar_init(&bars->x_ready[i], kXformWarps);
        hg::mbar_init(&bars->x_empty[i], 1);
      }
      hg::mbar_init(&bars->w_full, 1);
      for (int i = 0; i < 2; ++i) {
        hg::mbar_init(&bars->acc1_full[i], 1);
        hg::mbar_init(&bars->acc1_empty[i], kRoleWarps);
        hg::mbar_init(&bars->t1_full[i], kRoleWarps);
        hg::mbar_init(&bars->t1_empty[i], 1);
        hg::mbar_init(&bars->acc2_full[i], 1);
        hg::mbar_init(&bars->acc2_empty[i], kRoleWarps);
      }
      hg::fence_mbar_init();
    }
    __syncwarp();
    hg::tmem_alloc(&bars->tmem_base, tmem_cols);
  }
  if (threadIdx.x < C) {
    bars->b1[threadIdx.x] = p.b1[threadIdx.x];
    bars->b2[threadIdx.x] = p.b2[threadIdx.x];
  }
  // zero the intermediate buffers once: rows 128.. of T1 are read by conv2's last taps (they only feed
  // discarded output rows) and must stay finite
  for (uint32_t i = threadIdx.x * 16; i < 2 * p.t1_slot_bytes; i += kThreads * 16)
    *reinterpret_cast<uint4*>(t1_buf + i) = make_uint4(0, 0, 0, 0);
  hg::fence_proxy_async_smem();
  hg::tc_fence_before();
  __syncthreads();
  hg::tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&bars->tmem_base);
  const int n_local = (p.num_tiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) /
                      static_cast<int>(gridDim.x);

  if (warp == 0) {
    // ============================ TMA producer ============================
    if (lane == 0) {
      hg::mbar_arrive_expect_tx(&bars->w_full, (kSingle ? 1 : 2) * p.w_bytes);
      hg::tma_load_3d(w1_buf, &tm_w1, &bars->w_full, 0, 0, 0);
      if (!kSingle) hg::tma_load_3d(w2_buf, &tm_w2, &bars->w_full, 0, 0, 0);
      const uint32_t box_bytes = static_cast<uint32_t>(p.x_box_rows) * kRowBytes;
      int tt = blockIdx.x % p.tiles_t, b = blockIdx.x / p.tiles_t;
      const int tt_step = gridDim.x % p.tiles_t, b_step = gridDim.x / p.tiles_t;
      uint32_t slot = 0, phase = 0;
      for (int i = 0; i < n_local; ++i) {
        hg::mbar_wait(&bars->x_empty[slot], phase ^ 1u);
        hg::mbar_arrive_expect_tx(&bars->x_full[slot], box_bytes * p.x_boxes);
        for (int bx = 0; bx < p.x_boxes; ++bx)
          hg::tma_load_3d(x_buf + slot * p.x_slot_bytes + bx * box_bytes, &tm_x, &bars->x_full[slot], 0,
                          tt * p.r_out - p.pad2 - p.pad1 + bx * p.x_box_rows, b);
        if (++slot == static_cast<uint32_t>(p.x_slots)) { slot = 0; phase ^= 1u; }
        tt += tt_step; b += b_step;
        if (tt >= p.tiles_t) { tt -= p.tiles_t; ++b; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ============================ MMA issuer ==============================
    // whole warp converged, one elected lane issues; descriptors advanced by adds on the low word
    constexpr uint32_t idesc = hg::umma_idesc_bf16(kM, C);
    constexpr uint32_t kTapLo = kTapBytes >> 4;
    const uint32_t desc_hi = hg::umma_desc_hi(kSbo, kLayout);
    const uint32_t w1_lo = hg::umma_desc_lo(hg::smem_u32(w1_buf));
    const uint32_t w2_lo = hg::umma_desc_lo(hg::smem_u32(w2_buf));
    const uint32_t x_tap_step = static_cast<uint32_t>(p.dil1) * (kRowBytes >> 4);
    hg::mbar_wait(&bars->w_full, 0);
    hg::tc_fence_after();
    auto issue = [&](uint32_t d, uint32_t a_lo, uint32_t w_lo, uint32_t a_step) {
      uint32_t accumulate = 0;
      for (int j = 0; j < p.ktaps; ++j) {
#pragma unroll
        for (int kk = 0; kk < C / 16; ++kk) {
          hg::umma_bf16_ss_lo(d, a_lo + kk * 2, w_lo + kk * 2, desc_hi, idesc, accumulate);
          accumulate = 1;
        }
        a_lo += a_step;
        w_lo += kTapLo;
      }
    };
    uint32_t x_slot = 0, x_phase = 0;   // conv1 visits items in order: ring position without divisions
    auto conv1 = [&](int i) {
      const uint32_t slot = x_slot, a = i & 1u, ph = (i >> 1) & 1u;
      hg::mbar_wait(&bars->x_ready[slot], x_phase);
      if (++x_slot == static_cast<uint32_t>(p.x_slots)) { x_slot = 0; x_phase ^= 1u; }
      hg::mbar_wait(&bars->acc1_empty[a], ph ^ 1u);
      hg::tc_fence_after();
      if (hg::elect_one()) {
        const uint32_t x_lo = hg::umma_desc_lo(hg::smem_u32(x_buf + slot * p.x_slot_bytes));
        for (int m = 0; m < S; ++m)
          issue(tmem_base + a * acc_cols + m * C, x_lo + m * (kM * (kRowBytes >> 4)), w1_lo, x_tap_step);
        hg::umma_commit(&bars->x_empty[slot]);
        hg::umma_commit(&bars->acc1_full[a]);
      }
      __syncwarp();
    };
    auto conv2 = [&](int i) {
      const uint32_t a = i & 1u, ph = (i >> 1) & 1u;
      hg::mbar_wait(&bars->t1_full[a], ph);
      hg::mbar_wait(&bars->acc2_empty[a], ph ^ 1u);
      hg::tc_fence_after();
      if (hg::elect_one()) {
        const uint32_t t_lo = hg::umma_desc_lo(hg::smem_u32(t1_buf + a * p.t1_slot_bytes));
        for (int m = 0; m < S; ++m)
          issue(tmem_base + 2 * acc_cols + a * acc_cols + m * C, t_lo + m * (kM * (kRowBytes >> 4)), w2_lo,
                kRowBytes >> 4);
        hg::umma_commit(&bars->t1_empty[a]);
        hg::umma_commit(&bars->acc2_full[a]);
      }
      __syncwarp();
    };
    if (kSingle) {
      for (int i = 0; i < n_local; ++i) conv1(i);
    } else {
      if (n_local > 0) conv1(0);
      for (int i = 0; i < n_local; ++i) {
        if (i + 1 < n_local) conv1(i + 1);
        conv2(i);
      }
    }
  } else if (warp < 2 + kXformWarps) {
    // ============================ transform: in-place leaky_relu ==========
    const int tid = (warp - 2) * 32 + lane;
    const __nv_bfloat162 slope2 = __float2bfloat162_rn(p.in_slope);
    const int n_chunks = p.a_rows * kChunksPerRow;
    uint32_t slot = 0, phase = 0;
    for (int i = 0; i < n_local; ++i) {
      hg::mbar_wait(&bars->x_full[slot], phase);
      if (!kActIn) {
        uint4* xs = reinterpret_cast<uint4*>(x_buf + slot * p.x_slot_bytes);
        for (int q = tid; q < n_chunks; q += kXformWarps * 32) {
          uint4 v = xs[q];
          v.x = lrelu_bf16x2(v.x, slope2); v.y = lrelu_bf16x2(v.y, slope2);
          v.z = lrelu_bf16x2(v.z, slope2); v.w = lrelu_bf16x2(v.w, slope2);
          xs[q] = v;
        }
        hg::fence_proxy_async_smem();
      }
      __syncwarp();
      if (lane == 0) hg::mbar_arrive(&bars->x_ready[slot]);
      if (++slot == static_cast<uint32_t>(p.x_slots)) { slot = 0; phase ^= 1u; }
    }
  } else {
    // ============================ epilogue ================================
    // Two specialised groups of 8 warps (two warps per TMEM lane quarter, half of the C columns each) so
    // the intermediate writer (E1) and the output writer (E2) of consecutive tiles run concurrently.  The
    // epilogue is instruction-issue bound per warp (clock64 traces, profiles/r01_pair_trace.md), hence the
    // wide fan-out.
    const int ew = warp - (2 + kXformWarps);
    const int quarter = warp & 3;          // TMEM lane quarter this warp may read
    const int half = (ew >> 2) % kHalves;  // which slice of the C columns this warp owns
    const int row = quarter * 32 + lane;
    const uint32_t lane_base = static_cast<uint32_t>(quarter * 32) << 16;
    constexpr int kG = C / (16 * kHalves);  // 16-column groups per warp
    const int col0 = half * (C / kHalves);

    if (ew < kRoleWarps) {
      // ---- E1: t1 = leaky_relu(acc1 + b1), zero outside [0,T)  ->  swizzled K-major smem tile
      const float* bias = bars->b1;
      const uint32_t swz = (C == 64) ? (row & 7) : ((row >> 1) & 3);
      int tt = blockIdx.x % p.tiles_t;   // time-tile index of the current item, advanced without divisions
      int bb = blockIdx.x / p.tiles_t;   // its batch item
      const int tt_step = gridDim.x % p.tiles_t, b_step = gridDim.x / p.tiles_t;
      for (int i = 0; i < (kSingle ? 0 : n_local); ++i) {
        const uint32_t a = i & 1u, ph = (i >> 1) & 1u;
        hg::mbar_wait(&bars->acc1_full[a], ph);
        hg::mbar_wait(&bars->t1_empty[a], ph ^ 1u);
        hg::tc_fence_after();
        const int t_item = (kMrf && p.item_len) ? min(p.t, __ldg(p.item_len + bb) * p.item_mul) : p.t;
        for (int m = 0; m < S; ++m) {
          const int grow = m * kM + row;                       // row of the item's t1 tile
          const int time = tt * p.r_out - p.pad2 + grow;       // its time step
          const bool inside = time >= 0 && time < t_item;
          uint8_t* trow = t1_buf + a * p.t1_slot_bytes + static_cast<uint32_t>(grow) * kRowBytes;
#pragma unroll
          for (int g = 0; g < kG; ++g) {
            uint32_t raw[16];
            hg::tmem_ld_32x16(tmem_base + lane_base + a * acc_cols + m * C + col0 + g * 16, raw);
            hg::tmem_ld_wait();
            if (g == kG - 1 && m == S - 1) {   // accumulators fully read: hand them back before the stores
              hg::tc_fence_before();
              __syncwarp();
              if (lane == 0) hg::mbar_arrive(&bars->acc1_empty[a]);
            }
            uint32_t o[8];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float4 bq = *reinterpret_cast<const float4*>(bias + col0 + g * 16 + 4 * q);
              const float v0 = hg::lrelu(__uint_as_float(raw[4 * q]) + bq.x, p.in_slope);
              const float v1 = hg::lrelu(__uint_as_float(raw[4 * q + 1]) + bq.y, p.in_slope);
              const float v2 = hg::lrelu(__uint_as_float(raw[4 * q + 2]) + bq.z, p.in_slope);
              const float v3 = hg::lrelu(__uint_as_float(raw[4 * q + 3]) + bq.w, p.in_slope);
              o[2 * q] = inside ? hg::pack_bf16x2(v0, v1) : 0u;
              o[2 * q + 1] = inside ? hg::pack_bf16x2(v2, v3) : 0u;
            }
            const uint32_t chunk = (col0 >> 3) + g * 2;  // 16-byte chunk index within the row
            *reinterpret_cast<uint4*>(trow + ((chunk ^ swz) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
            *reinterpret_cast<uint4*>(trow + (((chunk + 1) ^ swz) << 4)) = make_uint4(o[4], o[5], o[6], o[7]);
          }
        }
        hg::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) hg::mbar_arrive(&bars->t1_full[a]);
        tt += tt_step; bb += b_step;
        if (tt >= p.tiles_t) { tt -= p.tiles_t; ++bb; }
      }
    } else {
      // ---- E2: y = (acc2 + b2 + x + res1 + res2) * scale  ->  global
      // single-conv mode: this role drains conv1's accumulators directly (bias b1, no intermediate)
      const float* bias = kSingle ? bars->b1 : bars->b2;
      uint64_t* full_bar = kSingle ? bars->acc1_full : bars->acc2_full;
      uint64_t* empty_bar = kSingle ? bars->acc1_empty : bars->acc2_empty;
      const uint32_t acc_base = kSingle ? 0u : 2 * acc_cols;
      // unit = (item, sub-tile m); residual rows are fetched one unit ahead so their (L2) latency hides.
      // The (time tile, batch, sub-tile) of the NEXT unit is advanced incrementally: integer divisions per unit
      // were the single largest cost of this warp role (clock64 traces).
      int n_tt = blockIdx.x % p.tiles_t, n_b = blockIdx.x / p.tiles_t, n_m = 0;
      const int tt_step = gridDim.x % p.tiles_t, b_step = gridDim.x / p.tiles_t;
      auto next_unit_off = [&](bool& valid, bool& keep) -> size_t {
        const int grow = n_m * kM + row;
        const int time = n_tt * p.r_out + grow;
        valid = grow < p.r_out && time < p.t;
        keep = !kMrf || !p.item_len || time < __ldg(p.item_len + n_b) * p.item_mul;
        const size_t o = (static_cast<size_t>(n_b) * p.t + (valid ? time : 0)) * C + col0;
        if (++n_m == S) {
          n_m = 0;
          n_tt += tt_step; n_b += b_step;
          if (n_tt >= p.tiles_t) { n_tt -= p.tiles_t; ++n_b; }
        }
        return o;
      };
      hg::U8 rcur[kG], rnext[kG];
      bool valid = false, valid_next = false, keep = true, keep_next = true;
      size_t off = 0, off_next = 0;
      const int n_units = n_local * S;
      if (n_units > 0) {
        off_next = next_unit_off(valid_next, keep_next);
        if (valid_next) {
#pragma unroll
          for (int g = 0; g < kG; ++g) rnext[g] = hg::ldg256(p.x + off_next + g * 16);
        }
      }
      int i = 0, m = 0;
      for (int u = 0; u < n_units; ++u) {
        const uint32_t a = i & 1u, ph = (i >> 1) & 1u;
        off = off_next; valid = valid_next; keep = keep_next;
#pragma unroll
        for (int g = 0; g < kG; ++g) rcur[g] = rnext[g];
        if (u + 1 < n_units) {
          off_next = next_unit_off(valid_next, keep_next);
          if (valid_next) {
#pragma unroll
            for (int g = 0; g < kG; ++g) rnext[g] = hg::ldg256(p.x + off_next + g * 16);
          }
        }
        // MRF-final launch: the two extra addends of this unit, issued before the accumulator wait
        // (C = 64 runs 704 threads under an 80-register cap: it keeps loading them at the point of use)
        constexpr bool kPreRes = kMrf && (C == 32);
        hg::U8 r1[kPreRes ? kG : 1], r2[kPreRes ? kG : 1];
        if (kPreRes && valid && p.res1) {
#pragma unroll
          for (int g = 0; g < kG; ++g) r1[kPreRes ? g : 0] = hg::ldg256(p.res1 + off + g * 16);
        }
        if (kPreRes && valid && p.res2) {
#pragma unroll
          for (int g = 0; g < kG; ++g) r2[kPreRes ? g : 0] = hg::ldg256(p.res2 + off + g * 16);
        }
        if (m == 0) {
          hg::mbar_wait(&full_bar[a], ph);
          hg::tc_fence_after();
        }
#pragma unroll
        for (int g = 0; g < kG; ++g) {
          uint32_t raw[16];
          hg::tmem_ld_32x16(tmem_base + lane_base + acc_base + a * acc_cols + m * C + col0 + g * 16, raw);
          hg::tmem_ld_wait();
          if (g == kG - 1 && m == S - 1) {
            hg::tc_fence_before();
            __syncwarp();
            if (lane == 0) hg::mbar_arrive(&empty_bar[a]);
          }
          if (valid) {
            float v[16];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float4 bq = *reinterpret_cast<const float4*>(bias + col0 + g * 16 + 4 * q);
              v[4 * q] = __uint_as_float(raw[4 * q]) + bq.x;
              v[4 * q + 1] = __uint_as_float(raw[4 * q + 1]) + bq.y;
              v[4 * q + 2] = __uint_as_float(raw[4 * q + 2]) + bq.z;
              v[4 * q + 3] = __uint_as_float(raw[4 * q + 3]) + bq.w;
            }
            if (kActIn) hg::add_bf16x16_unlrelu(v, rcur[g], p.x_inv);
            else hg::add_bf16x16(v, rcur[g]);
            if (kMrf && p.res1) hg::add_bf16x16(v, kPreRes ? r1[kPreRes ? g : 0] : hg::ldg256(p.res1 + off + g * 16));
            if (kMrf && p.res2) hg::add_bf16x16(v, kPreRes ? r2[kPreRes ? g : 0] : hg::ldg256(p.res2 + off + g * 16));
            if (kMrf) {
              const float sc = keep ? p.scale : 0.f;                           // rows past a ragged item's end: zeros
#pragma unroll
              for (int e = 0; e < 16; ++e) v[e] *= sc;
            }
            if (p.out_raw) {
              hg::U8 o;
#pragma unroll
              for (int q = 0; q < 8; ++q) o.v[q] = hg::pack_bf16x2(v[2 * q], v[2 * q + 1]);
              hg::stg256(p.out_raw + off + g * 16, o);
            }
            if (kMrf && p.out_act) {
              hg::U8 o;
#pragma unroll
              for (int q = 0; q < 8; ++q)
                o.v[q] = hg::pack_bf16x2(hg::lrelu(v[2 * q], p.out_slope), hg::lrelu(v[2 * q + 1], p.out_slope));
              hg::stg256(p.out_act + off + g * 16, o);
            }
          }
        }
        if (++m == S) { m = 0; ++i; }
      }
    }
  }

  hg::tc_fence_before();
  __syncthreads();
  hg::tc_fence_after();
  if (warp == 1) hg::tmem_dealloc(tmem_base, tmem_cols);
}

int g_sms = 0, g_smem = 0;

template <int C, bool kSingle, bool kMrf, bool kActIn>
int launch_pair_as(const CUtensorMap& tx, const CUtensorMap& tw1, const CUtensorMap& tw2, const PairArgs& p,
                size_t smem_bytes, int grid, cudaStream_t st) {
  static hg::PerDeviceOnce once;
  if (once.need())
    HG_CHECK_CUDA(cudaFuncSetAttribute(resblock_pair_kernel<C, kSingle, kMrf, kActIn>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, g_smem));
  resblock_pair_kernel<C, kSingle, kMrf, kActIn><<<grid, pair_threads(C), smem_bytes, st>>>(tx, tw1, tw2, p);
  HG_CHECK_CUDA(cudaGetLastError());
  return HG_OK;
}

template <int C, bool kSingle>
int launch_pair(const CUtensorMap& tx, const CUtensorMap& tw1, const CUtensorMap& tw2, const PairArgs& p,
                bool act_in, size_t smem_bytes, int grid, cudaStream_t st) {
  const bool mrf = p.res1 || p.res2 || p.out_act || p.item_len || p.scale != 1.f;   // anything beyond the plain step
  if (act_in)
    return mrf ? launch_pair_as<C, kSingle, true, true>(tx, tw1, tw2, p, smem_bytes, grid, st)
               : launch_pair_as<C, kSingle, false, true>(tx, tw1, tw2, p, smem_bytes, grid, st);
  return mrf ? launch_pair_as<C, kSingle, true, false>(tx, tw1, tw2, p, smem_bytes, grid, st)
             : launch_pair_as<C, kSingle, false, false>(tx, tw1, tw2, p, smem_bytes, grid, st);
}

size_t pair_smem_bytes(int c, int ktaps, int dil1, int subs, int x_slots, int single, PairArgs* out) {
  const uint32_t row = static_cast<uint32_t>(c) * 2;
  const uint32_t a_rows = subs * kM + (ktaps - 1) * dil1;
  const uint32_t boxes = (a_rows + 255) / 256;
  const uint32_t box_rows = ((a_rows + boxes - 1) / boxes + 15) & ~15u;   // 16-row multiples keep every box
  const uint32_t x_slot = (boxes * box_rows * row + 1023u) & ~1023u;      // 1024-byte aligned in smem
  const uint32_t t1_slot = single ? 0u : ((subs * kM + ktaps - 1) * row + 1023u) & ~1023u;
  const uint32_t w_bytes = static_cast<uint32_t>(ktaps) * c * row;
  if (box_rows > 256) return ~static_cast<size_t>(0);
  if (out) {
    out->subs = subs; out->a_rows = a_rows; out->x_boxes = boxes; out->x_box_rows = box_rows;
    out->x_slot_bytes = x_slot; out->t1_slot_bytes = t1_slot; out->w_bytes = w_bytes;
  }
  return 1024 + static_cast<size_t>(x_slots) * x_slot + 2 * static_cast<size_t>(t1_slot) +
         (single ? 1 : 2) * static_cast<size_t>(w_bytes) + sizeof(PairBarriers);
}

// Largest sub-tile count whose TMEM (4*subs*C columns <= 512) and shared memory (>= 2 x slots) fit.
int pick_subs(int c, int ktaps, int dil1, int single) {
  for (int subs = 512 / (4 * c); subs >= 1; subs >>= 1)
    if (pair_smem_bytes(c, ktaps, dil1, subs, 2, single, nullptr) <= static_cast<size_t>(g_smem)) return subs;
  return 0;
}

}  // namespace

extern "C" int hg_resblock_pair_supported(int c, int ktaps, int dil1) {
  if (!(c == 32 || c == 64) || ktaps < 1 || !(ktaps & 1) || dil1 < 1) return 0;
  if (kM + (ktaps - 1) * dil1 > 256 || ktaps > 65) return 0;
  if (!g_smem) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&g_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  }
  return pick_subs(c, ktaps, dil1, 0) > 0 ? 1 : 0;
}

extern "C" int hg_resblock_single_supported(int c, int ktaps, int dil1) {
  if (!hg_resblock_pair_supported(c, 1, 1) && !g_smem) return 0;   // also initialises the device limits
  if (!(c == 32 || c == 64) || ktaps < 1 || !(ktaps & 1) || dil1 < 1 || ktaps > 65) return 0;
  return pick_subs(c, ktaps, dil1, 1) > 0 ? 1 : 0;
}

namespace {

int resblock_pair_fwd(const void* x, bool act_in, const void* w1_packed, const float* b1, const void* w2_packed,
                      const float* b2, int batch, int t, int c, int ktaps, int dil1, float in_slope, const void* res1,
                      const void* res2, float scale, void* out_raw, void* out_act, float out_slope,
                      const int* item_len, int item_mul, void* stream) {
  const int single = w2_packed == nullptr;   // ResBlock2 step: one conv + residual
  HG_REQUIRE(x && w1_packed && b1 && (single || b2), "hg_resblock_pair_fwd: null input");
  HG_REQUIRE(out_raw || out_act, "hg_resblock_pair_fwd: no output requested");
  HG_REQUIRE(batch > 0 && t > 0, "hg_resblock_pair_fwd: empty batch/time");
  HG_REQUIRE(hg_resblock_pair_supported(c, ktaps, dil1) || (single && hg_resblock_single_supported(c, ktaps, dil1)),
             "hg_resblock_pair_fwd: unsupported shape c=%d k=%d d=%d (use hg_conv1d_fwd)", c, ktaps, dil1);
  PairArgs p{};
  p.batch = batch; p.t = t; p.c = c; p.ktaps = ktaps; p.dil1 = dil1;
  const int subs = pick_subs(c, ktaps, dil1, single);
  p.single = single;
  p.r_out = single ? subs * kM : subs * kM + 1 - ktaps;
  p.pad1 = (ktaps - 1) * dil1 / 2;
  p.pad2 = single ? 0 : (ktaps - 1) / 2;
  p.tiles_t = (t + p.r_out - 1) / p.r_out;
  p.num_tiles = batch * p.tiles_t;
  int slots = kMaxXSlots;
  while (slots > 2 && pair_smem_bytes(c, ktaps, dil1, subs, slots, single, nullptr) > static_cast<size_t>(g_smem)) --slots;
  p.x_slots = slots;
  const size_t smem_bytes = pair_smem_bytes(c, ktaps, dil1, subs, slots, single, &p);
  p.x = static_cast<const __nv_bfloat16*>(x);
  p.b1 = b1; p.b2 = single ? b1 : b2;
  p.res1 = static_cast<const __nv_bfloat16*>(res1);
  p.res2 = static_cast<const __nv_bfloat16*>(res2);
  p.scale = scale; p.in_slope = in_slope; p.out_slope = out_slope;
  p.out_raw = static_cast<__nv_bfloat16*>(out_raw);
  p.out_act = static_cast<__nv_bfloat16*>(out_act);
  p.item_len = item_len; p.item_mul = item_mul > 0 ? item_mul : 1;
  p.x_inv = act_in ? 1.f / in_slope : 1.f;

  CUtensorMap tx, tw1, tw2;
  const int swz = c * 2;
  int rc = hg_encode_tmap_bf16_3d(&tx, x, c, t, batch, static_cast<uint64_t>(c) * 2,
                                  static_cast<uint64_t>(t) * c * 2, c, p.x_box_rows, 1, swz);
  if (rc) return rc;
  rc = hg_encode_tmap_bf16_3d(&tw1, w1_packed, c, c, ktaps, static_cast<uint64_t>(c) * 2,
                              static_cast<uint64_t>(c) * c * 2, c, c, ktaps, swz);
  if (rc) return rc;
  rc = hg_encode_tmap_bf16_3d(&tw2, single ? w1_packed : w2_packed, c, c, ktaps, static_cast<uint64_t>(c) * 2,
                              static_cast<uint64_t>(c) * c * 2, c, c, ktaps, swz);
  if (rc) return rc;
  const int grid = p.num_tiles < g_sms ? p.num_tiles : g_sms;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (single)
    rc = (c == 64) ? launch_pair<64, true>(tx, tw1, tw2, p, act_in, smem_bytes, grid, st)
                   : launch_pair<32, true>(tx, tw1, tw2, p, act_in, smem_bytes, grid, st);
  else
    rc = (c == 64) ? launch_pair<64, false>(tx, tw1, tw2, p, act_in, smem_bytes, grid, st)
                   : launch_pair<32, false>(tx, tw1, tw2, p, act_in, smem_bytes, grid, st);
  if (rc) return rc;
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

}  // namespace

extern "C" int hg_resblock_pair_fwd(const void* x, const void* w1_packed, const float* b1,
                                    const void* w2_packed, const float* b2, int batch, int t, int c,
                                    int ktaps, int dil1, float in_slope, const void* res1,
                                    const void* res2, float scale, void* out_raw, void* out_act,
                                    float out_slope, const int* item_len, int item_mul, void* stream) {
  return resblock_pair_fwd(x, false, w1_packed, b1, w2_packed, b2, batch, t, c, ktaps, dil1, in_slope, res1, res2,
                           scale, out_raw, out_act, out_slope, item_len, item_mul, stream);
}

extern "C" int hg_resblock_pair_fwd_actin(const void* x_act, const void* w1_packed, const float* b1,
                                          const void* w2_packed, const float* b2, int batch, int t, int c,
                                          int ktaps, int dil1, float in_slope, const void* res1,
                                          const void* res2, float scale, void* out_raw, void* out_act,
                                          float out_slope, const int* item_len, int item_mul, void* stream) {
  HG_REQUIRE(in_slope > 0.f && in_slope <= 1.f, "hg_resblock_pair_fwd_actin: slope %g not in (0, 1]", in_slope);
  return resblock_pair_fwd(x_act, true, w1_packed, b1, w2_packed, b2, batch, t, c, ktaps, dil1, in_slope, res1, res2,
                           scale, out_raw, out_act, out_slope, item_len, item_mul, stream);
}
