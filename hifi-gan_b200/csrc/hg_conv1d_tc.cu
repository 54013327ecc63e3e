// hg_conv1d_tc.cu — stride-1 dilated Conv1d as a persistent tcgen05/TMEM implicit GEMM (sm_100a).
//
// Replaces the torch Conv1d / ConvTranspose1d library calls of the reference Generator
// (src/models.py:35-42 ResBlock1, :63-68 ResBlock2, :101 conv_pre, :104 ups via polyphase packing).
//
// GEMM view, per output tile of 128 time steps x NT output channels:
//     D[t, co] = sum_{tap j} sum_{chunk c}  A_c[t + j*dil, 0:KC] * W_{j,c}[co, 0:KC]^T
// * activations are channels-last bf16 [B][T][C]; ONE TMA box of (128 + (k-1)*dil) time rows x KC
//   channels is loaded per K chunk and every tap reads it through a row-shifted UMMA descriptor, so
//   the halo is fetched once instead of k times; TMA zero-fills rows outside [0,T) which implements
//   the conv's "same" zero padding.  Row-shifting works because both TMA and UMMA apply the 128B/64B
//   swizzle as a function of the absolute shared-memory address: a start address moved by r rows
//   (r*128 B, any r) with base_offset = 0 and SBO = 8 rows addresses logical rows r..r+127 of the box.
//   Verified on B200 for SW128 and SW64, dilations 1..12, k up to 11 (profiles/r01_bringup.md).
// * weights are bf16 [k][Cout][Cin] (K-major).  When the whole filter bank of the CTA's N tile fits in
//   shared memory next to the activation ring it is loaded ONCE per CTA ("resident", every C <= 64
//   layer and C = 128, k = 3); otherwise it streams through a ring whose stages hold several taps.
// * warp 0 = TMA producer, warp 1 = MMA issuer (one thread) + TMEM owner, warps 2..9 = epilogue
//   (two warps per TMEM lane quarter, each owning half of the tile's columns).
//   Accumulators are double-buffered in TMEM so the epilogue of tile i overlaps the MMAs of tile i+1.
// * epilogue: bias, up to three residual / MRF addends, scale, raw and leaky-relu'd bf16 outputs;
//   the first residual is prefetched into registers before the accumulator wait, global accesses are
//   256-bit (one full 32-byte sector per thread per instruction).
#include "hg_common.cuh"

#include <atomic>
#include <cstdlib>

extern std::atomic<int64_t> g_hg_launches;

namespace {

constexpr int kTileM = 128;
constexpr int kEpiWarps = 8;
constexpr int kThreads = 64 + kEpiWarps * 32;
constexpr int kMaxStages = 8;
constexpr int kMaxASlots = 4;

constexpr int kMaxBoxes = 4;

struct ConvArgs {
  int batch, t, cin, cout;       // t = OUTPUT length; cin = input channels consumed per N tile
  int t_pitch;                   // rows per batch item in the output / residual tensors (>= t)
  int ktaps, dil, pad_left;
  int nchunks, a_rows;
  // Strided convs read the activations through the view [B][T_in/stride][stride*C]: output step t and tap j
  // touch input row stride*t + j - pad = stride*(t + q) + rho, i.e. view row t + q, channel block rho.  Taps
  // are grouped by residue rho into "boxes"; inside a box consecutive taps are one view row apart, so the
  // row-shifted-descriptor trick applies per box.  stride == 1: one box, taps `dil` rows apart.
  int nboxes;
  int box_col[kMaxBoxes];        // channel-coordinate offset of the box (rho * C_total)
  int box_row[kMaxBoxes];        // view-row offset of the box relative to the tile's first output step
  int box_ntaps[kMaxBoxes];      // packed taps [box_tap0, box_tap0 + ntaps) belong to this box
  int box_tap0[kMaxBoxes];
  int tap_step;                  // view rows between consecutive taps of a box
  int grouped;                   // 1: N tile nt reads input channels [nt*cin, (nt+1)*cin)
  int tiles_t, tiles_n, num_tiles;
  int a_slots;          // activation ring depth (2..4)
  int resident;         // 1: all weights of the N tile live in smem for the whole kernel
  int tps;              // ring mode: taps per stage
  int groups;           // ring mode: ceil(ktaps / tps) stages per chunk
  int stages;           // ring mode: ring depth
  uint32_t a_slot_bytes, w_stage_bytes;
  const float* bias;
  const __nv_bfloat16* res0;
  const __nv_bfloat16* res1;
  const __nv_bfloat16* res2;
  float scale;
  __nv_bfloat16* out_raw;
  __nv_bfloat16* out_act;
  float slope;
  // backward-pass epilogue terms (hg_conv1d_dgrad): v = (acc + bias + fm_coef * sgn(fm_g - fm_r)) * lrelu'(mask) + res...
  const __nv_bfloat16* mask;     // activation whose sign selects 1 / mask_slope (leaky_relu backward)
  float mask_slope;
  const __nv_bfloat16* fm_r;     // feature-matching L1 term (src/models.py:251-257): d|r - g|/dg = sgn(g - r)
  const __nv_bfloat16* fm_g;
  float fm_coef;
  int group_mod;                 // grouped: N tile nt reads input channel block (nt % group_mod)
  // "flat" sequences: many short sequences laid end to end on the time axis (pitch rows each, zero rows between
  // them standing in for the conv padding).  Output element (row t, N tile nt) is stored only when
  // (t % seq_pitch) * seq_mul + (nt * NT) / seq_div < seq_valid, so the gap rows stay zero.  seq_pitch == 0: off.
  int seq_pitch, seq_valid, seq_mul, seq_div;
  const __nv_bfloat16* pre_add;  // added to the accumulator BEFORE the mask (an incoming feature-map gradient)
  // Bias gradient of the layer whose OUTPUT this launch differentiates: fp32 column sums of the values the
  // epilogue is about to round to bf16, folded modulo colsum_mod (a polyphase gradient holds `stride` phases of
  // every channel) and added to up to three destinations (the last convs of the MRF branches share one gradient).
  float* colsum[3];
  int colsum_mod;
  // Ragged batches (length-bucketed inference): batch item b is only item_len[b] * item_mul rows long; the rows
  // between that and `t` are stored as ZEROS, so that the next layer reads exactly the zero padding it would see if
  // the item were run alone (results stay bit-identical to the per-item call).  NULL: every item is t rows long.
  const int* item_len;
  int item_mul;
  // res0 holds bf16(leaky_relu(x, slope)) and res0_inv = 1 / slope: the residual x is rebuilt in the epilogue, so a
  // tensor that feeds both a conv and a residual add is stored once, activated.  1: res0 is raw.  Forward flavours
  // (kEpi 0 and 5) only.
  float res0_inv;
};

// One 16-column group of one accumulator row: everything the epilogue does between the TMEM load and the
// global stores.  `v` leaves holding the final fp32 values (zero for rows that are not stored).
// kEpi selects what the epilogue is compiled with:
//   0  forward: bias, residuals, scale, raw / activated outputs
//   1  forward over flat sequences (the discriminators' layout): + the gap-row test
//   2  data gradient of a discriminator / generator step: + leaky_relu mask, fp32 bias-gradient sums
//   3  data gradient of the generator step through a discriminator: + mask, feature-matching sign term
//   4  everything (+ the pre-add of an incoming feature-map gradient: the autograd path)
//   5  forward with the two extra addends of an MRF-final launch (flavours 0 and 1 take one residual only)
// Flavours 0 and 5 also rebuild an activated res0 (res0_inv); the others take a raw res0.
// Carrying the warp-uniform branches of the full epilogue in every kernel cost 9 % of the inference forward
// (55.4 -> 50.4 ms at 64 x 1024 frames) and 0.4 ms of the 11.9 ms training step (profiles/r02_summary.md).
__host__ __device__ constexpr bool epi_mask(int k) { return k >= 2; }
__host__ __device__ constexpr bool epi_sums(int k) { return k == 2 || k == 4; }
__host__ __device__ constexpr bool epi_fm(int k) { return k == 3 || k == 4; }
__host__ __device__ constexpr bool epi_pre(int k) { return k == 4; }
__host__ __device__ constexpr bool epi_mrf(int k) { return k >= 2; }   // second / third addend (res1, res2)
__host__ __device__ constexpr bool epi_actres(int k) { return k == 0 || k == 5; }
template <int kEpi>
__device__ __forceinline__ void epi_group(const ConvArgs& p, bool valid, bool keep, size_t off, int ch,
                                          const uint32_t (&raw)[16], const hg::U8* r0, const hg::U8* r1,
                                          const hg::U8* r2, float (&v)[16]) {
  if (!valid) {
#pragma unroll
    for (int e = 0; e < 16; ++e) v[e] = 0.f;
    return;
  }
#pragma unroll
  for (int e = 0; e < 16; ++e) v[e] = __uint_as_float(raw[e]);
  if (p.bias) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 bq = __ldg(reinterpret_cast<const float4*>(p.bias + ch + q * 4));
      v[4 * q] += bq.x; v[4 * q + 1] += bq.y; v[4 * q + 2] += bq.z; v[4 * q + 3] += bq.w;
    }
  }
  if (epi_fm(kEpi) && p.fm_g) {
    const hg::U8 fg = hg::ldg256(p.fm_g + off), fr = hg::ldg256(p.fm_r + off);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float2 a = hg::unpack_bf16x2(fg.v[i]), r = hg::unpack_bf16x2(fr.v[i]);
      v[2 * i] += p.fm_coef * ((a.x > r.x) ? 1.f : (a.x < r.x) ? -1.f : 0.f);
      v[2 * i + 1] += p.fm_coef * ((a.y > r.y) ? 1.f : (a.y < r.y) ? -1.f : 0.f);
    }
  }
  if (epi_pre(kEpi) && p.pre_add) hg::add_bf16x16(v, hg::ldg256(p.pre_add + off));
  if (epi_mask(kEpi) && p.mask) {
    const hg::U8 mk = hg::ldg256(p.mask + off);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float2 a = hg::unpack_bf16x2(mk.v[i]);
      if (!(a.x > 0.f)) v[2 * i] *= p.mask_slope;
      if (!(a.y > 0.f)) v[2 * i + 1] *= p.mask_slope;
    }
  }
  if (p.res0) {
    if (epi_actres(kEpi)) hg::add_bf16x16_unlrelu(v, *r0, p.res0_inv);
    else hg::add_bf16x16(v, *r0);
  }
  if (epi_mrf(kEpi) && p.res1) hg::add_bf16x16(v, r1 ? *r1 : hg::ldg256(p.res1 + off));
  if (epi_mrf(kEpi) && p.res2) hg::add_bf16x16(v, r2 ? *r2 : hg::ldg256(p.res2 + off));
  const float sc = keep ? p.scale : 0.f;                               // rows past a ragged item's end: zeros
#pragma unroll
  for (int e = 0; e < 16; ++e) v[e] *= sc;
  if (p.out_raw) {
    hg::U8 o;
#pragma unroll
    for (int i = 0; i < 8; ++i) o.v[i] = hg::pack_bf16x2(v[2 * i], v[2 * i + 1]);
    hg::stg256(p.out_raw + off, o);
  }
  if (p.out_act) {
    hg::U8 o;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      o.v[i] = hg::pack_bf16x2(hg::lrelu(v[2 * i], p.slope), hg::lrelu(v[2 * i + 1], p.slope));
    hg::stg256(p.out_act + off, o);
  }
}

// Column sums of a warp's 32 rows x 16 columns (16 shuffles), added into the CTA's shared-memory partials.
__device__ __forceinline__ void epi_colsum16(float (&v)[16], int lane, float* csum) {
  int col;
  const float sum = hg::warp_colsum<16>(v, lane, col);
  if (!(lane & 1)) atomicAdd(csum + col, sum);
}

// epilogue warps only (ids 2 .. 2+kEpiWarps-1): named barrier 1
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kEpiWarps * 32) : "memory"); }

// add the CTA's column sums of N tile `nt` to the bias gradients and clear them (called by all epilogue threads)
template <int NT>
__device__ __forceinline__ void epi_colsum_flush(const ConvArgs& p, float* csum, int nt, int epi_tid) {
  epi_bar_sync();
  for (int c = epi_tid; c < NT; c += kEpiWarps * 32) {
    const float sum = csum[c];
    csum[c] = 0.f;
    const int gc = (nt * NT + c) % p.colsum_mod;
    if (sum != 0.f) {
      atomicAdd(p.colsum[0] + gc, sum);
      if (p.colsum[1]) atomicAdd(p.colsum[1] + gc, sum);
      if (p.colsum[2]) atomicAdd(p.colsum[2] + gc, sum);
    }
  }
  epi_bar_sync();
}

struct Barriers {
  uint64_t a_full[kMaxASlots];
  uint64_t a_empty[kMaxASlots];
  uint64_t w_full[kMaxStages];
  uint64_t w_empty[kMaxStages];
  uint64_t acc_full[2];
  uint64_t acc_empty[2];
  uint32_t tmem_base;
  uint32_t pad;
};

// (n tile, time tile, batch) of the CTA's current tile, advanced by gridDim.x per step with mixed-radix
// carries instead of four integer divisions per tile (those dominated the per-tile cost of every warp role).
struct TileIter {
  int nt, tt, b, tile;
  int step_n, step_t, step_b;
  int tiles_n, tiles_t;
  __device__ __forceinline__ TileIter(const ConvArgs& p) {
    tiles_n = p.tiles_n; tiles_t = p.tiles_t;
    tile = blockIdx.x;
    nt = tile % tiles_n;
    const int r = tile / tiles_n;
    tt = r % tiles_t; b = r / tiles_t;
    const int g = gridDim.x;
    step_n = g % tiles_n;
    const int gr = g / tiles_n;
    step_t = gr % tiles_t; step_b = gr / tiles_t;
  }
  __device__ __forceinline__ void next() {
    tile += gridDim.x;
    nt += step_n;
    int carry = 0;
    if (nt >= tiles_n) { nt -= tiles_n; carry = 1; }
    tt += step_t + carry;
    carry = 0;
    if (tt >= tiles_t) { tt -= tiles_t; carry = 1; }
    b += step_b + carry;
  }
};

// KC = channels per K chunk: 64 -> 128-byte rows / SWIZZLE_128B, 32 -> 64-byte rows / SWIZZLE_64B.
// NT = output channels per tile (UMMA N).
template <int KC, int NT, int kEpi>
__global__ void __launch_bounds__(kThreads, 1)
conv1d_tc_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_w,
                 const ConvArgs p) {
  constexpr uint32_t kRowBytes = KC * 2;
  constexpr uint32_t kLayout = (KC == 64) ? 2u : 4u;  // UMMA layout type: SW128 / SW64
  constexpr uint32_t kSbo = 8 * kRowBytes;
  constexpr uint32_t kTapBytes = NT * kRowBytes;      // one (tap, chunk) weight block
  constexpr uint32_t kTmemCols = (2 * NT <= 32) ? 32u : (2 * NT <= 64) ? 64u
                                 : (2 * NT <= 128) ? 128u : (2 * NT <= 256) ? 256u : 512u;
  constexpr int kColsPerWarp = NT / 2;                // each epilogue warp owns half of the columns
  constexpr int kGroups16 = kColsPerWarp / 16;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* a_buf = smem;
  uint8_t* w_buf = smem + p.a_slots * p.a_slot_bytes;
  const uint32_t w_total = p.resident ? static_cast<uint32_t>(p.nchunks * p.ktaps) * kTapBytes
                                      : static_cast<uint32_t>(p.stages) * p.w_stage_bytes;
  Barriers* bars = reinterpret_cast<Barriers*>(w_buf + w_total);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    hg::tma_prefetch_desc(&tm_x);
    hg::tma_prefetch_desc(&tm_w);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int i = 0; i < kMaxASlots; ++i) {
        hg::mbar_init(&bars->a_full[i], 1);
        hg::mbar_init(&bars->a_empty[i], 1);
      }
      for (int i = 0; i < 2; ++i) {
        hg::mbar_init(&bars->acc_full[i], 1);
        hg::mbar_init(&bars->acc_empty[i], kEpiWarps);
      }
      for (int i = 0; i < kMaxStages; ++i) {
        hg::mbar_init(&bars->w_full[i], 1);
        hg::mbar_init(&bars->w_empty[i], 1);
      }
      hg::fence_mbar_init();
    }
    __syncwarp();
    hg::tmem_alloc(&bars->tmem_base, kTmemCols);
  }
  hg::tc_fence_before();
  __syncthreads();
  hg::tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&bars->tmem_base);

  if (warp == 0) {
    // ============================ TMA producer ============================
    if (lane == 0) {
      uint32_t a_slot = 0, a_phase = 0, w_slot = 0, w_phase = 0;   // ring positions, no divisions
      const uint32_t a_bytes = static_cast<uint32_t>(p.a_rows) * kRowBytes;
      if (p.resident) {
        // whole filter bank once: per chunk one box (KC, NT, ktaps) -> [tap][NT rows][KC] in smem
        hg::mbar_arrive_expect_tx(&bars->w_full[0], w_total);
        for (int c = 0; c < p.nchunks; ++c)
          hg::tma_load_3d(w_buf + static_cast<uint32_t>(c * p.ktaps) * kTapBytes, &tm_w,
                          &bars->w_full[0], c * KC, 0, 0);
      }
      for (TileIter it(p); it.tile < p.num_tiles; it.next()) {
        const int nt = it.nt, b = it.b;
        const int t0 = it.tt * kTileM;
        const int chan0 = p.grouped ? (nt % p.group_mod) * p.cin : 0;
        for (int c = 0; c < p.nchunks; ++c) {
          int in_stage = 0;   // position of the next packed tap inside its weight stage (no modulo per tap)
          for (int bx = 0; bx < p.nboxes; ++bx) {
            const uint32_t slot = a_slot;
            hg::mbar_wait(&bars->a_empty[slot], a_phase ^ 1u);
            hg::mbar_arrive_expect_tx(&bars->a_full[slot], a_bytes);
            hg::tma_load_3d(a_buf + slot * p.a_slot_bytes, &tm_x, &bars->a_full[slot],
                            p.box_col[bx] + chan0 + c * KC, t0 + p.box_row[bx], b);
            if (++a_slot == static_cast<uint32_t>(p.a_slots)) { a_slot = 0; a_phase ^= 1u; }
            if (!p.resident) {
              // weight stages are issued in the order the MMA warp consumes packed taps
              const int q_end = p.box_tap0[bx] + p.box_ntaps[bx];
              for (int q = p.box_tap0[bx]; q < q_end; ++q) {
                const bool first_of_stage = in_stage == 0;
                if (++in_stage == p.tps) in_stage = 0;
                if (!first_of_stage) continue;
                const uint32_t s = w_slot;
                hg::mbar_wait(&bars->w_empty[s], w_phase ^ 1u);
                hg::mbar_arrive_expect_tx(&bars->w_full[s], static_cast<uint32_t>(p.tps) * kTapBytes);
                hg::tma_load_3d(w_buf + s * p.w_stage_bytes, &tm_w, &bars->w_full[s], c * KC, nt * NT, q);
                if (++w_slot == static_cast<uint32_t>(p.stages)) { w_slot = 0; w_phase ^= 1u; }
              }
            }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ============================ MMA issuer ==============================
    // The whole warp walks the loop converged (so addresses stay in uniform registers); one elected
    // lane issues.  Descriptors: constant high word, low word advanced by plain adds.
    constexpr uint32_t idesc = hg::umma_idesc_bf16(kTileM, NT);
    constexpr uint32_t kTapLo = kTapBytes >> 4;
    const uint32_t desc_hi = hg::umma_desc_hi(kSbo, kLayout);
    const uint32_t a_tap_step = static_cast<uint32_t>(p.tap_step) * (kRowBytes >> 4);
    const uint32_t w_lo0 = hg::umma_desc_lo(hg::smem_u32(w_buf));
    uint32_t acc_it = 0;
    uint32_t a_slot = 0, a_phase = 0;
    uint32_t w_slot = 0, w_phase = 0;   // weight-ring position, advanced without divisions
    if (p.resident) {
      hg::mbar_wait(&bars->w_full[0], 0);
      hg::tc_fence_after();
    }
    const bool leader = hg::elect_one();
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const uint32_t acc = acc_it & 1u;
      hg::mbar_wait(&bars->acc_empty[acc], ((acc_it >> 1) & 1u) ^ 1u);
      hg::tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * NT;
      uint32_t accumulate = 0;
      for (int c = 0; c < p.nchunks; ++c) {
        int in_stage = 0;     // position of the current packed tap inside its weight stage
        uint32_t w_stage_lo = 0;
        for (int bx = 0; bx < p.nboxes; ++bx) {
          const uint32_t slot = a_slot;
          hg::mbar_wait(&bars->a_full[slot], a_phase);
          hg::tc_fence_after();
          uint32_t a_lo = hg::umma_desc_lo(hg::smem_u32(a_buf + slot * p.a_slot_bytes));
          const int q0 = p.box_tap0[bx], q_end = q0 + p.box_ntaps[bx];
          if (p.resident) {
            if (leader) {
              uint32_t w_lo = w_lo0 + static_cast<uint32_t>(c * p.ktaps + q0) * kTapLo;
              uint32_t acc_flag = accumulate;
              for (int q = q0; q < q_end; ++q) {
#pragma unroll
                for (int kk = 0; kk < KC / 16; ++kk) {
                  hg::umma_bf16_ss_lo(d_tmem, a_lo + kk * 2, w_lo + kk * 2, desc_hi, idesc, acc_flag);
                  acc_flag = 1;
                }
                a_lo += a_tap_step;
                w_lo += kTapLo;
              }
            }
            accumulate = 1;
          } else {
            for (int q = q0; q < q_end; ++q) {
              if (in_stage == 0) {
                hg::mbar_wait(&bars->w_full[w_slot], w_phase);
                hg::tc_fence_after();
                w_stage_lo = w_lo0 + ((w_slot * p.w_stage_bytes) >> 4);
              }
              const bool stage_done = (in_stage == p.tps - 1) || (q == p.ktaps - 1);
              if (leader) {
#pragma unroll
                for (int kk = 0; kk < KC / 16; ++kk) {
                  hg::umma_bf16_ss_lo(d_tmem, a_lo + kk * 2, w_stage_lo + kk * 2, desc_hi, idesc, accumulate);
                  accumulate = 1;
                }
                if (stage_done) hg::umma_commit(&bars->w_empty[w_slot]);
              }
              accumulate = 1;
              a_lo += a_tap_step;
              w_stage_lo += kTapLo;
              if (stage_done) {
                in_stage = 0;
                if (++w_slot == static_cast<uint32_t>(p.stages)) { w_slot = 0; w_phase ^= 1u; }
              } else {
                ++in_stage;
              }
            }
          }
          if (leader) hg::umma_commit(&bars->a_empty[slot]);
          __syncwarp();
          if (++a_slot == static_cast<uint32_t>(p.a_slots)) { a_slot = 0; a_phase ^= 1u; }
        }
      }
      if (leader) hg::umma_commit(&bars->acc_full[acc]);
      __syncwarp();
      ++acc_it;
    }
  } else {
    // ============================ epilogue ================================
    const int ew = warp - 2;
    const int quarter = warp & 3;          // TMEM lane quarter this warp may read
    const int half = ew >> 2;              // which half of the tile's columns
    const int row = quarter * 32 + lane;
    const int col0 = half * kColsPerWarp;  // first column (within the tile) owned by this warp
    uint32_t acc_it = 0;
    // bias-gradient column sums: per-CTA fp32 partials in shared memory, flushed when the N tile changes
    float* csum = reinterpret_cast<float*>(bars + 1);
    const int epi_tid = threadIdx.x - 64;
    int cs_nt = -1;
    if (epi_sums(kEpi) && p.colsum[0]) {
      for (int c = epi_tid; c < NT; c += kEpiWarps * 32) csum[c] = 0.f;
      epi_bar_sync();
    }
    for (TileIter it(p); it.tile < p.num_tiles; it.next()) {
      const int nt = it.nt, b = it.b;
      if (epi_sums(kEpi) && p.colsum[0] && nt != cs_nt) {
        if (cs_nt >= 0) epi_colsum_flush<NT>(p, csum, cs_nt, epi_tid);
        cs_nt = nt;
      }
      const int t = it.tt * kTileM + row;
      bool valid = t < p.t;
      if (kEpi >= 1 && p.seq_pitch) valid = valid && ((t % p.seq_pitch) * p.seq_mul + (nt * NT) / p.seq_div < p.seq_valid);
      const bool keep = !p.item_len || t < __ldg(p.item_len + b) * p.item_mul;
      const int ch0 = nt * NT + col0;
      const size_t off = (static_cast<size_t>(b) * p.t_pitch + (valid ? t : 0)) * p.cout + ch0;
      // residual prefetch: issued before the accumulator wait so its latency hides under the MMAs
      hg::U8 rpre[kGroups16];
      if (p.res0 && valid) {
#pragma unroll
        for (int g = 0; g < kGroups16; ++g) rpre[g] = hg::ldg256(p.res0 + off + g * 16);
      }
      // the MRF-final launch adds two more tensors: fetch them up front as well when the registers allow
      // (loading them at the point of use exposed their latency: +0.3 .. +1.2 ms on those launches)
      constexpr bool kPreAll = kGroups16 <= 4;
      hg::U8 rpre1[kPreAll ? kGroups16 : 1], rpre2[kPreAll ? kGroups16 : 1];
      if (epi_mrf(kEpi) && kPreAll && valid) {
        if (p.res1) {
#pragma unroll
          for (int g = 0; g < kGroups16; ++g) rpre1[kPreAll ? g : 0] = hg::ldg256(p.res1 + off + g * 16);
        }
        if (p.res2) {
#pragma unroll
          for (int g = 0; g < kGroups16; ++g) rpre2[kPreAll ? g : 0] = hg::ldg256(p.res2 + off + g * 16);
        }
      }
      const uint32_t acc = acc_it & 1u;
      hg::mbar_wait(&bars->acc_full[acc], (acc_it >> 1) & 1u);
      hg::tc_fence_after();
#pragma unroll
      for (int g = 0; g < kGroups16; ++g) {
        uint32_t raw[16];
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * NT +
                               col0 + g * 16;
        hg::tmem_ld_32x16(taddr, raw);
        hg::tmem_ld_wait();
        float v[16];
        epi_group<kEpi>(p, valid, keep, off + g * 16, ch0 + g * 16, raw, &rpre[g], kPreAll ? &rpre1[kPreAll ? g : 0] : nullptr,
                  kPreAll ? &rpre2[kPreAll ? g : 0] : nullptr, v);
        if (epi_sums(kEpi) && p.colsum[0]) epi_colsum16(v, lane, csum + col0 + g * 16);
      }
      hg::tc_fence_before();
      __syncwarp();
      if (lane == 0) hg::mbar_arrive(&bars->acc_empty[acc]);
      ++acc_it;
    }
    if (epi_sums(kEpi) && p.colsum[0] && cs_nt >= 0) epi_colsum_flush<NT>(p, csum, cs_nt, epi_tid);
  }

  hg::tc_fence_before();
  __syncthreads();
  hg::tc_fence_after();
  if (warp == 1) hg::tmem_dealloc(tmem_base, kTmemCols);
}

// ==================================================================================================
// CTA-pair variant (cta_group::2): one 256-row x NT tile per pair.  Each CTA loads the activation box
// of its own 128 rows and HALF of every weight stage (NT/2 filter rows); the leader issues M = 256
// MMAs that read both CTAs' shared memory, so per CTA an MMA costs 4 KB (A) + NT*16 B (half of B) of
// shared-memory bandwidth instead of 4 KB + NT*32 B, and the weight fill traffic per CTA halves too.
// Used for the dense stride-1 layers whose filter bank does not fit in shared memory (NT >= 128).
// ==================================================================================================
struct Barriers2 {
  uint64_t a_full[kMaxASlots];     // leader's copy is the live one (count 2: leader arm + peer arrive)
  uint64_t a_empty[kMaxASlots];    // per CTA, released by the leader's multicast commit
  uint64_t w_full[kMaxStages];
  uint64_t w_empty[kMaxStages];
  uint64_t acc_full[2];            // per CTA (multicast commit)
  uint64_t acc_empty[2];           // leader's copy, count 2 * kEpiWarps (both CTAs' epilogue warps)
  uint32_t tmem_base;
  uint32_t pad;
};

template <int NT, int kEpi>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
conv1d_tc2_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_w,
                  const ConvArgs p) {
  constexpr int KC = 64;
  constexpr uint32_t kRowBytes = KC * 2;
  constexpr uint32_t kLayout = 2u;
  constexpr uint32_t kSbo = 8 * kRowBytes;
  constexpr uint32_t kTapBytes = (NT / 2) * kRowBytes;   // per CTA: half of the filter rows of one tap
  constexpr uint32_t kTmemCols = (2 * NT <= 256) ? 256u : 512u;
  constexpr int kColsPerWarp = NT / 2;
  constexpr int kGroups16 = kColsPerWarp / 16;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* a_buf = smem;
  uint8_t* w_buf = smem + p.a_slots * p.a_slot_bytes;
  Barriers2* bars = reinterpret_cast<Barriers2*>(w_buf + static_cast<uint32_t>(p.stages) * p.w_stage_bytes);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = hg::cluster_ctarank();       // 0 = leader (issues the MMAs)
  const int n_clusters = gridDim.x >> 1;
  const int cluster_id = blockIdx.x >> 1;
  // pair tiles: (n tile, pair of time tiles, batch)
  const int tiles_pt = (p.tiles_t + 1) >> 1;
  const int num_pt = p.batch * tiles_pt * p.tiles_n;

  if (warp == 0 && lane == 0) {
    hg::tma_prefetch_desc(&tm_x);
    hg::tma_prefetch_desc(&tm_w);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int i = 0; i < kMaxASlots; ++i) {
        hg::mbar_init(&bars->a_full[i], 2);
        hg::mbar_init(&bars->a_empty[i], 1);
      }
      for (int i = 0; i < 2; ++i) {
        hg::mbar_init(&bars->acc_full[i], 1);
        hg::mbar_init(&bars->acc_empty[i], 2 * kEpiWarps);
      }
      for (int i = 0; i < kMaxStages; ++i) {
        hg::mbar_init(&bars->w_full[i], 2);
        hg::mbar_init(&bars->w_empty[i], 1);
      }
      hg::fence_mbar_init();
    }
    __syncwarp();
    hg::tmem_alloc_2sm(&bars->tmem_base, kTmemCols);
  }
  hg::tc_fence_before();
  __syncthreads();
  hg::cluster_sync_all();     // the peer's barriers must exist before anything is signalled across the pair
  hg::tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&bars->tmem_base);

  // incremental decode of the cluster's pair tiles
  auto decode = [&](int pt, int& nt, int& ptt, int& b) {
    nt = pt % p.tiles_n;
    const int r = pt / p.tiles_n;
    ptt = r % tiles_pt;
    b = r / tiles_pt;
  };

  if (warp == 0) {
    // ============================ TMA producer (both CTAs) ================
    if (lane == 0) {
      uint32_t a_slot = 0, a_phase = 0, w_slot = 0, w_phase = 0;
      const uint32_t a_bytes = static_cast<uint32_t>(p.a_rows) * kRowBytes;
      const uint32_t w_bytes = static_cast<uint32_t>(p.tps) * kTapBytes;
      for (int pt = cluster_id; pt < num_pt; pt += n_clusters) {
        int nt, ptt, b;
        decode(pt, nt, ptt, b);
        const int t0 = (2 * ptt + static_cast<int>(rank)) * kTileM - p.pad_left;
        for (int c = 0; c < p.nchunks; ++c) {
          hg::mbar_wait(&bars->a_empty[a_slot], a_phase ^ 1u);
          if (rank == 0) hg::mbar_arrive_expect_tx(&bars->a_full[a_slot], 2 * a_bytes);
          else hg::mbar_arrive_remote(&bars->a_full[a_slot], 0);
          hg::tma_load_3d_2sm(a_buf + a_slot * p.a_slot_bytes, &tm_x, &bars->a_full[a_slot], c * KC, t0, b);
          if (++a_slot == static_cast<uint32_t>(p.a_slots)) { a_slot = 0; a_phase ^= 1u; }
          for (int g = 0; g < p.groups; ++g) {
            hg::mbar_wait(&bars->w_empty[w_slot], w_phase ^ 1u);
            if (rank == 0) hg::mbar_arrive_expect_tx(&bars->w_full[w_slot], 2 * w_bytes);
            else hg::mbar_arrive_remote(&bars->w_full[w_slot], 0);
            hg::tma_load_3d_2sm(w_buf + w_slot * p.w_stage_bytes, &tm_w, &bars->w_full[w_slot], c * KC,
                                nt * NT + static_cast<int>(rank) * (NT / 2), g * p.tps);
            if (++w_slot == static_cast<uint32_t>(p.stages)) { w_slot = 0; w_phase ^= 1u; }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ============================ MMA issuer (leader CTA only) ============
    if (rank == 0) {
      constexpr uint32_t idesc = hg::umma_idesc_bf16(2 * kTileM, NT);
      constexpr uint32_t kTapLo = kTapBytes >> 4;
      const uint32_t desc_hi = hg::umma_desc_hi(kSbo, kLayout);
      const uint32_t a_tap_step = static_cast<uint32_t>(p.tap_step) * (kRowBytes >> 4);
      const uint32_t w_lo0 = hg::umma_desc_lo(hg::smem_u32(w_buf));
      const bool leader = hg::elect_one();
      uint32_t acc_it = 0, a_slot = 0, a_phase = 0, w_slot = 0, w_phase = 0;
      for (int pt = cluster_id; pt < num_pt; pt += n_clusters) {
        const uint32_t acc = acc_it & 1u;
        hg::mbar_wait(&bars->acc_empty[acc], ((acc_it >> 1) & 1u) ^ 1u);
        hg::tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * NT;
        uint32_t accumulate = 0;
        for (int c = 0; c < p.nchunks; ++c) {
          hg::mbar_wait(&bars->a_full[a_slot], a_phase);
          hg::tc_fence_after();
          uint32_t a_lo = hg::umma_desc_lo(hg::smem_u32(a_buf + a_slot * p.a_slot_bytes));
          int q = 0;
          for (int g = 0; g < p.groups; ++g) {
            hg::mbar_wait(&bars->w_full[w_slot], w_phase);
            hg::tc_fence_after();
            if (leader) {
              uint32_t w_lo = w_lo0 + ((w_slot * p.w_stage_bytes) >> 4);
              const int q_end = min(p.ktaps, q + p.tps);
              for (int j = q; j < q_end; ++j) {
#pragma unroll
                for (int kk = 0; kk < KC / 16; ++kk) {
                  hg::umma_bf16_ss_lo_2sm(d_tmem, a_lo + kk * 2, w_lo + kk * 2, desc_hi, idesc, accumulate);
                  accumulate = 1;
                }
                a_lo += a_tap_step;
                w_lo += kTapLo;
              }
              hg::umma_commit_2sm(&bars->w_empty[w_slot]);
            } else {
              a_lo += a_tap_step * static_cast<uint32_t>(min(p.ktaps, q + p.tps) - q);
            }
            accumulate = 1;
            q += p.tps;
            __syncwarp();
            if (++w_slot == static_cast<uint32_t>(p.stages)) { w_slot = 0; w_phase ^= 1u; }
          }
          if (leader) hg::umma_commit_2sm(&bars->a_empty[a_slot]);
          __syncwarp();
          if (++a_slot == static_cast<uint32_t>(p.a_slots)) { a_slot = 0; a_phase ^= 1u; }
        }
        if (leader) hg::umma_commit_2sm(&bars->acc_full[acc]);
        __syncwarp();
        ++acc_it;
      }
    }
  } else {
    // ============================ epilogue (both CTAs, own 128 rows) ======
    const int ew = warp - 2;
    const int quarter = warp & 3;
    const int half = ew >> 2;
    const int row = quarter * 32 + lane;
    const int col0 = half * kColsPerWarp;
    uint32_t acc_it = 0;
    float* csum = reinterpret_cast<float*>(bars + 1);
    const int epi_tid = threadIdx.x - 64;
    int cs_nt = -1;
    if (epi_sums(kEpi) && p.colsum[0]) {
      for (int c = epi_tid; c < NT; c += kEpiWarps * 32) csum[c] = 0.f;
      epi_bar_sync();
    }
    for (int pt = cluster_id; pt < num_pt; pt += n_clusters) {
      int nt, ptt, b;
      decode(pt, nt, ptt, b);
      if (epi_sums(kEpi) && p.colsum[0] && nt != cs_nt) {
        if (cs_nt >= 0) epi_colsum_flush<NT>(p, csum, cs_nt, epi_tid);
        cs_nt = nt;
      }
      const int t = (2 * ptt + static_cast<int>(rank)) * kTileM + row;
      bool valid = t < p.t;
      if (kEpi >= 1 && p.seq_pitch) valid = valid && ((t % p.seq_pitch) * p.seq_mul + (nt * NT) / p.seq_div < p.seq_valid);
      const bool keep = !p.item_len || t < __ldg(p.item_len + b) * p.item_mul;
      const int ch0 = nt * NT + col0;
      const size_t off = (static_cast<size_t>(b) * p.t_pitch + (valid ? t : 0)) * p.cout + ch0;
      hg::U8 rpre[kGroups16];
      if (p.res0 && valid) {
#pragma unroll
        for (int g = 0; g < kGroups16; ++g) rpre[g] = hg::ldg256(p.res0 + off + g * 16);
      }
      constexpr bool kPreAll = kGroups16 <= 4;
      hg::U8 rpre1[kPreAll ? kGroups16 : 1], rpre2[kPreAll ? kGroups16 : 1];
      if (epi_mrf(kEpi) && kPreAll && valid) {
        if (p.res1) {
#pragma unroll
          for (int g = 0; g < kGroups16; ++g) rpre1[kPreAll ? g : 0] = hg::ldg256(p.res1 + off + g * 16);
        }
        if (p.res2) {
#pragma unroll
          for (int g = 0; g < kGroups16; ++g) rpre2[kPreAll ? g : 0] = hg::ldg256(p.res2 + off + g * 16);
        }
      }
      const uint32_t acc = acc_it & 1u;
      hg::mbar_wait(&bars->acc_full[acc], (acc_it >> 1) & 1u);
      hg::tc_fence_after();
#pragma unroll
      for (int g = 0; g < kGroups16; ++g) {
        uint32_t raw[16];
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * NT + col0 + g * 16;
        hg::tmem_ld_32x16(taddr, raw);
        hg::tmem_ld_wait();
        float v[16];
        epi_group<kEpi>(p, valid, keep, off + g * 16, ch0 + g * 16, raw, &rpre[g], kPreAll ? &rpre1[kPreAll ? g : 0] : nullptr,
                  kPreAll ? &rpre2[kPreAll ? g : 0] : nullptr, v);
        if (epi_sums(kEpi) && p.colsum[0]) epi_colsum16(v, lane, csum + col0 + g * 16);
      }
      hg::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (rank == 0) hg::mbar_arrive(&bars->acc_empty[acc]);
        else hg::mbar_arrive_remote(&bars->acc_empty[acc], 0);
      }
      ++acc_it;
    }
    if (epi_sums(kEpi) && p.colsum[0] && cs_nt >= 0) epi_colsum_flush<NT>(p, csum, cs_nt, epi_tid);
  }

  hg::tc_fence_before();
  __syncthreads();
  hg::cluster_sync_all();     // nobody leaves (or frees TMEM) while the peer may still signal / read
  hg::tc_fence_after();
  if (warp == 1) hg::tmem_dealloc_2sm(tmem_base, kTmemCols);
}

int g_num_sms = 0;
int g_max_smem = 0;

int device_props() {
  if (g_num_sms) return HG_OK;
  int dev = 0;
  HG_CHECK_CUDA(cudaGetDevice(&dev));
  HG_CHECK_CUDA(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
  HG_CHECK_CUDA(cudaDeviceGetAttribute(&g_max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  return HG_OK;
}

template <int KC, int NT, int kEpi>
int launch_as(const CUtensorMap& tm_x, const CUtensorMap& tm_w, const ConvArgs& p, size_t smem_bytes,
              int grid, cudaStream_t st) {
  static hg::PerDeviceOnce once;  // per instantiation
  if (once.need())
    HG_CHECK_CUDA(cudaFuncSetAttribute(conv1d_tc_kernel<KC, NT, kEpi>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, g_max_smem));
  conv1d_tc_kernel<KC, NT, kEpi><<<grid, kThreads, smem_bytes, st>>>(tm_x, tm_w, p);
  HG_CHECK_CUDA(cudaGetLastError());
  return HG_OK;
}

// the cheapest epilogue flavour that serves this launch
int epi_flavour(const ConvArgs& p) {
  if (p.pre_add || (p.fm_g && p.colsum[0])) return 4;
  if (p.fm_g) return 3;
  if (p.mask || p.colsum[0]) return 2;
  if (p.res1 || p.res2) return 5;
  return p.seq_pitch ? 1 : 0;
}

template <int KC, int NT>
int launch(const CUtensorMap& tm_x, const CUtensorMap& tm_w, const ConvArgs& p, size_t smem_bytes,
           int grid, cudaStream_t st) {
  switch (epi_flavour(p)) {
    case 0: return launch_as<KC, NT, 0>(tm_x, tm_w, p, smem_bytes, grid, st);
    case 1: return launch_as<KC, NT, 1>(tm_x, tm_w, p, smem_bytes, grid, st);
    case 2: return launch_as<KC, NT, 2>(tm_x, tm_w, p, smem_bytes, grid, st);
    case 3: return launch_as<KC, NT, 3>(tm_x, tm_w, p, smem_bytes, grid, st);
    case 5: return launch_as<KC, NT, 5>(tm_x, tm_w, p, smem_bytes, grid, st);
    default: return launch_as<KC, NT, 4>(tm_x, tm_w, p, smem_bytes, grid, st);
  }
}

template <int NT, int kEpi>
int launch2_as(const CUtensorMap& tm_x, const CUtensorMap& tm_w, const ConvArgs& p, size_t smem_bytes, int grid,
               cudaStream_t st) {
  static hg::PerDeviceOnce once;
  if (once.need())
    HG_CHECK_CUDA(cudaFuncSetAttribute(conv1d_tc2_kernel<NT, kEpi>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       g_max_smem));
  conv1d_tc2_kernel<NT, kEpi><<<grid, kThreads, smem_bytes, st>>>(tm_x, tm_w, p);   // __cluster_dims__(2,1,1)
  HG_CHECK_CUDA(cudaGetLastError());
  return HG_OK;
}

template <int NT>
int launch2(const CUtensorMap& tm_x, const CUtensorMap& tm_w, const ConvArgs& p, size_t smem_bytes, int grid,
            cudaStream_t st) {
  switch (epi_flavour(p)) {
    case 0: return launch2_as<NT, 0>(tm_x, tm_w, p, smem_bytes, grid, st);
    case 1: return launch2_as<NT, 1>(tm_x, tm_w, p, smem_bytes, grid, st);
    case 2: return launch2_as<NT, 2>(tm_x, tm_w, p, smem_bytes, grid, st);
    case 3: return launch2_as<NT, 3>(tm_x, tm_w, p, smem_bytes, grid, st);
    case 5: return launch2_as<NT, 5>(tm_x, tm_w, p, smem_bytes, grid, st);
    default: return launch2_as<NT, 4>(tm_x, tm_w, p, smem_bytes, grid, st);
  }
}

int g_use_2cta = -1;

// Packed tap order / residue boxes of a (ktaps, stride, dilation, pad_left) convolution.
struct TapPlan {
  int nboxes;
  int box_col_mult[kMaxBoxes];  // residue rho (multiplied by C_total by the caller)
  int box_row[kMaxBoxes], box_ntaps[kMaxBoxes], box_tap0[kMaxBoxes];
  int tap_step, max_ntaps;
  int order[256];               // packed index -> original tap j
};

int make_tap_plan(int ktaps, int stride, int dilation, int pad_left, TapPlan* tp) {
  if (ktaps < 1 || ktaps > 256 || stride < 1 || stride > kMaxBoxes || dilation < 1) return -1;
  if (stride > 1 && dilation != 1) return -1;
  tp->nboxes = 0;
  tp->max_ntaps = 0;
  if (stride == 1) {
    tp->nboxes = 1;
    tp->box_col_mult[0] = 0; tp->box_row[0] = -pad_left; tp->box_ntaps[0] = ktaps; tp->box_tap0[0] = 0;
    tp->tap_step = dilation; tp->max_ntaps = ktaps;
    for (int j = 0; j < ktaps; ++j) tp->order[j] = j;
    return 0;
  }
  tp->tap_step = 1;
  int q_packed = 0;
  for (int rho = 0; rho < stride; ++rho) {
    int n = 0, qmin = 0;
    for (int j = 0; j < ktaps; ++j) {
      const int e = j - pad_left;
      const int r = ((e % stride) + stride) % stride;
      if (r != rho) continue;
      const int q = (e - r) / stride;
      if (n == 0) qmin = q;
      tp->order[q_packed + n] = j;
      ++n;
    }
    if (!n) continue;
    const int b = tp->nboxes++;
    tp->box_col_mult[b] = rho; tp->box_row[b] = qmin; tp->box_ntaps[b] = n; tp->box_tap0[b] = q_packed;
    q_packed += n;
    if (n > tp->max_ntaps) tp->max_ntaps = n;
  }
  return 0;
}

struct ConvExtra {
  const void* mask = nullptr;
  float mask_slope = 1.f;
  const void* fm_r = nullptr;
  const void* fm_g = nullptr;
  float fm_coef = 0.f;
  int group_mod = 0;      // 0: one input channel block per N tile (forward grouped convs)
  int t_in_valid = -1;    // stride 1 only: input rows >= this are read as zero (TMA bound); -1 = t_in_rows
  int seq_pitch = 0, seq_valid = 0, seq_mul = 1, seq_div = 1 << 30;
  const void* pre_add = nullptr;
  float* colsum[3] = {nullptr, nullptr, nullptr};
  int colsum_mod = 0;     // 0: the launch's output channel count
  const int* item_len = nullptr;
  int item_mul = 1;
  float res0_inv = 1.f;   // 1 / slope of an activated res0 (forward launches only); 1: raw
};

int conv_forward(const void* x, const void* w_packed, const float* bias, int batch, int t_in_rows,
                 int c_total, int t_out, int t_out_rows, int cin_tile, int cout, int n_tile, int grouped, int ktaps,
                 int stride, int dilation, int pad_left, const void* res0, const void* res1,
                 const void* res2, float scale, void* out_raw, void* out_act, float act_slope,
                 void* stream, const ConvExtra& ex = ConvExtra()) {
  HG_REQUIRE(x && w_packed, "conv: null input");
  HG_REQUIRE(out_raw || out_act, "conv: no output requested");
  HG_REQUIRE(batch > 0 && t_out > 0 && t_in_rows > 0, "conv: empty batch/time");
  HG_REQUIRE(cin_tile % 32 == 0 && cin_tile > 0, "conv: cin=%d must be a multiple of 32", cin_tile);
  HG_REQUIRE(cout % 32 == 0 && cout > 0, "conv: cout=%d must be a multiple of 32", cout);
  HG_REQUIRE(n_tile == 32 || n_tile == 64 || n_tile == 128 || n_tile == 256, "conv: bad N tile %d", n_tile);
  HG_REQUIRE(cout % n_tile == 0, "conv: cout %d is not a multiple of the N tile %d", cout, n_tile);
  HG_REQUIRE(t_in_rows % stride == 0, "conv: input rows %d must be a multiple of the stride %d",
             t_in_rows, stride);
  TapPlan tp;
  HG_REQUIRE(make_tap_plan(ktaps, stride, dilation, pad_left, &tp) == 0,
             "conv: unsupported taps/stride/dilation (%d,%d,%d)", ktaps, stride, dilation);
  const int a_rows = kTileM + (tp.max_ntaps - 1) * tp.tap_step;
  HG_REQUIRE(a_rows <= 256, "conv: halo too large for one TMA box (rows=%d > 256)", a_rows);
  int rc = device_props();
  if (rc) return rc;

  const int kc = (cin_tile % 64 == 0) ? 64 : 32;
  ConvArgs p{};
  HG_REQUIRE(t_out_rows >= t_out, "conv: output pitch %d < rows %d", t_out_rows, t_out);
  p.batch = batch; p.t = t_out; p.t_pitch = t_out_rows; p.cin = cin_tile; p.cout = cout;
  p.ktaps = ktaps; p.dil = dilation; p.pad_left = pad_left;
  p.nchunks = cin_tile / kc;
  p.a_rows = a_rows;
  p.nboxes = tp.nboxes;
  for (int b = 0; b < tp.nboxes; ++b) {
    p.box_col[b] = tp.box_col_mult[b] * c_total;
    p.box_row[b] = tp.box_row[b];
    p.box_ntaps[b] = tp.box_ntaps[b];
    p.box_tap0[b] = tp.box_tap0[b];
  }
  p.tap_step = tp.tap_step;
  p.grouped = grouped;
  p.tiles_t = (t_out + kTileM - 1) / kTileM;
  p.tiles_n = cout / n_tile;
  p.num_tiles = batch * p.tiles_t * p.tiles_n;
  p.a_slot_bytes = (static_cast<uint32_t>(a_rows) * kc * 2 + 1023u) & ~1023u;
  const uint32_t tap_bytes = static_cast<uint32_t>(n_tile) * kc * 2;
  // bias-gradient launches keep n_tile fp32 column sums behind the barriers
  const int colsum_bytes = ex.colsum[0] ? 1024 : 0;
  const int budget = g_max_smem - 1024 /*align*/ - static_cast<int>(sizeof(Barriers)) - colsum_bytes;

  // resident filter bank: needs all taps of all chunks + at least 2 activation slots
  const long long w_all = static_cast<long long>(ktaps) * p.nchunks * tap_bytes;
  uint32_t w_bytes_total;
  if (p.tiles_n == 1 && w_all + 2LL * p.a_slot_bytes <= budget && w_all < (1 << 20)) {
    p.resident = 1;
    p.tps = ktaps; p.groups = 1; p.stages = 1;
    p.w_stage_bytes = static_cast<uint32_t>(w_all);
    w_bytes_total = static_cast<uint32_t>(w_all);
  } else {
    p.resident = 0;
    p.tps = tap_bytes >= 32768 ? 1 : static_cast<int>(32768 / tap_bytes);
    if (p.tps > ktaps) p.tps = ktaps;
    p.groups = (ktaps + p.tps - 1) / p.tps;
    p.w_stage_bytes = static_cast<uint32_t>(p.tps) * tap_bytes;
    int stages = (budget - 2 * static_cast<int>(p.a_slot_bytes)) / static_cast<int>(p.w_stage_bytes);
    if (stages > 4) stages = 4;
    HG_REQUIRE(stages >= 2, "conv: not enough shared memory for the weight ring");
    p.stages = stages;
    w_bytes_total = static_cast<uint32_t>(stages) * p.w_stage_bytes;
  }
  if (g_use_2cta < 0) g_use_2cta = getenv("HG_DISABLE_2CTA") ? 0 : 1;
  // CTA-pair path: dense stride-1 layers with streamed weights and wide N tiles (stages 1-2, ups 0-1)
  const bool pair = g_use_2cta && !p.resident && stride == 1 && !grouped && kc == 64 && n_tile >= 128 &&
                    (g_num_sms % 2 == 0) && batch * p.tiles_t * p.tiles_n >= g_num_sms;
  if (pair) {
    const uint32_t half_tap = tap_bytes / 2;          // each CTA holds half of the filter rows
    p.tps = half_tap >= 32768 ? 1 : static_cast<int>(32768 / half_tap);
    if (p.tps > ktaps) p.tps = ktaps;
    p.groups = (ktaps + p.tps - 1) / p.tps;
    p.w_stage_bytes = static_cast<uint32_t>(p.tps) * half_tap;
    int stages = (budget - 2 * static_cast<int>(p.a_slot_bytes)) / static_cast<int>(p.w_stage_bytes);
    if (stages > 4) stages = 4;
    HG_REQUIRE(stages >= 2, "conv: not enough shared memory for the weight ring");
    p.stages = stages;
    w_bytes_total = static_cast<uint32_t>(stages) * p.w_stage_bytes;
  }
  int a_slots = (budget - static_cast<int>(w_bytes_total)) / static_cast<int>(p.a_slot_bytes);
  if (a_slots > kMaxASlots) a_slots = kMaxASlots;
  HG_REQUIRE(a_slots >= 2, "conv: not enough shared memory for the activation ring");
  p.a_slots = a_slots;

  p.bias = bias;
  p.res0 = static_cast<const __nv_bfloat16*>(res0);
  p.res1 = static_cast<const __nv_bfloat16*>(res1);
  p.res2 = static_cast<const __nv_bfloat16*>(res2);
  p.scale = scale;
  p.out_raw = static_cast<__nv_bfloat16*>(out_raw);
  p.out_act = static_cast<__nv_bfloat16*>(out_act);
  p.slope = act_slope;
  p.mask = static_cast<const __nv_bfloat16*>(ex.mask);
  p.mask_slope = ex.mask_slope;
  p.fm_r = static_cast<const __nv_bfloat16*>(ex.fm_r);
  p.fm_g = static_cast<const __nv_bfloat16*>(ex.fm_g);
  p.fm_coef = ex.fm_coef;
  p.group_mod = ex.group_mod > 0 ? ex.group_mod : p.tiles_n;
  p.seq_pitch = ex.seq_pitch; p.seq_valid = ex.seq_valid; p.seq_mul = ex.seq_mul;
  p.pre_add = static_cast<const __nv_bfloat16*>(ex.pre_add);
  for (int i = 0; i < 3; ++i) p.colsum[i] = ex.colsum[i];
  p.colsum_mod = ex.colsum_mod > 0 ? ex.colsum_mod : cout;
  p.item_len = ex.item_len; p.item_mul = ex.item_mul;
  p.res0_inv = ex.res0_inv;
  HG_REQUIRE(!ex.colsum[1] || ex.colsum[0], "conv: bias-gradient destinations must be filled from slot 0");
  p.seq_div = ex.seq_div > 0 ? ex.seq_div : (1 << 30);
  HG_REQUIRE(ex.seq_pitch >= 0 && (ex.seq_pitch == 0 || batch == 1), "conv: flat sequences need batch == 1");
  HG_REQUIRE(!p.fm_g || p.fm_r, "conv: fm_g without fm_r");
  HG_REQUIRE(ex.t_in_valid < 0 || (stride == 1 && ex.t_in_valid <= t_in_rows), "conv: bad input bound");
  const int t_in_bound = ex.t_in_valid >= 0 ? ex.t_in_valid : t_in_rows / stride;

  CUtensorMap tm_x, tm_w;
  const int swz = kc * 2;
  // activations through the strided view [B][T_in/stride][stride*C_total]
  rc = hg_encode_tmap_bf16_3d(&tm_x, x, static_cast<uint64_t>(stride) * c_total, t_in_bound, batch,
                              static_cast<uint64_t>(stride) * c_total * 2,
                              static_cast<uint64_t>(t_in_rows) * c_total * 2, kc, a_rows, 1, swz);
  if (rc) return rc;
  rc = hg_encode_tmap_bf16_3d(&tm_w, w_packed, cin_tile, cout, ktaps, static_cast<uint64_t>(cin_tile) * 2,
                              static_cast<uint64_t>(cout) * cin_tile * 2, kc, pair ? n_tile / 2 : n_tile, p.tps,
                              swz);
  if (rc) return rc;

  const size_t smem_bytes = 1024 + static_cast<size_t>(a_slots) * p.a_slot_bytes + w_bytes_total +
                            sizeof(Barriers) + colsum_bytes;
  const int grid = p.num_tiles < g_num_sms ? p.num_tiles : g_num_sms;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (pair) {
    const size_t smem2 = 1024 + static_cast<size_t>(a_slots) * p.a_slot_bytes + w_bytes_total + sizeof(Barriers2) +
                         colsum_bytes;
    const int grid2 = g_num_sms;     // whole CTA pairs: `pair` requires an even SM count
    rc = (n_tile == 256) ? launch2<256>(tm_x, tm_w, p, smem2, grid2, st)
                         : launch2<128>(tm_x, tm_w, p, smem2, grid2, st);
    if (rc) return rc;
    g_hg_launches.fetch_add(1, std::memory_order_relaxed);
    return HG_OK;
  }
#define HG_LAUNCH(KC_, NT_) rc = launch<KC_, NT_>(tm_x, tm_w, p, smem_bytes, grid, st)
  if (kc == 64) {
    if (n_tile == 256) HG_LAUNCH(64, 256);
    else if (n_tile == 128) HG_LAUNCH(64, 128);
    else if (n_tile == 64) HG_LAUNCH(64, 64);
    else HG_LAUNCH(64, 32);
  } else {
    if (n_tile == 256) HG_LAUNCH(32, 256);
    else if (n_tile == 128) HG_LAUNCH(32, 128);
    else if (n_tile == 64) HG_LAUNCH(32, 64);
    else HG_LAUNCH(32, 32);
  }
#undef HG_LAUNCH
  if (rc) return rc;
  g_hg_launches.fetch_add(1, std::memory_order_relaxed);
  return HG_OK;
}

}  // namespace

namespace {

int conv1d_fwd(const void* x, const void* w_packed, const float* bias, int batch, int t, int cin, int cout, int ktaps,
               int dilation, int pad_left, const void* res0, float res0_inv, const void* res1, const void* res2,
               float scale, void* out_raw, void* out_act, float act_slope, const int* item_len, int item_mul,
               void* stream) {
  HG_REQUIRE(cout > 0 && cout % 32 == 0, "hg_conv1d_fwd: cout=%d must be a multiple of 32", cout);
  HG_REQUIRE(cin > 0 && cin % 32 == 0, "hg_conv1d_fwd: cin=%d must be a multiple of 32", cin);
  HG_REQUIRE(ktaps > 0 && dilation > 0 && 128 + (ktaps - 1) * dilation <= 256,
             "hg_conv1d_fwd: halo too large for one TMA box (taps=%d dilation=%d)", ktaps, dilation);
  const int n_tile = (cout % 256 == 0) ? 256 : (cout % 128 == 0) ? 128 : (cout % 64 == 0) ? 64 : 32;
  ConvExtra ex;
  ex.item_len = item_len; ex.item_mul = item_mul > 0 ? item_mul : 1;
  ex.res0_inv = res0_inv;
  return conv_forward(x, w_packed, bias, batch, t, cin, t, t, cin, cout, n_tile, 0, ktaps, 1, dilation, pad_left,
                      res0, res1, res2, scale, out_raw, out_act, act_slope, stream, ex);
}

}  // namespace

extern "C" int hg_conv1d_fwd(const void* x, const void* w_packed, const float* bias, int batch, int t,
                             int cin, int cout, int ktaps, int dilation, int pad_left,
                             const void* res0, const void* res1, const void* res2, float scale,
                             void* out_raw, void* out_act, float act_slope, const int* item_len, int item_mul,
                             void* stream) {
  return conv1d_fwd(x, w_packed, bias, batch, t, cin, cout, ktaps, dilation, pad_left, res0, 1.f, res1, res2, scale,
                    out_raw, out_act, act_slope, item_len, item_mul, stream);
}

extern "C" int hg_conv1d_fwd_actres(const void* x, const void* w_packed, const float* bias, int batch, int t,
                                    int cin, int cout, int ktaps, int dilation, int pad_left,
                                    const void* res0, float res0_slope, const void* res1, const void* res2,
                                    float scale, void* out_raw, void* out_act, float act_slope, const int* item_len,
                                    int item_mul, void* stream) {
  HG_REQUIRE(res0 && res0_slope > 0.f && res0_slope <= 1.f,
             "hg_conv1d_fwd_actres: needs res0 and a slope in (0, 1] (got %g)", res0_slope);
  return conv1d_fwd(x, w_packed, bias, batch, t, cin, cout, ktaps, dilation, pad_left, res0, 1.f / res0_slope, res1,
                    res2, scale, out_raw, out_act, act_slope, item_len, item_mul, stream);
}

extern "C" int hg_conv1d_tap_order(int ktaps, int stride, int pad_left, int* host_order) {
  TapPlan tp;
  HG_REQUIRE(host_order && make_tap_plan(ktaps, stride, 1, pad_left, &tp) == 0,
             "hg_conv1d_tap_order: unsupported (taps=%d stride=%d)", ktaps, stride);
  for (int q = 0; q < ktaps; ++q) host_order[q] = tp.order[q];
  return HG_OK;
}

extern "C" int hg_conv1d_general_fwd(const void* x, const void* w_packed, const float* bias, int batch,
                                     int t_in_rows, int c_total, int t_out, int t_out_rows, int groups,
                                     int cout, int ktaps,
                                     int stride, int pad_left, void* out_act, float act_slope,
                                     void* out_raw, int seq_pitch, int seq_valid, void* stream) {
  HG_REQUIRE(groups >= 1 && c_total % groups == 0 && cout % groups == 0, "hg_conv1d_general_fwd: bad groups");
  const int cin_tile = c_total / groups, n_tile_g = cout / groups;
  ConvExtra ex;
  ex.seq_pitch = seq_pitch; ex.seq_valid = seq_valid;
  if (groups == 1) {
    const int n_tile = (cout % 256 == 0) ? 256 : (cout % 128 == 0) ? 128 : (cout % 64 == 0) ? 64 : 32;
    return conv_forward(x, w_packed, bias, batch, t_in_rows, c_total, t_out, t_out_rows, c_total, cout, n_tile, 0,
                        ktaps,
                        stride, 1, pad_left, nullptr, nullptr, nullptr, 1.f, out_raw, out_act, act_slope,
                        stream, ex);
  }
  return conv_forward(x, w_packed, bias, batch, t_in_rows, c_total, t_out, t_out_rows, cin_tile, cout, n_tile_g, 1,
                      ktaps,
                      stride, 1, pad_left, nullptr, nullptr, nullptr, 1.f, out_raw, out_act, act_slope,
                      stream, ex);
}

// hg_conv1d_dgrad — data gradient of a conv layer, run on the same implicit-GEMM kernel: the gradient of a
// stride-1 dilated conv is a conv with flipped taps and transposed filters (hg_pack_dgrad_weight), the gradient
// of a strided conv (or the forward of its transpose) is its polyphase form (hg_pack_convtr1d_weight on the
// conv weight).  The epilogue applies the leaky_relu backward mask of the layer input, the feature-matching L1
// term and up to two gradient addends (residual path / MRF branch sum):
//   out[b,t,n] = ((sum_{j,c} dy[b, t + j*dil - pad_left, blk(n) + c] * w[j][n][c] + fm_coef * sgn(fm_g - fm_r) + pre_add)
//                 * (mask_src > 0 ? 1 : mask_slope) + res0 + res1 + res2) * scale
//   bias_grad*[n % bias_mod] += sum_{b,t} out[b,t,n]   (fp32, before the bf16 rounding of `out`)
extern "C" int hg_conv1d_dgrad(const void* dy, const void* w_packed, int batch, int t_dy_valid, int t_dy_rows,
                               int c_dy_total, int t_out, int t_out_rows, int groups, int n_tile, int cout, int ktaps,
                               int dilation, int pad_left, const void* mask_src, float mask_slope,
                               const void* fm_r, const void* fm_g, float fm_coef, const void* res0, const void* res1,
                               const void* res2, float scale, void* out, int seq_pitch, int seq_valid, int seq_mul,
                               int seq_div, const void* pre_add, float* bias_grad0, float* bias_grad1,
                               float* bias_grad2, int bias_mod, void* stream) {
  HG_REQUIRE(groups >= 1 && c_dy_total % groups == 0, "hg_conv1d_dgrad: bad groups");
  HG_REQUIRE(ktaps > 0 && dilation > 0 && 128 + (ktaps - 1) * dilation <= 256,
             "hg_conv1d_dgrad: halo too large for one TMA box (taps=%d dilation=%d)", ktaps, dilation);
  ConvExtra ex;
  ex.mask = mask_src; ex.mask_slope = mask_slope;
  ex.fm_r = fm_r; ex.fm_g = fm_g; ex.fm_coef = fm_coef;
  ex.t_in_valid = t_dy_valid;
  ex.seq_pitch = seq_pitch; ex.seq_valid = seq_valid; ex.seq_mul = seq_mul > 0 ? seq_mul : 1; ex.seq_div = seq_div;
  ex.pre_add = pre_add;
  ex.colsum[0] = bias_grad0; ex.colsum[1] = bias_grad1; ex.colsum[2] = bias_grad2; ex.colsum_mod = bias_mod;
  const int cin_tile = c_dy_total / groups;
  if (groups == 1) {
    if (n_tile <= 0) n_tile = (cout % 256 == 0) ? 256 : (cout % 128 == 0) ? 128 : (cout % 64 == 0) ? 64 : 32;
    return conv_forward(dy, w_packed, nullptr, batch, t_dy_rows, c_dy_total, t_out, t_out_rows, cin_tile, cout,
                        n_tile, 0, ktaps, 1, dilation, pad_left, res0, res1, res2, scale, out, nullptr, 1.f,
                        stream, ex);
  }
  HG_REQUIRE(n_tile > 0, "hg_conv1d_dgrad: grouped layers need an explicit N tile");
  ex.group_mod = groups;
  return conv_forward(dy, w_packed, nullptr, batch, t_dy_rows, c_dy_total, t_out, t_out_rows, cin_tile, cout,
                      n_tile, 1, ktaps, 1, dilation, pad_left, res0, res1, res2, scale, out, nullptr, 1.f,
                      stream, ex);
}
