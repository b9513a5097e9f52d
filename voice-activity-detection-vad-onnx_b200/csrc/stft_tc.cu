// stft_tc.cu -- framed real DFT + power (a1 + a2) on the tensor cores, straight from int16 audio.
//
//   power[(s*T + t)][f] = | sum_n y[s][t*hop - pad_left + n] * w[n] e^{-i 2 pi f n / n_fft} |^2 ,
//   y[i] = scale * (x[i] - c * x[i-1])            (x int16, x[-1] = 0: the reference's pad(1,0)+conv)
//
// as ONE tensor-core GEMM with fp32-grade accuracy and no prepared-signal round trip:
//   * an int16 sample splits EXACTLY into two bf16 / fp16 terms, x = 256*(x >> 8) + (x & 255);
//   * pre-emphasis and the int16 scale are folded into the basis on the host, in double:
//       B'[k][col] = scale * (b[k-8][col] - c * b[k-7][col])      (k-8 = tap index; 8 leading zero
//     rows keep every 8-sample group of a frame 16-byte aligned and make room for the x[i-1] tap);
//   * B' is split into TWO terms b0 + b1, stacked as one N = 160 operand, so x_hi * [b0|b1] and x_lo * [b0|b1] are the two
//     MMAs of a K = 16 step; the epilogue adds the two column blocks of the fp32 TMEM accumulator.
// Centre-padded frontends (frames reaching outside [0, L): zero samples) and DC removal (integer part of the mean taken
// off the samples by the loaders, the fractional part and the pre-emphasised pad's tail put back from per-frame tables in
// the epilogue) are the EX variant.
//
// Hop rows instead of frames.  With hop % 16 == 0, K16 step k = (hop/16)*q + j of frame t reads samples
// [origin(t) + 16k, +16), origin(t) = t*hop - pad_left - 8: slice j of HOP ROW t + q, where hop row h holds the hop samples
// from h*hop - pad_left - 8.  The A operand is stored without swizzle, K-major, one 8-sample slice of all rows at a time
// with the rows 16 B apart, so "hop row t + q" for the 128 frames of a tile is the same slice 16*q bytes further on.  A
// tile of 128 M rows therefore needs its 128 + Q - 1 hop rows (Q = hop rows a frame spans) converted once, instead of
// 128 frames that overlap Q-fold.  M rows are SLOTS: T + Q - 1 per stream, so a frame's hop rows never cross into the
// next stream; the Q - 1 extra slots compute rows that are never stored.
//
// Work decomposition: the (re, im)-interleaved output columns are cut into N-tiles of 80; a CTA keeps the 2-term basis
// image of ITS N-tile resident in shared memory (143 KB for 400 taps, fetched once with cp.async.bulk) and streams
// 128-slot tiles through a 3-deep ring of stages, each holding kStJ K16 columns of all the tile's hop rows as (hi, lo).
// Warp roles: 16 loader warps (int16 -> (hi, lo), register buffers keep the loads of several stages in flight), 4
// epilogue warps (TMEM -> re^2+im^2 -> global), 1 MMA issuer, two TMEM accumulators in ping-pong.
#include "tc_ptx.cuh"

namespace vadx {

constexpr int kStNPad = 80;                          // columns per N-tile (40 bins)
constexpr int kStTerms = 2;                          // terms of the folded basis
constexpr int kStLead = 8;                           // leading zero rows of the folded basis
constexpr int kStJ = 2;                              // K16 columns of the hop rows per ring stage
constexpr int kStSlices = 2 * kStJ;                  // 8-sample slices per stage
constexpr int kStStages = 3;
constexpr int kStLoaderWarps = 16;
constexpr int kStOutLd = 44;                         // floats per staged output row (40 used; 44 keeps float4 stores conflict-free)
// epilogue warps kStLoaderWarps..+3 ((warp & 3) = TMEM lane quarter), MMA warp kStLoaderWarps + 4

struct StftTcArgs {
  const int16_t* X;
  int64_t in_stride;   // samples between streams
  int64_t L;           // valid samples per stream
  int64_t S;           // streams
  int n_frames, hop;
  int h16;             // hop / 16: K16 columns per hop row
  int n_q;             // Q: hop rows one frame's n_k16 steps span
  int tq;              // slots per stream (n_frames + Q - 1)
  int rows;            // hop rows of one tile (kTcBM + Q - 1)
  int slice_units;     // 16-byte units between two 8-sample slices of a stage (>= rows)
  int n_st;            // ring stages per tile (ceil(h16 / kStJ))
  const uint8_t* Wimg;  // [n_ntiles][kc][2][kStNPad*128]
  float* P;
  int64_t ldp;
  int n_bins, kc, n_k16, n_tiles, vec_p;
  int pad_left;          // zero samples before sample 0 (centre pad minus the window's dead taps); multiple of 8
  const float* mean;     // [S] FRACTIONAL part of the per-stream mean (removed in the epilogue), or null
  const int* mean_int;   // [S] integer part of the mean, subtracted from the samples by the loaders (exact: the
                         // 17-bit difference still splits into two bf16-exact terms)
  const float* dc;       // [(1 + n_edge) + n_edge_hi][n_ntiles * kStNPad]: the folded basis applied to the mean's
                         // coefficient pattern -- row 0 for interior frames, one row per frame that touches the zero
                         // pad -- then one tail row per frame that runs past the end of the stream
  int n_edge_lo, t_edge_hi;   // frames t < n_edge_lo and t >= t_edge_hi are edge frames
  float power_scale;     // multiplies re^2 + im^2 (a scale kept out of an fp16 basis, e.g. (1/32768)^2)
  int stage_out;   // 1: the epilogue transposes each warp's 32 x 40 powers through shared memory (coalesced stores)
  unsigned backoff_ld, backoff_epi;   // nanoseconds between mbarrier probes of the loader / epilogue warps
  int debug;  // VADX_TC_DEBUG perf experiments: 1 no stores, 4 x_hi product only, 8 loaders write no shared memory
};

// Exact int -> bf16 without the (quarter-rate) conversion pipe: for 0 <= v < 2^23,
// as_float(0x4B000000 | v) == 8388608 + v, so one FADD/FFMA yields float(v); integers with <= 8
// significant bits are exact in bf16, i.e. the bf16 word is just the upper half of the fp32 word.
__device__ __forceinline__ uint32_t bf16x2_lo(uint32_t w) {
  // (w & 0xff) and ((w >> 16) & 0xff): the low bytes of the two packed int16 samples, both in [0, 255]
  const float a = __uint_as_float(0x4B000000u | (w & 0xffu)) - 8388608.0f;
  const float b = __uint_as_float(0x4B000000u | ((w >> 16) & 0xffu)) - 8388608.0f;
  return __byte_perm(__float_as_uint(a), __float_as_uint(b), 0x7632);
}
__device__ __forceinline__ uint32_t bf16x2_hi(uint32_t w) {
  // 256 * (x >> 8) for the two packed int16 samples: ((x >> 8) + 128) is in [0, 255]
  const uint32_t ha = (((w >> 8) & 0xffu) ^ 0x80u);          // (x_a >> 8) + 128 (two's complement high byte)
  const uint32_t hb = (((w >> 24) & 0xffu) ^ 0x80u);
  const float a = fmaf(__uint_as_float(0x4B000000u | ha), 256.0f, -(8388608.0f + 128.0f) * 256.0f);
  const float b = fmaf(__uint_as_float(0x4B000000u | hb), 256.0f, -(8388608.0f + 128.0f) * 256.0f);
  return __byte_perm(__float_as_uint(a), __float_as_uint(b), 0x7632);
}

// fp16 operands: the same exact split in three half2 operations per pair of samples.  as_half(0x6400 | v) is
// 1024 + v for 0 <= v < 1024, so (w & 0x00ff00ff) | 0x64006400 minus 1024 is the pair of low bytes, and the
// sign-flipped high bytes minus (1024 + 128), times 256, is the pair 256 * (x >> 8) (|.| <= 32768 fits fp16).
__device__ __forceinline__ uint32_t f16x2_lo(uint32_t w) {
  const uint32_t m = (w & 0x00ff00ffu) | 0x64006400u;
  uint32_t r;
  asm("sub.rn.f16x2 %0, %1, %2;" : "=r"(r) : "r"(m), "r"(0x64006400u));
  return r;
}
__device__ __forceinline__ uint32_t f16x2_hi(uint32_t w) {
  const uint32_t m = (((w >> 8) & 0x00ff00ffu) ^ 0x00800080u) | 0x64006400u;
  uint32_t r;
  asm("sub.rn.f16x2 %0, %1, %2;" : "=r"(r) : "r"(m), "r"(0x64806480u));      // 1024 + 128
  asm("mul.rn.f16x2 %0, %1, %2;" : "=r"(r) : "r"(r), "r"(0x5c005c00u));      // x 256
  return r;
}

// same trick for a sample with an integer offset removed: d in [-65535, 65535] -> (256 * (d >> 8), d & 255)
__device__ __forceinline__ void split17(int d, float& hi, float& lo) {
  lo = __uint_as_float(0x4B000000u | (uint32_t)(d & 255)) - 8388608.0f;
  const uint32_t h = (uint32_t)((d >> 8) + 256);   // [0, 511]
  hi = fmaf(__uint_as_float(0x4B000000u | h), 256.0f, -(8388608.0f + 256.0f) * 256.0f);
}

// EX = false: every frame inside the stream, no DC removal (FireRed) -- the padded / mean-removing code is compiled out
// F16 = true: fp16 operands (cheaper exact conversion; not with the 17-bit mean-removed samples)
template <bool EX, bool F16>
__global__ void __launch_bounds__((kStLoaderWarps + 5) * 32, 1) stft_power_tc_kernel(const StftTcArgs g) {
  constexpr int kStEpiWarp0 = kStLoaderWarps, kStMmaWarp = kStLoaderWarps + 4;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* w_smem = smem_raw;
  const uint32_t img_bytes = kStNPad * 128u;
  const int w_bytes = g.kc * kStTerms * (int)img_bytes;
  uint8_t* a_smem = w_smem + w_bytes;
  // stage = [x_hi | x_lo], each [kStSlices][slice_units * 16 B]: slice i of a stage holds 8 samples of every hop row
  const uint32_t slice_bytes = (uint32_t)g.slice_units * 16u;
  const uint32_t term_bytes = kStSlices * slice_bytes;
  const uint32_t stage_bytes = 2u * term_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(a_smem + (size_t)kStStages * stage_bytes);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 13);
  float* out_stage = reinterpret_cast<float*>(bars + 16);   // [4 warps][32 rows][kStOutLd], only when g.stage_out

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t bar0 = smem_u32(bars);
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (4 + s); };
  auto tfull_bar = [&](int b) { return bar0 + 8u * (8 + b); };
  auto tempty_bar = [&](int b) { return bar0 + 8u * (10 + b); };
  const uint32_t wbar = bar0 + 8u * 12;
  constexpr int kAccN = 2 * kStNPad;   // x * b0 | x * b1
  constexpr uint32_t kTmemCols = 512;  // 2 accumulators of 160 columns

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStStages; ++s) {
      mbar_init(full_bar(s), kStLoaderWarps);     // one elected lane per loader warp
      mbar_init(empty_bar(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(tfull_bar(b), 1);
      mbar_init(tempty_bar(b), 4);   // one elected lane per epilogue warp
    }
    mbar_init(wbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kStMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int ntile = blockIdx.y;

  if (warp == kStMmaWarp) {
    if (lane == 0) {
      mbar_expect_tx(wbar, (uint32_t)w_bytes);
      const uint8_t* src = g.Wimg + (size_t)ntile * w_bytes;
      for (int t = 0; t < g.kc * kStTerms; ++t) bulk_g2s(smem_u32(w_smem) + t * img_bytes, src + (size_t)t * img_bytes, img_bytes, wbar);
      mbar_wait(wbar, 0);
      const uint32_t idesc = F16 ? umma_idesc_f16(kAccN) : umma_idesc_bf16(kAccN);
      // descriptors advance in their 16-byte address units: B by one 64-wide basis chunk (both terms) per 4 K16 steps and
      // 32 B per step inside it (the SW128 image, as umma_k64 reads it); A by one row per q, two slices per K16 column
      const uint64_t dw = umma_desc_sw128(smem_u32(w_smem));
      const uint64_t da0 = umma_desc_noswz(smem_u32(a_smem), slice_bytes, 128u);
      const uint32_t chunk_units = (kStTerms * img_bytes) >> 4, lo_units = term_bytes >> 4, stage_units = stage_bytes >> 4;
      const uint32_t col_units = (2u * slice_bytes) >> 4;
      const int h16 = g.h16, n_k16 = g.n_k16;
      const uint32_t lo_on = (g.debug & 4) ? 0u : 1u;
      // Issue pacing, measured on a B200 (bench.py, tools/stft_microbench.py): with fp16 operands and no padding or mean
      // removal -- the cheapest loader -- the issuing thread bounds the kernel, and a column's up to three MMA pairs from
      // one asm block take FireRed's STFT from 1.28 to 1.10 ms per 8192 chunks.  A build that issued every variant that
      // way was 10-20 % slower in the bf16 and the padded / mean-removing variants, so those issue one pair at a time.
      constexpr bool kBurst = F16 && !EX;
      auto b_desc = [&](int k) { return dw + (uint64_t)((uint32_t)(k >> 2) * chunk_units + 2u * (uint32_t)(k & 3)); };
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < g.n_tiles; tile += gridDim.x, ++it) {
        const int b = it & 1;
        const uint32_t use = (uint32_t)(it >> 1);
        mbar_wait(tempty_bar(b), (use & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(b * kAccN);
        for (int st = 0; st < g.n_st; ++st) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint64_t da_st = da0 + (uint64_t)stage * stage_units;
#pragma unroll
          for (int jj = 0; jj < kStJ; ++jj) {
            const int j = st * kStJ + jj;
            if (j >= h16) break;
            const uint64_t da_j = da_st + (uint64_t)jj * col_units;
            // column j, K16 steps k = j + h16 * q: the frame's q-th hop row is 16 bytes (one row) further on.  The first
            // MMA of a tile (k = 0, the dominant x_hi * b0 | x_hi * b1 term) overwrites the accumulator
            if (kBurst) {
              for (int q0 = 0, k = j; k < n_k16; q0 += 3, k += 3 * h16) {
                const int n_pairs = 1 + (k + h16 < n_k16 ? 1 : 0) + (k + 2 * h16 < n_k16 ? 1 : 0);
                umma_split_x3(d_tmem, da_j + (uint64_t)q0, 1u, lo_units, b_desc(k), b_desc(k + h16), b_desc(k + 2 * h16),
                              idesc, k ? 1u : 0u, n_pairs, lo_on);
              }
            } else {
              for (int q = 0, k = j; k < n_k16; ++q, k += h16) {
                const uint64_t da = da_j + (uint64_t)q;
                if (g.debug & 4) umma_bf16(d_tmem, da, b_desc(k), idesc, k ? 1u : 0u);
                else umma_x2(d_tmem, da, da + lo_units, b_desc(k), idesc, k ? 1u : 0u);
              }
            }
          }
          umma_commit(empty_bar(stage));
          if (++stage == kStStages) { stage = 0; phase ^= 1u; }
        }
        umma_commit(tfull_bar(b));
      }
    }
  } else if (warp < kStLoaderWarps) {
    // ===================== loaders: int16 hop rows -> exact (hi, lo) =====================
    // thread = (slice of the stage, row mod 128): the 4 lanes of a row read its 64 contiguous bytes of the stage, 8 rows
    // per warp.  A quarter-warp's 16-byte stores land on 2 rows x 4 slices; slice_units = 2 (mod 4) spreads them over all
    // 8 16-byte bank groups.  Rows 128.. (the Q - 1 halo rows) take a second pass on the first warp.
    constexpr int kRowsPerPass = kStLoaderWarps * 32 / kStSlices;   // 128
    constexpr int kPasses = 2;                                      // rows <= 256
    const int t = threadIdx.x;
    const int sl = t % kStSlices;
    const int r_in = t / kStSlices;
    // per row of the tile being PREFETCHED: stream base and first sample of the hop row (recomputed once per tile: the
    // 64-bit divisions must not sit on the per-stage path)
    const int16_t* xs_n[kPasses];
    int h0_n[kPasses];
    uint32_t rok_n = 0u;
    int tile_cached = -1;
    struct Seq { int tile, st; };
    auto valid = [&](const Seq& q) { return q.tile < g.n_tiles; };
    auto advance = [&](Seq& q) { if (++q.st == g.n_st) { q.st = 0; q.tile += gridDim.x; } };
    const int n_groups = 2 * g.h16;   // 8-sample groups of a hop row
    auto issue = [&](const Seq& q, uint4* raw, uint32_t& msk) {
      msk = 0u;
      if (q.tile != tile_cached) {
        rok_n = 0u;
#pragma unroll
        for (int pass = 0; pass < kPasses; ++pass) {
          const int r = pass * kRowsPerPass + r_in;
          const int64_t slot = (int64_t)q.tile * kTcBM + r;
          const int64_t s = slot / g.tq;
          const int h = (int)(slot - s * g.tq);
          const bool ok = r < g.rows && s < g.S;
          xs_n[pass] = g.X + (ok ? s : 0) * g.in_stride;
          h0_n[pass] = h * g.hop - (EX ? g.pad_left : 0) - kStLead;
          if (ok) rok_n |= 1u << pass;
        }
        tile_cached = q.tile;
      }
      const int grp = q.st * kStSlices + sl;
#pragma unroll
      for (int pass = 0; pass < kPasses; ++pass) {
        const int i0 = h0_n[pass] + 8 * grp;  // first of 8 consecutive samples (stream-relative)
        // hop, pad_left, the lead (8) and the stream length are all multiples of 8 samples, so an 8-sample group lies
        // either entirely inside [0, L) or entirely outside it (zero pad): no element-wise edge path
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (((rok_n >> pass) & 1u) && grp < n_groups && i0 >= 0 && i0 + 7 < g.L) {
          v = __ldg(reinterpret_cast<const uint4*>(xs_n[pass] + i0));
          msk |= 1u << pass;
        }
        raw[pass] = v;
      }
    };
    int stage = 0;
    uint32_t phase = 0;
    int mi_c[kPasses];        // integer mean of each row's stream, for the tile being CONSUMED
#pragma unroll
    for (int pass = 0; pass < kPasses; ++pass) mi_c[pass] = 0;
    int tile_cached_c = -1;
    auto consume = [&](const Seq& q, const uint4* raw, uint32_t msk) {
      if (EX && g.mean_int && q.tile != tile_cached_c) {
#pragma unroll
        for (int pass = 0; pass < kPasses; ++pass) {
          const int64_t s = ((int64_t)q.tile * kTcBM + pass * kRowsPerPass + r_in) / g.tq;
          mi_c[pass] = s < g.S ? __ldg(g.mean_int + s) : 0;
        }
        tile_cached_c = q.tile;
      }
      mbar_wait(empty_bar(stage), phase ^ 1u, g.backoff_ld);
      uint8_t* st_hi = a_smem + (size_t)stage * stage_bytes + sl * slice_bytes;
      uint8_t* st_lo = st_hi + term_bytes;
      if (!(g.debug & 8) && q.st * kStSlices + sl < n_groups)
#pragma unroll
      for (int pass = 0; pass < kPasses; ++pass) {
        const int r = pass * kRowsPerPass + r_in;
        if (r >= g.rows) break;
        const uint32_t wds[4] = {raw[pass].x, raw[pass].y, raw[pass].z, raw[pass].w};
        uint32_t hi[4], lo[4];
        if (EX && g.mean_int) {
          // integer part of the stream's mean removed from the real samples only (the zero pad stays zero)
          const int mi = ((msk >> pass) & 1u) ? mi_c[pass] : 0;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t w = wds[j];
            const int a = ((int)(w << 16) >> 16) - mi;
            const int b = ((int)w >> 16) - mi;
            float ah, al, bh, bl;
            split17(a, ah, al);
            split17(b, bh, bl);
            hi[j] = __byte_perm(__float_as_uint(ah), __float_as_uint(bh), 0x7632);
            lo[j] = __byte_perm(__float_as_uint(al), __float_as_uint(bl), 0x7632);
          }
        } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint32_t w = wds[j];
          hi[j] = F16 ? f16x2_hi(w) : bf16x2_hi(w);
          lo[j] = F16 ? f16x2_lo(w) : bf16x2_lo(w);
        }
        }
        *reinterpret_cast<uint4*>(st_hi + r * 16) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(st_lo + r * 16) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      }
      if (!(g.debug & 16)) fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(full_bar(stage));
      if (++stage == kStStages) { stage = 0; phase ^= 1u; }
    };
    // kStBufs register buffers rotate: the loads of kStBufs - 1 stages are in flight while one is converted
    // (the padded / mean-removing variant carries more live state per thread and keeps fewer)
    constexpr int kStBufs = EX ? 4 : 6;
    uint4 bufs[kStBufs][kPasses];
    uint32_t msks[kStBufs];
#pragma unroll
    for (int i = 0; i < kStBufs; ++i) msks[i] = 0u;
    Seq nxt{(int)blockIdx.x, 0}, cur{(int)blockIdx.x, 0};
#pragma unroll
    for (int i = 0; i < kStBufs - 1; ++i)
      if (valid(nxt)) { issue(nxt, bufs[i], msks[i]); advance(nxt); }
    while (valid(cur)) {
#pragma unroll
      for (int i = 0; i < kStBufs; ++i) {
        constexpr int kPrev = kStBufs - 1;
        if (valid(nxt)) { issue(nxt, bufs[(i + kPrev) % kStBufs], msks[(i + kPrev) % kStBufs]); advance(nxt); }
        consume(cur, bufs[i], msks[i]); advance(cur);
        if (!valid(cur)) break;
      }
    }
  } else {
    // ===================== epilogue: re^2 + im^2 =====================
    const int q = warp - kStEpiWarp0;
    int it = 0;
    const int f0 = ntile * (kStNPad / 2);
    for (int tile = blockIdx.x; tile < g.n_tiles; tile += gridDim.x, ++it) {
      const int b = it & 1;
      const uint32_t use = (uint32_t)(it >> 1);
      mbar_wait(tfull_bar(b), use & 1u, g.backoff_epi);   // a tile takes microseconds: poll rarely
      tc_fence_after();
      // slot -> (stream, frame); the Q - 1 slots past a stream's last frame hold no frame
      const int64_t slot = (int64_t)tile * kTcBM + q * 32 + lane;
      const int64_t sidx = slot / g.tq;
      const int t = (int)(slot - sidx * g.tq);
      const bool row_ok = sidx < g.S && t < g.n_frames;
      const int64_t row = row_ok ? sidx * g.n_frames + t : -1;
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(b * kAccN);
      float* const my_out = out_stage + (size_t)q * 32 * kStOutLd;
      // DC removal in the frequency domain: X(x - m) = X(x) - m * (folded basis applied to the mean's
      // coefficient pattern), exact in fp32; only frames touching the zero pad need their own row of the table
      // Frames that run past the end of the stream: the reference pads the PRE-EMPHASISED signal with zeros, the
      // folded basis sees y[L] = 0 - c*x[L-1] there; the tail table (c * b[L - origin(t)][col]) puts it back.
      float m_row = 0.f, x_last = 0.f;
      const float* dc_row = nullptr;
      const float* tail_row = nullptr;
      if (EX && g.dc && row_ok) {
        const int n_edge = g.n_edge_lo + (g.n_frames - g.t_edge_hi);
        if (g.mean) {
          m_row = __ldg(g.mean + sidx);
          const int e = t < g.n_edge_lo ? 1 + t : (t >= g.t_edge_hi ? 1 + g.n_edge_lo + (t - g.t_edge_hi) : 0);
          dc_row = g.dc + ((size_t)e * gridDim.y + ntile) * kStNPad;
        }
        if (t >= g.t_edge_hi) {
          x_last = (float)((int)__ldg(g.X + sidx * g.in_stride + (g.L - 1)) - (g.mean_int ? __ldg(g.mean_int + sidx) : 0));
          tail_row = g.dc + ((size_t)(1 + n_edge + (t - g.t_edge_hi)) * gridDim.y + ntile) * kStNPad;
        }
      }
#pragma unroll
      for (int c0 = 0; c0 < kStNPad; c0 += 16) {
        float v[16], v2[16];
        tmem_ld16(taddr + (uint32_t)c0, v);
        tmem_ld16(taddr + (uint32_t)(kStNPad + c0), v2);
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] += v2[j];
        if (!row_ok || (g.debug & 1)) continue;
        if (EX && dc_row) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = fmaf(-m_row, __ldg(dc_row + c0 + j), v[j]);
        }
        if (EX && tail_row) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = fmaf(x_last, __ldg(tail_row + c0 + j), v[j]);
        }
        float* out = g.P + row * g.ldp + f0 + c0 / 2;
        float pw[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) pw[j] = (v[2 * j] * v[2 * j] + v[2 * j + 1] * v[2 * j + 1]) * g.power_scale;
        const int fb = f0 + c0 / 2;
        if (g.stage_out) {
          float4* d4 = reinterpret_cast<float4*>(my_out + lane * kStOutLd + c0 / 2);
          d4[0] = make_float4(pw[0], pw[1], pw[2], pw[3]);
          d4[1] = make_float4(pw[4], pw[5], pw[6], pw[7]);
        } else if (g.vec_p && fb + 7 < g.n_bins) {
          reinterpret_cast<float4*>(out)[0] = make_float4(pw[0], pw[1], pw[2], pw[3]);
          reinterpret_cast<float4*>(out)[1] = make_float4(pw[4], pw[5], pw[6], pw[7]);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (fb + j < g.n_bins) out[j] = pw[j];
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(b));   // the accumulator is free; the staged rows still have to go out
      if (g.stage_out && !(g.debug & 1)) {
        // 32 rows x 40 powers, written 16 bytes per lane with consecutive lanes on consecutive columns: a row's 160 bytes
        // leave in one piece instead of as ten 16-byte stores scattered over ten instructions.  The warp's 32 slots are
        // not 32 consecutive output rows (a stream's halo slots sit between streams): each staged row asks its own lane
        constexpr int kC4 = kStNPad / 8;   // 10 float4 per row
#pragma unroll
        for (int itr = 0; itr < kC4; ++itr) {
          const int idx = itr * 32 + lane;
          const int r = idx / kC4, c4 = idx - r * kC4;
          const long long grow = __shfl_sync(0xffffffffu, (long long)row, r);
          const int fbin = f0 + c4 * 4;
          if (grow >= 0 && fbin < g.n_bins) {
            const float4 val = *reinterpret_cast<const float4*>(my_out + r * kStOutLd + c4 * 4);
            float* out = g.P + grow * g.ldp + fbin;
            if (fbin + 3 < g.n_bins) {
              *reinterpret_cast<float4*>(out) = val;
            } else {
              out[0] = val.x;
              if (fbin + 1 < g.n_bins) out[1] = val.y;
              if (fbin + 2 < g.n_bins) out[2] = val.z;
            }
          }
        }
        __syncwarp();
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kStMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// hop rows of a tile and the 16-byte units between two slices of a stage: >= rows and = 2 (mod 4), so that the 8 lanes of
// a quarter-warp (2 rows x 4 slices) store to 8 different 16-byte bank groups
struct StftTcRing {
  int n_q, rows, slice_units;
  size_t bytes;
};
static StftTcRing stft_tc_ring(int n_k16, int h16) {
  StftTcRing r{};
  r.n_q = (n_k16 - 1) / h16 + 1;
  r.rows = kTcBM + r.n_q - 1;
  r.slice_units = r.rows + ((2 - r.rows % 4) + 4) % 4;
  r.bytes = (size_t)kStStages * 2 * kStSlices * r.slice_units * 16;
  return r;
}

struct StftTcShape {
  int kc, n_k16, n_ntiles;
  size_t tile_bytes, img_bytes, smem_bytes, stage_bytes;   // stage_bytes: optional output staging on top of smem_bytes
  bool ok;
};
// hop = 16 sizes the ring for the most hop rows a frame can span: a shape that is supported runs at every hop % 16 == 0
StftTcShape stft_tc_shape(int n_taps, int n_bins, int hop = 16) {
  StftTcShape s{};
  const int k_used = n_taps + kStLead;
  s.kc = (int)ceil_div(k_used, kTcBK);
  s.n_k16 = (int)ceil_div(k_used, 16);
  s.n_ntiles = (int)ceil_div(2 * n_bins, kStNPad);
  s.tile_bytes = (size_t)s.kc * kStTerms * kStNPad * 128;
  s.img_bytes = s.tile_bytes * s.n_ntiles;
  s.smem_bytes = s.tile_bytes + stft_tc_ring(s.n_k16, std::max(1, hop / 16)).bytes + 16 * 8;
  s.stage_bytes = (size_t)4 * 32 * kStOutLd * sizeof(float);
  s.ok = s.smem_bytes <= (size_t)kTcSmemBudget;
  return s;
}

}  // namespace vadx

using namespace vadx;

extern "C" int vadx_stft_tc_supported(int n_taps, int n_bins) { return stft_tc_shape(n_taps, n_bins).ok ? 1 : 0; }

// h_basis: the fp32 table of vadx_stft_power_f32 ([n_taps][ld_basis], re/im interleaved).  The loader
// feeds the operand pair (256*(x >> 8), x & 255) -- both exact in bf16 -- so one image per basis term
// serves both halves of the sample.
extern "C" int vadx_pack_stft_basis_tc(const float* h_basis, int ld_basis, int n_taps, int n_bins, double preemph,
                                       double scale, void* h_img, size_t img_capacity, size_t* img_bytes) {
  return vadx_pack_stft_basis_tc_fmt(h_basis, ld_basis, n_taps, n_bins, preemph, scale, VADX_TC_FMT_BF16, h_img, img_capacity,
                                     img_bytes);
}

extern "C" int vadx_pack_stft_basis_tc_fmt(const float* h_basis, int ld_basis, int n_taps, int n_bins, double preemph,
                                           double scale, int operand_format, void* h_img, size_t img_capacity,
                                           size_t* img_bytes) {
  VADX_REQUIRE(h_basis && img_bytes && n_taps > 0 && n_bins > 0 && ld_basis >= 2 * n_bins,
               "vadx_pack_stft_basis_tc: bad argument");
  VADX_REQUIRE(operand_format == VADX_TC_FMT_BF16 || operand_format == VADX_TC_FMT_F16, "vadx_pack_stft_basis_tc: operand format %d",
               operand_format);
  const bool f16 = operand_format == VADX_TC_FMT_F16;
  StftTcShape s = stft_tc_shape(n_taps, n_bins);
  VADX_REQUIRE(s.ok, "vadx_pack_stft_basis_tc: %d taps x %d bins does not fit the tensor-core DFT", n_taps, n_bins);
  *img_bytes = s.img_bytes;
  if (!h_img) return VADX_OK;
  VADX_REQUIRE(img_capacity >= s.img_bytes, "vadx_pack_stft_basis_tc: image buffer too small");
  uint8_t* img = static_cast<uint8_t*>(h_img);
  memset(img, 0, s.img_bytes);
  const int n_cols = 2 * n_bins;
  const size_t term = (size_t)kStNPad * 128;
  for (int col = 0; col < n_cols; ++col) {
    const int nt = col / kStNPad, r = col % kStNPad;
    for (int k = 0; k < n_taps + kStLead; ++k) {
      const int n0 = k - kStLead, n1 = k - kStLead + 1;  // y[n0] uses x[i] (+1), y[n1] uses x[i] (-c)
      double v = 0.0;
      if (n0 >= 0 && n0 < n_taps) v += (double)h_basis[(size_t)n0 * ld_basis + col];
      if (n1 >= 0 && n1 < n_taps) v -= preemph * (double)h_basis[(size_t)n1 * ld_basis + col];
      v *= scale;
      const float f = (float)v;
      const uint16_t b0 = f16 ? f16_rn_host(f) : bf16_rn_host(f);
      const float r1 = (float)(v - (double)(f16 ? f16_to_f_host(b0) : bf16_to_f_host(b0)));
      const uint16_t b1 = f16 ? f16_rn_host(r1) : bf16_rn_host(r1);
      const int c = k / kTcBK, kk = k % kTcBK;
      uint8_t* base = img + (size_t)nt * s.tile_bytes + (size_t)(c * kStTerms) * term + sw128_offset(r, kk);
      memcpy(base, &b0, 2);
      memcpy(base + term, &b1, 2);
    }
  }
  return VADX_OK;
}

// Folded-basis response to the DC term of a centre-padded, DC-removed frontend: with y[0] = x[0] - m and
// y[i] = (x[i] - m) - c (x[i-1] - m) = x[i] - c x[i-1] - (1 - c) m for 1 <= i < L, frame t of the mean alone is
// sum_n coef(t*hop - pad_left + n) * b[n][col], coef(0) = 1, coef(i) = 1 - c inside, 0 in the pad.
extern "C" int vadx_pack_stft_dc_tc(const float* h_basis, int ld_basis, int n_taps, int n_bins, double preemph, double scale,
                                    int64_t n_samples, int hop, int pad_left, int n_frames, float* h_tables,
                                    size_t capacity_floats, size_t* n_floats, int* n_edge_lo, int* t_edge_hi) {
  VADX_REQUIRE(h_basis && n_floats && n_edge_lo && t_edge_hi && n_taps > 0 && n_bins > 0 && hop > 0 && pad_left >= 0 &&
                   n_frames > 0 && ld_basis >= 2 * n_bins,
               "vadx_pack_stft_dc_tc: bad argument");
  StftTcShape s = stft_tc_shape(n_taps, n_bins);
  VADX_REQUIRE(s.ok, "vadx_pack_stft_dc_tc: shape not supported");
  // frame t is interior when every tap index lies in [1, n_samples)
  int lo = 0;
  while (lo < n_frames && (int64_t)lo * hop - pad_left < 1) ++lo;
  int hi = n_frames;
  while (hi > lo && (int64_t)(hi - 1) * hop - pad_left + n_taps - 1 >= n_samples) --hi;
  *n_edge_lo = lo;
  *t_edge_hi = hi;
  const int n_edge = lo + (n_frames - hi);
  const size_t ncp = (size_t)s.n_ntiles * kStNPad;
  *n_floats = (size_t)(1 + n_edge + (n_frames - hi)) * ncp;   // DC rows, then one tail row per right-edge frame
  if (!h_tables) return VADX_OK;
  VADX_REQUIRE(capacity_floats >= *n_floats, "vadx_pack_stft_dc_tc: table buffer too small");
  memset(h_tables, 0, *n_floats * sizeof(float));
  auto fill = [&](float* row, int64_t origin, bool interior) {
    for (int col = 0; col < 2 * n_bins; ++col) {
      double acc = 0.0;
      for (int n = 0; n < n_taps; ++n) {
        const int64_t i = origin + n;
        double coef = interior ? 1.0 - preemph : (i < 0 || i >= n_samples ? 0.0 : (i == 0 ? 1.0 : 1.0 - preemph));
        acc += coef * (double)h_basis[(size_t)n * ld_basis + col];
      }
      row[col] = (float)(acc * scale);
    }
  };
  fill(h_tables, 0, true);
  int e = 1;
  for (int t = 0; t < lo; ++t, ++e) fill(h_tables + (size_t)e * ncp, (int64_t)t * hop - pad_left, false);
  for (int t = hi; t < n_frames; ++t, ++e) fill(h_tables + (size_t)e * ncp, (int64_t)t * hop - pad_left, false);
  // tail rows: c * scale * b[n_L][col], n_L = tap index of sample L in frame t (zero row when outside the window)
  for (int t = hi; t < n_frames; ++t, ++e) {
    const int64_t n_l = n_samples - ((int64_t)t * hop - pad_left);
    if (n_l < 0 || n_l >= n_taps) continue;
    float* row = h_tables + (size_t)e * ncp;
    for (int col = 0; col < 2 * n_bins; ++col) row[col] = (float)(preemph * scale * (double)h_basis[(size_t)n_l * ld_basis + col]);
  }
  return VADX_OK;
}

namespace vadx {
__global__ void __launch_bounds__(256) stream_mean_i16_kernel(const int16_t* __restrict__ x, int64_t in_stride, int64_t n,
                                                              float* __restrict__ mean_frac, int* __restrict__ mean_int) {
  const int64_t s = blockIdx.x;
  const int16_t* p = x + s * in_stride;
  long long acc = 0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) acc += (long long)__ldg(p + i);
  __shared__ long long part[8];
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long t = 0;
    for (int w = 0; w < 8; ++w) t += part[w];
    const double m = (double)t / (double)n;
    const int mi = (int)llrint(m);
    mean_int[s] = mi;
    mean_frac[s] = (float)(m - (double)mi);
  }
}
}  // namespace vadx

extern "C" int vadx_stream_mean_i16(const int16_t* d_audio, int64_t in_stride, int64_t n_samples, int64_t n_streams,
                                    float* d_mean_frac, int32_t* d_mean_int, void* stream) {
  StageTimer _timer(VADX_STAGE_PREP, (cudaStream_t)stream, "stream_mean_i16_kernel", 2.0 * n_streams * n_samples);
  VADX_REQUIRE(d_audio && d_mean_frac && d_mean_int && n_samples > 0 && in_stride >= n_samples && n_streams >= 0,
               "vadx_stream_mean_i16: bad argument");
  if (n_streams == 0) return VADX_OK;
  stream_mean_i16_kernel<<<(unsigned)n_streams, 256, 0, (cudaStream_t)stream>>>(d_audio, in_stride, n_samples, d_mean_frac,
                                                                                d_mean_int);
  return after_launch("vadx_stream_mean_i16");
}

extern "C" int vadx_stft_power_tc_i16(const int16_t* d_audio, int64_t in_stride, int64_t n_samples, int64_t n_streams,
                                      int n_frames, int hop, int n_taps, const void* d_img, int n_bins, float* d_power,
                                      int64_t ld_power, void* stream) {
  VADX_REQUIRE((int64_t)(n_frames - 1) * hop + n_taps <= n_samples,
               "vadx_stft_power_tc_i16: frames must lie inside the %lld samples of a stream", (long long)n_samples);
  return vadx_stft_power_tc_i16_ex(d_audio, in_stride, n_samples, n_streams, n_frames, hop, n_taps, d_img, n_bins, d_power,
                                   ld_power, 0, nullptr, nullptr, nullptr, 0, n_frames, 1.0f, VADX_TC_FMT_BF16, stream);
}

extern "C" int vadx_stft_power_tc_i16_ex(const int16_t* d_audio, int64_t in_stride, int64_t n_samples, int64_t n_streams,
                                         int n_frames, int hop, int n_taps, const void* d_img, int n_bins, float* d_power,
                                         int64_t ld_power, int pad_left, const float* d_mean_frac, const int32_t* d_mean_int,
                                         const float* d_dc_tables, int n_edge_lo, int t_edge_hi, float power_scale,
                                         int operand_format, void* stream) {
  const float* d_mean = d_mean_frac;
  VADX_REQUIRE(operand_format == VADX_TC_FMT_BF16 || (operand_format == VADX_TC_FMT_F16 && !d_mean_frac),
               "vadx_stft_power_tc_i16: fp16 operands cannot carry the mean-removed (17-bit) samples");
  VADX_REQUIRE((d_mean_frac == nullptr) == (d_mean_int == nullptr), "vadx_stft_power_tc_i16: mean needs both its parts");
  StageTimer _timer(VADX_STAGE_STFT, (cudaStream_t)stream, "stft_power_tc_kernel",
                    2.0 * n_streams * n_samples + 4.0 * n_streams * n_frames * n_bins,      // int16 audio in, power out
                    2.0 * n_streams * n_frames * n_taps * 2.0 * n_bins);
  VADX_REQUIRE(d_audio && d_img && d_power, "vadx_stft_power_tc_i16: null pointer");
  VADX_REQUIRE(n_streams >= 0 && n_frames > 0 && hop > 0 && n_taps > 0 && n_bins > 0 && ld_power >= n_bins,
               "vadx_stft_power_tc_i16: bad shape");
  VADX_REQUIRE(in_stride >= n_samples && pad_left >= 0 && (pad_left % 8) == 0 && (n_samples % 8) == 0,
               "vadx_stft_power_tc_i16: stride shorter than the stream, or pad_left / n_samples not a multiple of 8");
  const bool leaves_stream = pad_left > 0 || (int64_t)(n_frames - 1) * hop - pad_left + n_taps > n_samples;
  VADX_REQUIRE(!(d_mean || leaves_stream) || (d_dc_tables && n_edge_lo >= 0 && t_edge_hi >= n_edge_lo && t_edge_hi <= n_frames),
               "vadx_stft_power_tc_i16: padded frames / DC removal need the tables of vadx_pack_stft_dc_tc");
  VADX_REQUIRE((hop % 16) == 0,
               "vadx_stft_power_tc_i16: hop %d is not a multiple of 16 samples (frames are read as shifted rows of 16-sample "
               "hop slices); use vadx_stft_power_f32", hop);
  VADX_REQUIRE((in_stride % 8) == 0 && aligned16(d_audio) && aligned16(d_img),
               "vadx_stft_power_tc_i16: stream stride must be a multiple of 8 samples, pointers 16-byte aligned");
  StftTcShape s = stft_tc_shape(n_taps, n_bins, hop);
  VADX_REQUIRE(s.ok, "vadx_stft_power_tc_i16: shape not supported");
  if (n_streams == 0) return VADX_OK;
  static PerDevice per_device;
  int n_sm = 148;
  VADX_TRY(per_device.ensure(&n_sm, [] {
    cudaError_t e = cudaSuccess;
    auto opt_in = [&](auto kern) {
      if (e == cudaSuccess) e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemBudget);
    };
    opt_in(stft_power_tc_kernel<false, false>);
    opt_in(stft_power_tc_kernel<true, false>);
    opt_in(stft_power_tc_kernel<false, true>);
    opt_in(stft_power_tc_kernel<true, true>);
    return e;
  }));
  const StftTcRing ring = stft_tc_ring(s.n_k16, hop / 16);
  StftTcArgs g{};
  g.X = d_audio; g.in_stride = in_stride; g.L = n_samples; g.S = n_streams; g.n_frames = n_frames; g.hop = hop;
  g.h16 = hop / 16; g.n_q = ring.n_q; g.tq = n_frames + ring.n_q - 1; g.rows = ring.rows; g.slice_units = ring.slice_units;
  g.n_st = (int)ceil_div(g.h16, kStJ);
  g.Wimg = static_cast<const uint8_t*>(d_img); g.P = d_power; g.ldp = ld_power;
  g.n_bins = n_bins; g.kc = s.kc; g.n_k16 = s.n_k16;
  g.pad_left = pad_left; g.mean = d_mean; g.mean_int = d_mean_int; g.dc = d_dc_tables; g.power_scale = power_scale; g.n_edge_lo = n_edge_lo; g.t_edge_hi = t_edge_hi;
  g.vec_p = ((ld_power & 3) == 0) && aligned16(d_power);
  {
    static const int dbg = ab_env("VADX_TC_DEBUG", 0);
    g.debug = dbg;
  }
  static const int opt = ab_env("VADX_ST_OPT", 2);   // bit 1 staged output
  {
    static const int bl = ab_env("VADX_TC_BACKOFF_LD", 64);
    static const int be = ab_env("VADX_TC_BACKOFF_EPI", 256);
    g.backoff_ld = (unsigned)bl; g.backoff_epi = (unsigned)be;
  }
  g.stage_out = ((opt & 2) && g.vec_p && s.smem_bytes + s.stage_bytes <= (size_t)kTcSmemBudget) ? 1 : 0;
  const size_t smem = s.smem_bytes + (g.stage_out ? s.stage_bytes : 0);
  // M rows are slots: each stream's frames and the Q - 1 halo slots behind them
  int64_t tiles = ceil_div(n_streams * g.tq, kTcBM);
  VADX_REQUIRE(tiles <= 0x7fffffffLL, "vadx_stft_power_tc_i16: too many rows");
  g.n_tiles = (int)tiles;
  int per = std::max(1, n_sm / s.n_ntiles);
  dim3 grid((unsigned)std::min<int64_t>(tiles, per), (unsigned)s.n_ntiles);
  const bool ex = leaves_stream || d_mean, f16 = operand_format == VADX_TC_FMT_F16;
  constexpr int kThreads = (kStLoaderWarps + 5) * 32;
  if (ex && f16) stft_power_tc_kernel<true, true><<<grid, kThreads, smem, (cudaStream_t)stream>>>(g);
  else if (ex) stft_power_tc_kernel<true, false><<<grid, kThreads, smem, (cudaStream_t)stream>>>(g);
  else if (f16) stft_power_tc_kernel<false, true><<<grid, kThreads, smem, (cudaStream_t)stream>>>(g);
  else stft_power_tc_kernel<false, false><<<grid, kThreads, smem, (cudaStream_t)stream>>>(g);
  return after_launch("vadx_stft_power_tc_i16");
}
