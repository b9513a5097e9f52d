// tc_ptx.cuh -- inline-PTX building blocks shared by the tcgen05 kernels: mbarrier, bulk async copy,
// UMMA shared-memory / instruction descriptors, tcgen05.mma / commit / ld, bf16 splitting.
#pragma once
#include "common.cuh"

namespace vadx {

constexpr int kTcBM = 128;                       // UMMA M (rows of a tile)
constexpr int kTcBK = 64;                        // K chunk = one 128-byte swizzle atom of bf16
constexpr int kTcTileBytes = kTcBM * 128;        // one 128-row x 64-k bf16 tile
constexpr int kTcSmemBudget = 227 * 1024;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// bounded wait: a protocol bug becomes a trap (an error the host sees), never a hung GPU
// backoff_ns > 0: the polling warp sleeps between probes instead of competing for issue slots with the
// warps it is waiting for (loader / epilogue waits; the single MMA thread polls tightly)
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, unsigned backoff_ns = 0) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (backoff_ns) __nanosleep(backoff_ns);
    if (clock64() - t0 > 20000000000LL) __trap();
  }
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// shared -> global bulk copy, tracked by the issuing thread's bulk async-group (commit_group / wait_group[.read])
__device__ __forceinline__ void bulk_s2g(void* dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}

__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);  // start address, 16-byte units
  d |= (uint64_t)1 << 16;                        // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;              // stride byte offset: 8-row atoms are 1024 B apart
  d |= (uint64_t)1 << 46;                        // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                        // SWIZZLE_128B
  return d;
}
// no-swizzle K-major operand: 8 x 16-byte core matrices, rows 16 B apart inside one; lbo = bytes between the two 8-element
// halves of a K = 16 step, sbo = bytes between consecutive 8-row groups.  The start address only needs 16-byte alignment,
// so an operand can begin any number of rows into a run of back-to-back core matrices (sbo = 128)
__device__ __forceinline__ uint64_t umma_desc_noswz(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);  // start address, 16-byte units
  d |= (uint64_t)((lbo >> 4) & 0x3FFFu) << 16;   // leading byte offset: the next 8 elements along K
  d |= (uint64_t)((sbo >> 4) & 0x3FFFu) << 32;   // stride byte offset: the next 8 rows
  d |= (uint64_t)1 << 46;                        // descriptor version (sm_100); layout type 0 (no swizzle) in bits 61-63
  return d;
}
// kind::f16, A = B = bf16, D = fp32, both K-major, M = 128
__device__ __forceinline__ uint32_t umma_idesc_bf16(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTcBM >> 4) << 24);
}
// kind::f16, A = B = fp16, D = fp32
__device__ __forceinline__ uint32_t umma_idesc_f16(int n) {
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTcBM >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Up to four K=16 steps of one 64-wide K chunk in a single asm block: the operand descriptors advance by 32 bytes
// (2 in the descriptors' 16-byte address units) per step, the accumulate predicate is built once.  The issuing
// thread spends ~12 instructions per chunk instead of ~10 per MMA -- with N = 80 an MMA occupies the tensor core for
// only 40 cycles, so the issue rate of that one thread matters.
__device__ __forceinline__ void umma_k64(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate_first, int n_steps) {
  asm volatile(
      "{\n"
      ".reg .pred p0, pt, q1, q2, q3;\n"
      ".reg .b64 a1, a2, a3, b1, b2, b3;\n"
      "setp.ne.b32 p0, %4, 0;\n"
      "setp.eq.b32 pt, 0, 0;\n"
      "setp.gt.s32 q1, %5, 1;\n"
      "setp.gt.s32 q2, %5, 2;\n"
      "setp.gt.s32 q3, %5, 3;\n"
      "add.u64 a1, %1, 2;\n"
      "add.u64 a2, %1, 4;\n"
      "add.u64 a3, %1, 6;\n"
      "add.u64 b1, %2, 2;\n"
      "add.u64 b2, %2, 4;\n"
      "add.u64 b3, %2, 6;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p0;\n"
      "@q1 tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, pt;\n"
      "@q2 tcgen05.mma.cta_group::1.kind::f16 [%0], a2, b2, %3, pt;\n"
      "@q3 tcgen05.mma.cta_group::1.kind::f16 [%0], a3, b3, %3, pt;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate_first), "r"(n_steps)
      : "memory");
}
// two MMAs into one accumulator that share the B operand (the hi and lo terms of a split A operand), one predicate
__device__ __forceinline__ void umma_x2(uint32_t tmem_d, uint64_t adesc0, uint64_t adesc1, uint64_t bdesc, uint32_t idesc,
                                        uint32_t accumulate_first) {
  asm volatile(
      "{\n.reg .pred p, pt;\n"
      "setp.ne.b32 p, %5, 0;\n"
      "setp.eq.b32 pt, 0, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %3, %4, p;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %2, %3, %4, pt;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc0), "l"(adesc1), "l"(bdesc), "r"(idesc), "r"(accumulate_first)
      : "memory");
}
// Up to three K=16 MMA pairs of a split A operand (hi at a, lo at a + a_lo) in one asm block: pair i reads A at
// a + i * a_step and B at b_i, so one column of a shifted-row operand is issued with its descriptor deltas added
// inside the block (the issuing thread's instruction rate bounds short MMAs, see umma_k64).  n_pairs in 1..3; the
// first MMA accumulates iff accumulate_first; lo_on = 0 drops the lo terms (a measurement switch).
__device__ __forceinline__ void umma_split_x3(uint32_t tmem_d, uint64_t a, uint32_t a_step, uint32_t a_lo, uint64_t b0,
                                              uint64_t b1, uint64_t b2, uint32_t idesc, uint32_t accumulate_first,
                                              int n_pairs, uint32_t lo_on) {
  asm volatile(
      "{\n"
      ".reg .pred p0, pt, q1, q2, l0, l1, l2;\n"
      ".reg .b64 st, lo, a0h, a1, a1h, a2, a2h;\n"
      "setp.ne.b32 p0, %7, 0;\n"
      "setp.eq.b32 pt, 0, 0;\n"
      "setp.gt.s32 q1, %8, 1;\n"
      "setp.gt.s32 q2, %8, 2;\n"
      "setp.ne.b32 l0, %9, 0;\n"
      "and.pred l1, l0, q1;\n"
      "and.pred l2, l0, q2;\n"
      "cvt.u64.u32 st, %2;\n"
      "cvt.u64.u32 lo, %3;\n"
      "add.u64 a0h, %1, lo;\n"
      "add.u64 a1, %1, st;\n"
      "add.u64 a1h, a1, lo;\n"
      "add.u64 a2, a1, st;\n"
      "add.u64 a2h, a2, lo;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %4, %6, p0;\n"
      "@l0 tcgen05.mma.cta_group::1.kind::f16 [%0], a0h, %4, %6, pt;\n"
      "@q1 tcgen05.mma.cta_group::1.kind::f16 [%0], a1, %5, %6, pt;\n"
      "@l1 tcgen05.mma.cta_group::1.kind::f16 [%0], a1h, %5, %6, pt;\n"
      "@q2 tcgen05.mma.cta_group::1.kind::f16 [%0], a2, %10, %6, pt;\n"
      "@l2 tcgen05.mma.cta_group::1.kind::f16 [%0], a2h, %10, %6, pt;\n"
      "}\n" ::"r"(tmem_d),
      "l"(a), "r"(a_step), "r"(a_lo), "l"(b0), "l"(b1), "r"(idesc), "r"(accumulate_first), "r"(n_pairs), "r"(lo_on),
      "l"(b2)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// Split TMEM load: issue now, use later.  The destination registers are only valid after tmem_ld8_finish, which takes
// them as read-write operands so that no use can be scheduled above the wait.
__device__ __forceinline__ void tmem_ld8_issue(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8_finish(uint32_t* r) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7])
               :
               : "memory");
}

// 8 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

// 32 consecutive fp32 columns of this thread's TMEM lane, one wait for both halves
// bulk L2 prefetch (no destination, no completion): p 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void l2_prefetch(const void* p, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

// 256-bit read-only global load (sm_100: LDG.E.256); p must be 32-byte aligned
__device__ __forceinline__ void ldg256_nc(const float* p, float4& a, float4& b) {
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
               : "l"(p));
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// two floats -> packed (hi, lo) bf16x2 words: hi = rn(x), lo = rn(x - hi)
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));  // upper half <- b, lower half <- a
  float ah = __uint_as_float(hi << 16), bh = __uint_as_float(hi & 0xffff0000u);
  float al = a - ah, bl = b - bh;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(bl), "f"(al));
}


// host-side bf16 helpers (round to nearest even)
static inline uint16_t bf16_rn_host(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7f800000u) == 0x7f800000u) return (uint16_t)(u >> 16);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
static inline float bf16_to_f_host(uint16_t h) {
  uint32_t u = (uint32_t)h << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
// IEEE half, round to nearest even (subnormals included)
static inline uint16_t f16_rn_host(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  const uint32_t sign = (u >> 16) & 0x8000u;
  const int32_t exp = (int32_t)((u >> 23) & 0xffu) - 127 + 15;
  uint32_t man = u & 0x7fffffu;
  if (((u >> 23) & 0xffu) == 0xffu) return (uint16_t)(sign | 0x7c00u | (man ? 0x200u : 0u));
  if (exp >= 31) return (uint16_t)(sign | 0x7c00u);
  if (exp <= 0) {
    if (exp < -10) return (uint16_t)sign;
    man |= 0x800000u;
    const int shift = 14 - exp;                       // 14..24
    uint32_t h = man >> shift;
    const uint32_t rem = man & ((1u << shift) - 1u), halfway = 1u << (shift - 1);
    if (rem > halfway || (rem == halfway && (h & 1u))) ++h;
    return (uint16_t)(sign | h);
  }
  uint32_t h = ((uint32_t)exp << 10) | (man >> 13);
  const uint32_t rem = man & 0x1fffu;
  if (rem > 0x1000u || (rem == 0x1000u && (h & 1u))) ++h;   // may carry into the exponent: still correct
  return (uint16_t)(sign | h);
}
static inline float f16_to_f_host(uint16_t h) {
  const uint32_t sign = (uint32_t)(h & 0x8000u) << 16;
  const uint32_t exp = (h >> 10) & 0x1fu, man = h & 0x3ffu;
  float f;
  if (exp == 0) {
    f = ldexpf((float)man, -24);
    uint32_t u;
    memcpy(&u, &f, 4);
    u |= sign;
    memcpy(&f, &u, 4);
    return f;
  }
  const uint32_t u = exp == 31 ? (sign | 0x7f800000u | (man << 13)) : (sign | ((exp - 15 + 127) << 23) | (man << 13));
  memcpy(&f, &u, 4);
  return f;
}
// byte offset of element (row r, k) inside a K-major, 128-byte-swizzled tile of 64 k-columns
static inline size_t sw128_offset(int r, int kk) {
  return (size_t)(r / 8) * 1024 + (size_t)(r % 8) * 128 + (size_t)(((kk / 8) ^ (r % 8)) * 16) + (size_t)(kk % 8) * 2;
}

}  // namespace vadx
