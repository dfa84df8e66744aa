// Inline-PTX wrappers for the sm_100a tensor-core path: mbarrier, TMA (cp.async.bulk[.tensor]), tcgen05
// (alloc / mma / commit / ld) and the UMMA shared-memory / instruction descriptors.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace sb
{
namespace ptx
{
__device__ __forceinline__ uint32_t smem_u32(const void * p)
{
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one()
{
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---- explicit shared-state-space accesses (keeps the compiler from falling back to generic LD/ST) ----
__device__ __forceinline__ float4 lds128(uint32_t addr)
{
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float2 lds64(uint32_t addr)
{
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts32(uint32_t addr, float v)
{
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}

__device__ __forceinline__ void sts64(uint32_t addr, float2 v)
{
  asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t addr, float4 v)
{
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float lds32(uint32_t addr)
{
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}

// ---- mbarrier ----
__device__ __forceinline__ void mbar_init(uint64_t * bar, uint32_t count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init()
{
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t * bar, uint32_t bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t * bar)
{
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t * bar, uint32_t parity)
{
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// non-blocking test (try_wait may suspend the thread for a system-dependent time when the phase is not complete, so a
// thread that polls several barriers uses this one)
__device__ __forceinline__ bool mbar_test_wait(uint64_t * bar, uint32_t parity)
{
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol error becomes a trap (cudaErrorLaunchFailure) instead of a hung GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t * bar, uint32_t parity)
{
  uint32_t spins = 0;
  while(!mbar_try_wait(bar, parity))
  {
    if(++spins > (1u << 26)) __trap();
  }
}

// The same operations on a 32-bit shared-memory address computed once (a generic pointer costs a cvta sequence of ~8
// uniform-datapath instructions at every use: measurable in single-thread issue loops and per-sub-batch epilogues).
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity)
{
  uint32_t spins = 0, ok;
  do
  {
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if(!ok && ++spins > (1u << 26)) __trap();
  } while(!ok);
}
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar)
{
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_a(uint32_t bar, uint32_t bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load_1d_a(uint32_t smem_dst, const void * gmem_src, uint32_t bytes, uint32_t bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :
               : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(gmem_src)), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void tc_commit_a(uint32_t bar)
{
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// ---- TMA ----
__device__ __forceinline__ void prefetch_tensormap(const void * tmap)
{
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
// 2-D tiled load: coordinates (c0 = inner / K element index, c1 = row)
__device__ __forceinline__ void tma_load_2d(void * smem_dst, const void * tmap, int c0, int c1, uint64_t * bar)
{
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               :
               : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
               : "memory");
}
// 1-D bulk copy global -> shared (bytes % 16 == 0, both addresses 16-byte aligned)
__device__ __forceinline__ void bulk_load_1d(void * smem_dst, const void * gmem_src, uint32_t bytes, uint64_t * bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :
               : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gmem_src)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// 1-D bulk copy shared -> global (bytes % 16 == 0, both addresses 16-byte aligned), tracked by the issuing
// thread's bulk async-group; the writer must fence_proxy_async() its st.shared before the copy is issued
__device__ __forceinline__ void bulk_store_1d(void * gmem_dst, uint32_t smem_src, uint32_t bytes)
{
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               :
               : "l"(reinterpret_cast<uint64_t>(gmem_dst)), "r"(smem_src), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit()
{
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// waits until at most kPending of this thread's bulk groups still READ their shared-memory source
template<int kPending>
__device__ __forceinline__ void bulk_wait_read()
{
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kPending) : "memory");
}

// ---- tcgen05 ----
template<int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t * smem_result)
{
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template<int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr)
{
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before()
{
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after()
{
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// arrives (count 1) on `bar` once every tcgen05.mma issued so far by this thread has completed
__device__ __forceinline__ void tc_commit(uint64_t * bar)
{
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// D[tmem] (+)= A[smem] . B[smem]^T ; both operands K-major.  kTf32: kind::tf32 (K = 8 per instruction), else
// kind::f16 (bf16 inputs, K = 16).  fp32 accumulation in TMEM.
template<bool kTf32>
__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
  if constexpr(kTf32)
  {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
  else
  {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}

// 32 lanes x 8 consecutive 32-bit columns: thread t of the warp gets TMEM lane (lane_base + t), columns col .. col + 7
__device__ __forceinline__ void tmem_ld_x8(uint32_t taddr, float (&v)[8])
{
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
#pragma unroll
  for(int i = 0; i < 8; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_x2(uint32_t taddr, float (&v)[2])
{
  uint32_t r[2];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(taddr));
  v[0] = __uint_as_float(r[0]), v[1] = __uint_as_float(r[1]);
}
__device__ __forceinline__ void tmem_ld_x8p(uint32_t taddr, float * v)
{
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
#pragma unroll
  for(int i = 0; i < 8; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_x4(uint32_t taddr, float (&v)[4])
{
  uint32_t r[4];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(taddr));
#pragma unroll
  for(int i = 0; i < 4; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, float * v)
{
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
#pragma unroll
  for(int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
}
// 32 lanes x 16 consecutive 32-bit columns, registers -> TMEM (thread t writes lane (lane_base + t))
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t (&r)[16])
{
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      :
      : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait()
{
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// D[tmem] (+)= A[tmem] . B[smem]^T, kind::f16: A is an M x 16 fp16 tile in TMEM (row i in lane i, two K elements per
// 32-bit column: 8 columns per instruction), B is K-major in shared memory.
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_f16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// the same two instructions with the shared-memory descriptors given as (constant high word, address >> 4): the
// single issuing thread then spends one integer add per operand instead of rebuilding 64-bit descriptors
template<int kRowBytes>
__host__ __device__ constexpr uint32_t smem_desc_hi()
{
  static_assert(kRowBytes == 32 || kRowBytes == 64 || kRowBytes == 128, "row = one swizzle span");
  return static_cast<uint32_t>((8 * kRowBytes) >> 4) | (1u << 14) | ((kRowBytes == 128 ? 2u : kRowBytes == 64 ? 4u : 6u) << 29);
}
__device__ __forceinline__ void umma_f16_ss_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc,
                                               uint32_t accumulate)
{
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 da, {%1, %3};\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_f16_ts_lo(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc,
                                               uint32_t accumulate)
{
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// instruction descriptor for kind::f16 with FP16 inputs (a/b format 0), fp32 accumulate, K-major A and B
__host__ __device__ constexpr uint32_t make_idesc_f16(int m, int n)
{
  return (1u << 4) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
__device__ __forceinline__ void tmem_ld_wait()
{
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// UMMA instruction descriptor (upper 32 bits of the 64-bit runtime descriptor): fp32 accumulate, K-major A and B.
//   bits [4,6) c format (1 = F32) | [7,10) a format | [10,13) b format (1 = BF16, 2 = TF32) | 15/16 majors (0 = K)
//   | [17,23) N >> 3 | [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc(bool tf32, int m, int n)
{
  return (1u << 4) | ((tf32 ? 2u : 1u) << 7) | ((tf32 ? 2u : 1u) << 10) | (static_cast<uint32_t>(n >> 3) << 17)
         | (static_cast<uint32_t>(m >> 4) << 24);
}

// UMMA shared-memory matrix descriptor for a K-major tile whose rows are exactly one swizzle span wide
// (32 B -> SWIZZLE_32B, 64 B -> SWIZZLE_64B, 128 B -> SWIZZLE_128B): 8-row atoms are contiguous, SBO = 8 * row bytes,
// LBO unused.
//   bits [0,14) address >> 4 | [16,30) LBO >> 4 | [32,46) SBO >> 4 | [46,48) version = 1 | [61,64) layout type
template<int kRowBytes>
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr)
{
  static_assert(kRowBytes == 32 || kRowBytes == 64 || kRowBytes == 128, "row = one swizzle span");
  constexpr uint64_t layout = kRowBytes == 128 ? 2 : kRowBytes == 64 ? 4 : 6;
  constexpr uint64_t sbo = (8 * kRowBytes) >> 4;
  return static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4) | (sbo << 32) | (1ull << 46) | (layout << 61);
}
} // namespace ptx
} // namespace sb
