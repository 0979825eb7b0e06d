// tcgen05 / TMA / mbarrier PTX wrappers for sm_100a (hand-written; bit layouts follow the PTX ISA
// "tcgen05" matrix-descriptor / instruction-descriptor tables).
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---------------- mbarrier ----------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Spin on the phase parity.  A bounded spin: a protocol bug traps (context error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  uint32_t spins = 0;
  while (true) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
    if (++spins > (1u << 28)) __trap();
  }
}

// ---------------- TMA ----------------
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, "
      "%7}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

// ---------------- tcgen05 ----------------
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// whole warp; writes the TMEM base address to *slot (shared memory)
__device__ __forceinline__ void tmem_alloc(uint32_t slot_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// shared-memory matrix descriptor, K-major operand, swizzled rows of `row_bytes` (32/64/128):
//   bits [0,14)  start address >> 4         bits [16,30) leading byte offset >> 4 (unused for swizzled K-major)
//   bits [32,46) stride byte offset >> 4 (distance between 8-row groups)      bits [46,48) version = 1
//   bits [61,64) layout: 2 = SWIZZLE_128B, 4 = SWIZZLE_64B, 6 = SWIZZLE_32B
__device__ __forceinline__ uint64_t make_sdesc(uint32_t saddr, uint32_t row_bytes) {
  const uint32_t layout = row_bytes == 128 ? 2u : (row_bytes == 64 ? 4u : 6u);
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)((8u * row_bytes) >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout << 61;
  return d;
}

// instruction descriptor, both operands K-major, F32 accumulate
//   bits [4,6) D format (1 = F32)  [7,10) A format  [10,13) B format  [15] A major  [16] B major
//   bits [17,23) N >> 3            [24,29) M >> 4
//   A/B format: kind::f16 -> 1 = BF16;  kind::tf32 -> 2 = TF32
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// kind::f16 (BF16 operands); the accumulate flag is an immediate (no per-instruction setp in the issue loop)
template <int ACC>
__device__ __forceinline__ void mma_bf16_imm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "n"(ACC)
      : "memory");
}

// kind::tf32: fp32 containers in shared memory, the tensor core reads the TF32 bits (sign, 8-bit exponent, 10-bit
// mantissa); one instruction consumes K = 8 elements = 32 bytes per row, the same 32 bytes as 16 bf16
template <int ACC>
__device__ __forceinline__ void mma_tf32_imm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "n"(ACC)
      : "memory");
}

// element-type dispatch: T = __nv_bfloat16 (kind::f16) or float (kind::tf32); a 32-byte K slice per instruction
template <typename T> struct Mma;
template <> struct Mma<__nv_bfloat16> {
  static __host__ __device__ constexpr uint32_t idesc(int M, int N) { return make_idesc_bf16(M, N); }
  template <int ACC>
  static __device__ __forceinline__ void issue(uint32_t d, uint64_t a, uint64_t b, uint32_t id) {
    mma_bf16_imm<ACC>(d, a, b, id);
  }
};
template <> struct Mma<float> {
  static __host__ __device__ constexpr uint32_t idesc(int M, int N) { return make_idesc_tf32(M, N); }
  template <int ACC>
  static __device__ __forceinline__ void issue(uint32_t d, uint64_t a, uint64_t b, uint32_t id) {
    mma_tf32_imm<ACC>(d, a, b, id);
  }
};

// one K chunk: NMMA instructions over consecutive 32-byte slices of the A / B rows (descriptor address units of 16
// bytes); `first` starts the accumulator with the chunk's first instruction instead of adding to it
template <typename T, int NMMA>
__device__ __forceinline__ void mma_kchunk(uint32_t d, uint64_t da, uint64_t db, uint32_t idesc, bool first) {
  if (first) Mma<T>::template issue<0>(d, da, db, idesc);
  else Mma<T>::template issue<1>(d, da, db, idesc);
#pragma unroll
  for (int k = 1; k < NMMA; ++k) Mma<T>::template issue<1>(d, da + 2 * k, db + 2 * k, idesc);
}

// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// TMEM -> registers: this warp's 32 lanes x 16 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
      "[%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// split form for software pipelining: issue the load of the next 16 columns, process the previous ones, then
// wait; the wait names the destination registers so the compiler cannot hoist their uses above it
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
      "[%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait16(uint32_t* r) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}

// after one tmem_ld_wait16: ties further destination arrays of loads issued before that wait to the wait's position
// (asm volatile statements keep their order), so their uses cannot be scheduled above it
__device__ __forceinline__ void tmem_ld_dep16(uint32_t* r) {
  asm volatile(""
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}

}  // namespace tc
