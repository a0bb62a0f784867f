// Inline PTX for sm_100a (tcgen05, TMA, mbarrier, thread-block clusters) and the operand formats of the tensor-core
// kernels.  Every asm statement of csrc/*.cu lives here, one function per instruction form, named after the PTX.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace sg {

// ---- shared memory ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
// Bytes to skip for 1024-byte alignment (the 128B swizzle atom): `smem_raw + smem_pad1024(smem_raw)`.  Keep the addition on
// the __shared__ array itself: an integer round trip, or even a helper that returns the aligned pointer, makes the compiler
// lose the address space and demote shared-memory accesses to generic LD/ST.
__device__ __forceinline__ uint32_t smem_pad1024(const void* smem_raw) {
  return (1024u - (smem_u32(smem_raw) & 1023u)) & 1023u;
}

// ---- mbarrier ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbarrier_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbarrier_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbarrier_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbarrier_inval(uint64_t* bar) {
  asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_mbarrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

// Parity waits.  After 2^kSpinLog2 unsuccessful polls the kernel traps: a lost arrival must fail, not hang the GPU.
template <int kSpinLog2>
__device__ __forceinline__ void mbarrier_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0;
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (spin > (1u << kSpinLog2)) __trap();
  }
}
// for a barrier completed by st.async stores of OTHER CTAs of the cluster: acquire at cluster scope
template <int kSpinLog2>
__device__ __forceinline__ void mbarrier_wait_acquire_cluster(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0;
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (spin > (1u << kSpinLog2)) __trap();
  }
}

// ---- TMA and bulk copies ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// multicast to every CTA of `mask` (same CTA-relative smem offset and mbarrier in each)
__device__ __forceinline__ void tma_load_2d_multicast(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                                      uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}
__device__ __forceinline__ void bulk_load_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// ---- thread-block cluster ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive_release() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void cluster_wait_acquire() {
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same variable in CTA `rank`
__device__ __forceinline__ uint32_t mapa_shared_cluster(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// 16-byte remote store that signals its bytes on the destination CTA's mbarrier when it lands
__device__ __forceinline__ void st_async_v4(uint32_t remote_addr, uint4 v, uint32_t remote_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];"
               ::"r"(remote_addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(remote_bar)
               : "memory");
}

// ---- named barrier ----------------------------------------------------------------------------------------------------
template <int kId, int kThreads>
__device__ __forceinline__ void bar_sync() {
  asm volatile("bar.sync %0, %1;" ::"n"(kId), "n"(kThreads) : "memory");
}

// ---- tcgen05: tensor memory, fences, issue ----------------------------------------------------------------------------
__device__ __forceinline__ void tcgen05_alloc(uint32_t* slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tcgen05_relinquish_alloc_permit() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (TMA, tensor core)
__device__ __forceinline__ void fence_proxy_async_shared() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ uint32_t elect_one_sync() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred;
}

// D (+)= A B^T with A and B from shared-memory descriptors; `acc` = 0 overwrites D
__device__ __forceinline__ void tcgen05_mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                 uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void tcgen05_mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
// A from tensor memory
__device__ __forceinline__ void tcgen05_mma_f16_tmem_a(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                                       uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
// arrive on `bar` once every MMA this thread issued so far has completed
__device__ __forceinline__ void tcgen05_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// ... on the barrier at the same offset in every CTA of `mask`
__device__ __forceinline__ void tcgen05_commit_multicast(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(mask)
               : "memory");
}

// ---- tcgen05: tensor memory <-> registers (thread = TMEM lane) --------------------------------------------------------
__device__ __forceinline__ void tcgen05_ld_32x32b_x16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tcgen05_ld_32x32b_x32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tcgen05_st_32x32b_x8(uint32_t taddr, uint4 a, uint4 b) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"r"(taddr), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
               : "memory");
}
__device__ __forceinline__ void tcgen05_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- UMMA descriptors -------------------------------------------------------------------------------------------------
// layout type of a K-major shared-memory operand: rows of 128 (64) bytes, 16-byte granules XOR-swizzled by row % 8
enum UmmaSwizzle : uint32_t { UMMA_SWIZZLE_128B = 2, UMMA_SWIZZLE_64B = 4 };
// K-major swizzled operand tile; `sbo` = byte distance of consecutive 8-row groups (8 x the row bytes for a dense tile)
constexpr __host__ __device__ uint64_t umma_desc_kmajor(uint32_t smem_addr, uint32_t sbo, UmmaSwizzle swizzle) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFFu)      // start address                     bits [0,14)
         | (uint64_t)1 << 16                          // leading byte offset (unused for swizzled K-major)
         | (uint64_t)(sbo >> 4) << 32                 // stride byte offset                bits [32,46)
         | (uint64_t)1 << 46                          // descriptor version (sm_100)
         | (uint64_t)swizzle << 61;                   // layout type                       bits [61,64)
}
// A / B element format of the instruction descriptor (kind::f16: F16 or BF16; kind::tf32: TF32)
enum UmmaFormat : uint32_t { UMMA_F16 = 0, UMMA_BF16 = 1, UMMA_TF32 = 2 };
// instruction descriptor: fp32 accumulate, A and B K-major, M = 128, N = n
constexpr __host__ __device__ uint32_t umma_idesc_m128(UmmaFormat ab, int n) {
  return (1u << 4) | ((uint32_t)ab << 7) | ((uint32_t)ab << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

// ---- operand formats --------------------------------------------------------------------------------------------------
// fp32 -> 16-bit operand image(s).  fp16: hi = fp16(sat(x)), lo = fp16(sat(x) - hi), unscaled (absolute error <= 2^-25,
// |x| saturated to the fp16 maximum 65504);  bf16: hi = bf16(x), lo = 0.  The GLU chain (glu_h.cu) reads these images, and
// the graph-Fourier epilogue (spec_tc.cu) writes them for it.  `bf16` stays an int: that epilogue passes its runtime flag,
// and a bool parameter changes the code generated for it.
__device__ __forceinline__ void split_f16_hi_lo(float x, int bf16, unsigned short& hi, unsigned short& lo) {
  if (bf16) {
    hi = __bfloat16_as_ushort(__float2bfloat16_rn(x));
    lo = 0;
  } else {
    const float xs = fminf(fmaxf(x, -65504.f), 65504.f);
    const __half h = __float2half_rn(xs);
    hi = __half_as_ushort(h);
    lo = __half_as_ushort(__float2half_rn(xs - __half2float(h)));
  }
}
// The GRU's scaled split: x = hi + lo / F16_LO_SCALE with hi, lo in fp16 (lo pre-scaled by 2^11 so that it stays in the
// normal range; 22 significant bits)
constexpr float F16_LO_SCALE = 2048.0f;
__device__ __forceinline__ void split_f16_hi_lo_scaled(float x, unsigned short& hi, unsigned short& lo) {
  const __half h = __float2half_rn(x);
  hi = __half_as_ushort(h);
  lo = __half_as_ushort(__float2half_rn((x - __half2float(h)) * F16_LO_SCALE));
}

// Fast gate nonlinearities (ex2.approx + approximate division: ~2 ulp, abs error < 3e-7 on the gates)
__device__ __forceinline__ float fast_sigmoid(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float fast_tanh(float x) { return 2.0f * fast_sigmoid(2.0f * x) - 1.0f; }

}  // namespace sg
