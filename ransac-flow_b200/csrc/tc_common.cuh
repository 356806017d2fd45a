// tcgen05 / TMEM / TMA building blocks shared by the tensor-core translation units (sm_100a): PTX wrappers,
// shared-memory matrix descriptors, instruction descriptors and the cached tensor-map encoder.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace rf {

constexpr int TC_THREADS = 192;
constexpr int TC_BK = 32;                 // fp32 elements per 128-byte swizzle row
constexpr int TC_BK_F16 = 64;             // fp16 elements per 128-byte swizzle row (engine 2)
template <bool F16> constexpr int tc_bk() { return F16 ? TC_BK_F16 : TC_BK; }
constexpr int TC_A_BYTES = 128 * 128;     // 128 rows x 128 B


// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// bounded wait: a lost arrival becomes a CUDA error (trap) instead of a hung GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    for (uint32_t spin = 0; !mbar_try_wait(bar, parity); ++spin)
        if (spin > (1u << 26)) __trap();
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(smem_u32(smem_dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(smem_dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"((uint64_t)map), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_store_commit_and_wait_read() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)map) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], TF32 operands, fp32 accumulate, M = 128, N from idesc
// Called by ALL 32 lanes of the (converged) MMA warp with warp-uniform operands; one elected lane issues.  Keeping the
// control flow and the descriptors warp-uniform lets the compiler hold them in uniform registers: issuing from a
// divergent `if (lane == 0)` branch cost ~14 SASS instructions (ELECT / R2UR.BROADCAST per operand) per MMA and made
// the single issuing thread, not the tensor pipe, the bottleneck (profiles/README.md).
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .pred e;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

// Four MMAs (the four K = 8 steps of one 32-wide, 128-byte-swizzled K block) from ONE elected lane with one
// elect.sync: descriptors advance by 32 bytes (+2 in the 16-byte address field) per step.  `acc_first` = 0 makes the
// first MMA overwrite the accumulator.
__device__ __forceinline__ void umma_tf32_x4(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc_first) {
    asm volatile(
        "{\n\t.reg .pred e, p, t;\n\t.reg .b64 a1, a2, a3, b1, b2, b3;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.eq.u32 t, 0, 0;\n\t"
        "add.u64 a1, %1, 2;\n\tadd.u64 a2, %1, 4;\n\tadd.u64 a3, %1, 6;\n\t"
        "add.u64 b1, %2, 2;\n\tadd.u64 b2, %2, 4;\n\tadd.u64 b3, %2, 6;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], a1, b1, %3, t;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], a2, b2, %3, t;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], a3, b3, %3, t;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc_first) : "memory");
}
// fp16 operands (engine 2): same 128-byte K block, now 64 channels = four K = 16 steps; 10-bit mantissa like TF32, half
// the bytes per element and twice the tensor rate
__device__ __forceinline__ void umma_f16_x4(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc_first) {
    asm volatile(
        "{\n\t.reg .pred e, p, t;\n\t.reg .b64 a1, a2, a3, b1, b2, b3;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.eq.u32 t, 0, 0;\n\t"
        "add.u64 a1, %1, 2;\n\tadd.u64 a2, %1, 4;\n\tadd.u64 a3, %1, 6;\n\t"
        "add.u64 b1, %2, 2;\n\tadd.u64 b2, %2, 4;\n\tadd.u64 b3, %2, 6;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, t;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], a2, b2, %3, t;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], a3, b3, %3, t;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc_first) : "memory");
}
template <bool F16>
__device__ __forceinline__ void umma_x4(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc_first) {
    if constexpr (F16) umma_f16_x4(tmem_d, adesc, bdesc, idesc, acc_first);
    else umma_tf32_x4(tmem_d, adesc, bdesc, idesc, acc_first);
}
// 3xTF32: per K step lo*hi, hi*lo, hi*hi (12 MMAs per K block)
__device__ __forceinline__ void umma_3xtf32_x4(uint32_t tmem_d, uint64_t ahi, uint64_t alo, uint64_t bhi, uint64_t blo, uint32_t idesc, uint32_t acc_first) {
    asm volatile(
        "{\n\t.reg .pred e, p, t;\n\t.reg .b64 ah, al, bh, bl;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "setp.eq.u32 t, 0, 0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], %2, %3, %5, p;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %4, %5, t;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %3, %5, t;\n\t"
        "add.u64 ah, %1, 2;\n\tadd.u64 al, %2, 2;\n\tadd.u64 bh, %3, 2;\n\tadd.u64 bl, %4, 2;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], al, bh, %5, t;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], ah, bl, %5, t;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], ah, bh, %5, t;\n\t"
        "add.u64 ah, %1, 4;\n\tadd.u64 al, %2, 4;\n\tadd.u64 bh, %3, 4;\n\tadd.u64 bl, %4, 4;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], al, bh, %5, t;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], ah, bl, %5, t;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], ah, bh, %5, t;\n\t"
        "add.u64 ah, %1, 6;\n\tadd.u64 al, %2, 6;\n\tadd.u64 bh, %3, 6;\n\tadd.u64 bl, %4, 6;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], al, bh, %5, t;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], ah, bl, %5, t;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], ah, bh, %5, t;\n\t}"
        ::"r"(tmem_d), "l"(ahi), "l"(alo), "l"(bhi), "l"(blo), "r"(idesc), "r"(acc_first) : "memory");
}
// fp16 split: x = hi + lo * 2^-11 with hi = fp16(x), lo = fp16((x - hi) * 2^11).  Per K = 16 step hi*hi accumulates into the
// main accumulator, lo*hi and hi*lo into the cross one (scaled by 2^11); the epilogue adds cross * 2^-11.  Same 22 significand
// bits as 3xTF32 at half the MMAs per channel.  The three products take TWO MMAs: the hi and lo B planes are adjacent in
// shared memory ([N rows hi][N rows lo], N * 128 bytes each) and the main and cross accumulators are adjacent in TMEM
// ([tmem_d, tmem_d + N) main, [tmem_d + N, tmem_d + 2N) cross):
//   A hi x [B hi | B lo]  as ONE N' = 2N instruction  -> main += hi*hi, cross += hi*lo
//   A lo x  B hi                                      -> cross += lo*hi
// A tcgen05.mma costs ~36 cycles + 0.62 cycles per column on B200 whatever its width (measured: N = 64 / 128 / 256 ->
// 75 / 131 / 194 cycles), so wider instructions are cheaper per MAC: 3 x 131 -> 194 + 131 cycles at N = 128.
__device__ __forceinline__ void umma_f16split2_x4(uint32_t tmem_d, uint32_t n, uint64_t ahi, uint64_t alo, uint64_t bhi,
                                                  uint32_t idesc_wide, uint32_t idesc, uint32_t acc_first) {
    asm volatile(
        "{\n\t.reg .pred e, p, t;\n\t.reg .b64 ah, al, bh;\n\t.reg .b32 tx;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "setp.eq.u32 t, 0, 0;\n\t"
        "add.u32 tx, %0, %1;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %2, %4, %5, p;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [tx], %3, %4, %7, t;\n\t"
        "add.u64 ah, %2, 2;\n\tadd.u64 al, %3, 2;\n\tadd.u64 bh, %4, 2;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], ah, bh, %5, t;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [tx], al, bh, %7, t;\n\t"
        "add.u64 ah, %2, 4;\n\tadd.u64 al, %3, 4;\n\tadd.u64 bh, %4, 4;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], ah, bh, %5, t;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [tx], al, bh, %7, t;\n\t"
        "add.u64 ah, %2, 6;\n\tadd.u64 al, %3, 6;\n\tadd.u64 bh, %4, 6;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], ah, bh, %5, t;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [tx], al, bh, %7, t;\n\t}"
        ::"r"(tmem_d), "r"(n), "l"(ahi), "l"(alo), "l"(bhi), "r"(idesc_wide), "r"(acc_first), "r"(idesc) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .pred e;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
        ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// shared-memory matrix descriptor: K-major tile, 128-byte swizzle, 8-row atoms 1024 B apart
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)(saddr >> 4);                      // start address, bits [0,14) (shared addresses are < 256 KB)
    d |= (uint64_t)1 << 16;                           // leading byte offset (unused for swizzled K-major), bits [16,30)
    d |= (uint64_t)(1024 >> 4) << 32;                 // stride byte offset between 8-row groups, bits [32,46)
    d |= (uint64_t)1 << 46;                           // descriptor version (Blackwell), bits [46,48)
    d |= (uint64_t)2 << 61;                           // layout type SWIZZLE_128B, bits [61,64)
    return d;
}
// instruction descriptor: D fp32, A/B TF32, both K-major, M = 128, N = n
__host__ __device__ constexpr uint32_t make_idesc_tf32(int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

// instruction descriptor: D fp32, A/B fp16 (format 0), both K-major, M = 128, N = n
__host__ __device__ constexpr uint32_t make_idesc_f16(int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
template <bool F16>
__host__ __device__ constexpr uint32_t make_idesc(int n) { return F16 ? make_idesc_f16(n) : make_idesc_tf32(n); }

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// two 32-column TMEM loads in flight, one wait
__device__ __forceinline__ void tmem_ld32x2(uint32_t t0, uint32_t (&a)[32], uint32_t t1, uint32_t (&b)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]), "=r"(a[4]), "=r"(a[5]), "=r"(a[6]), "=r"(a[7]),
          "=r"(a[8]), "=r"(a[9]), "=r"(a[10]), "=r"(a[11]), "=r"(a[12]), "=r"(a[13]), "=r"(a[14]), "=r"(a[15]),
          "=r"(a[16]), "=r"(a[17]), "=r"(a[18]), "=r"(a[19]), "=r"(a[20]), "=r"(a[21]), "=r"(a[22]), "=r"(a[23]),
          "=r"(a[24]), "=r"(a[25]), "=r"(a[26]), "=r"(a[27]), "=r"(a[28]), "=r"(a[29]), "=r"(a[30]), "=r"(a[31])
        : "r"(t0) : "memory");
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(b[0]), "=r"(b[1]), "=r"(b[2]), "=r"(b[3]), "=r"(b[4]), "=r"(b[5]), "=r"(b[6]), "=r"(b[7]),
          "=r"(b[8]), "=r"(b[9]), "=r"(b[10]), "=r"(b[11]), "=r"(b[12]), "=r"(b[13]), "=r"(b[14]), "=r"(b[15]),
          "=r"(b[16]), "=r"(b[17]), "=r"(b[18]), "=r"(b[19]), "=r"(b[20]), "=r"(b[21]), "=r"(b[22]), "=r"(b[23]),
          "=r"(b[24]), "=r"(b[25]), "=r"(b[26]), "=r"(b[27]), "=r"(b[28]), "=r"(b[29]), "=r"(b[30]), "=r"(b[31])
        : "r"(t1) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// cached cuTensorMapEncodeTiled (gemm_tc.cu): fp32 (esize 4) or fp16 (esize 2) tensor (d0 innermost, d1, d2[, d3]), dense strides
// except the outermost one of the 4-D form (`plane_bytes`), box of (b0, b1, b2[, b3]) ELEMENTS LOADED, traversal stride `es` on
// d1 / d2, 128-byte swizzle, zero fill out of bounds
int get_map(CUtensorMap* out, const void* ptr, unsigned long long d0, unsigned long long d1, unsigned long long d2,
            unsigned b0, unsigned b1, unsigned b2, unsigned es_ = 1, unsigned esize = 4);
int get_map4(CUtensorMap* out, const void* ptr, unsigned long long d0, unsigned long long d1, unsigned long long d2, unsigned long long d3,
             unsigned long long plane_bytes, unsigned b0, unsigned b1, unsigned b2, unsigned b3, unsigned es_, unsigned esize);
int pick_tw(int Ho, int Wo);

}  // namespace rf
