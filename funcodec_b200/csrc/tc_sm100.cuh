// sm_100a tensor-core primitives used by the implicit-GEMM conv and the RVQ distance kernels:
// mbarrier, tcgen05 (alloc / mma kind::tf32 / commit / ld), UMMA shared-memory and instruction descriptors,
// 1-D bulk async copies (cp.async.bulk, the TMA engine without a tensor map).
//
// Bit layouts follow the PTX ISA "tcgen05 matrix descriptor" / "instruction descriptor" tables (the same
// fields CUTLASS exposes as cute::UMMA::SmemDescriptor / InstrDescriptor).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace fcb {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ------------------------------------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) { }
}
// Same, with a back-off between polls: for waiters that are NOT on the critical path (a spinning warp still takes
// issue slots away from the producer warps of its SM sub-partition).
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity, unsigned ns) {
    while (!mbar_try_wait(bar, parity)) { __nanosleep(ns); }
}

// generic-proxy writes (st.shared by threads) -> visible to the async proxy (tcgen05.mma / bulk copies)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ bulk copy (TMA engine, 1-D)
// global -> shared, completion signalled on an mbarrier (complete_tx::bytes).  16-byte aligned, size % 16 == 0.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// TMA tensor load (cp.async.bulk.tensor, SASS UTMALDG): a 4-D box of the tensor described by `tmap` (a CUtensorMap passed as a
// __grid_constant__ kernel parameter) -> dense shared-memory tile, completion on an mbarrier (complete_tx::bytes).
// Out-of-bounds coordinates are zero-filled by the hardware.
__device__ __forceinline__ void tma_load_4d(void* dst_smem, const void* tmap, int c0, int c1, int c2, int c3, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
            smem_u32(dst_smem)),
        "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

// ------------------------------------------------------------------------------------------------ tcgen05
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {   // one full warp; ncols pow2 >= 32
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {      // same warp that allocated
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, kind::tf32, issued by ONE thread.
__device__ __forceinline__ void mma_tf32_ss(uint32_t d_tmem, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// kind::f16 (fp16 operands, fp32 accumulate): K = 16 per instruction
__device__ __forceinline__ void mma_f16_ss(uint32_t d_tmem, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// all previously issued MMAs of this thread -> arrive on the mbarrier when they have completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// TMEM -> registers: 32 lanes x 32 columns of 32-bit (one warp reads its own 32-lane slice)
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
// registers -> TMEM (same shape as tmem_ld_32x32b_x32)
__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
        "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]),
        "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]),
        "r"(v[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ descriptors
// K-major operand tile in the canonical SWIZZLE_128B layout: rows of 128 bytes (32 tf32), 8-row groups
// 1024 bytes apart (SBO), 16-byte chunk index XOR (row & 7).  `addr` = shared address of row 0 (+ k*32 bytes to
// step along K inside the 128-byte row).  The row-0 address may be any multiple of 128 bytes inside a slab whose
// base is 1024-byte aligned and that was written with chunk ^= (absolute_row & 7): tap-shifted views.
__device__ __forceinline__ uint64_t make_desc_k_sw128(uint32_t addr) {
    uint64_t d = 0;
    d |= (uint64_t)((addr & 0x3FFFFu) >> 4);            // [0,14)  start address >> 4
    d |= (uint64_t)1 << 16;                              // [16,30) leading byte offset (unused for swizzled K-major) = 1
    d |= (uint64_t)(1024 >> 4) << 32;                    // [32,46) stride byte offset = 1024 B between 8-row groups
    d |= (uint64_t)1 << 46;                              // [46,48) descriptor version = 1 (sm_100)
    // [49,52) base offset = 0: measured on B200 -- the 128B swizzle XOR is taken from the ABSOLUTE shared-memory
    // address bits [7,10), so a view that starts r rows into a 1024-byte-aligned slab needs no phase correction
    // (setting base_offset = r & 7 double-corrects and scrambles the operand).
    d |= (uint64_t)2 << 61;                              // [61,64) layout type: SWIZZLE_128B
    return d;
}
// byte offset of element (row, col) (col in tf32 elements, < 32) inside a SWIZZLE_128B K-major slab whose row 0
// sits at a 1024-byte aligned address
__device__ __forceinline__ uint32_t sw128_offset(uint32_t row, uint32_t col) {
    return row * 128u + ((((col >> 2) ^ (row & 7u)) << 4) | ((col & 3u) << 2));
}

// kind::tf32 instruction descriptor: D fp32, A/B tf32, both K-major, dense, no negate.
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N) {
    return (1u << 4)                      // c_format = F32
           | (2u << 7)                    // a_format = TF32
           | (2u << 10)                   // b_format = TF32
           | (0u << 15) | (0u << 16)      // a_major = K, b_major = K
           | ((uint32_t)(N >> 3) << 17)   // n_dim
           | ((uint32_t)(M >> 4) << 24);  // m_dim
}

// kind::f16 instruction descriptor: D fp32, A/B fp16 (format 0), both K-major, dense, no negate.
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
    return (1u << 4)                      // c_format = F32
           | (0u << 7)                    // a_format = F16
           | (0u << 10)                   // b_format = F16
           | (0u << 15) | (0u << 16)      // a_major = K, b_major = K
           | ((uint32_t)(N >> 3) << 17)   // n_dim
           | ((uint32_t)(M >> 4) << 24);  // m_dim
}

// FP16 split of two (pre-scaled) fp32 values: hi = fp16(x) round-to-nearest, lo = fp16(x - hi) (x - hi is exact in fp32);
// element 0 in the low half.  Saturating conversions: |x| beyond the fp16 range clamps instead of producing inf.
__device__ __forceinline__ void split_f16x2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));
    float f0, f1;
    asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %2;\n\tcvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, h;\n\t}" : "=f"(f0), "=f"(f1) : "r"(hi));
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(x1 - f1), "f"(x0 - f0));
}
__device__ __forceinline__ float exp2f_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// 3xTF32 split: hi = x with the low 13 mantissa bits cleared after round-to-nearest on the tf32 grid,
// lo = x - hi (exact in fp32); the tensor core ignores lo's bits below tf32 precision.
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
    uint32_t u = __float_as_uint(x);
    u = (u + 0x1000u) & 0xFFFFE000u;       // round half up in magnitude on the 10-bit-mantissa grid
    hi = __uint_as_float(u);
    lo = x - hi;
}

}  // namespace tc
}  // namespace fcb
