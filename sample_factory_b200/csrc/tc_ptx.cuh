// tcgen05 / TMA / mbarrier PTX wrappers, UMMA descriptors and compile-time activations shared by the GEMM engine
// (gemm_tc.cu) and the persistent rollout kernel (rollout_fused.cu).  sm_100a only.
#pragma once
#include <cuda.h>
#include <cudaTypedefs.h>

#include "common.cuh"

namespace sfb {

constexpr int TBM = 128;        // tile rows  (UMMA M, cta_group::1)
constexpr int TBK = 32;         // k per stage: 32 fp32 = 128 B = one swizzle row
constexpr int UMMA_K = 8;       // tf32
constexpr int TC_THREADS = 448;   // TMA, MMA, 4 split warps, 8 epilogue warps

// ------------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// 1024-byte aligned start inside the dynamic shared-memory window (the 128B swizzle atoms need it).  Plain pointer
// arithmetic on the __shared__ array -- NOT a round trip through uintptr_t, which makes the compiler forget the address
// space and emit generic LD.E / ST.E for every shared-memory access derived from it.
__device__ __forceinline__ uint8_t* smem_align_1024(uint8_t* raw) {
    return raw + ((1024u - (smem_u32(raw) & 1023u)) & 1023u);
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra.uni WAIT_DONE;\n"
        "bra.uni WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc], kind::tf32, issued by ONE thread
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
// D[tmem] (+)= A[tmem] * B[smem desc]: the A operand is read from tensor memory (rows = TMEM lanes, k = 32-bit columns)
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// kind::f16 (fp16 operands, fp32 accumulate), A from tensor memory: two K elements per 32-bit TMEM column
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// kind::f16, both operands from shared memory
__device__ __forceinline__ void umma_f16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
        "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
        "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
template <int N>
__device__ __forceinline__ void tmem_st_cols(uint32_t taddr, const uint32_t (&r)[N]) {
    static_assert(N == 16 || N == 32, "16 or 32 consecutive TMEM columns per thread");
    if constexpr (N == 32) tmem_st_32x32b_x32(taddr, r);
    else tmem_st_32x32b_x16(taddr, r);
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ descriptors
// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) |
// version=1 [46,48) | layout type [61,64).
//   K-major  tile [rows][32 fp32], SWIZZLE_128B (type 2, 16 B chunks XOR row%8): 128 B rows, 8-row atoms 1024 B apart
//            -> SBO = 1024, LBO unused (1)
//   MN-major tile = boxes of [32 k][32 rows] (4096 B each, k rows 128 B apart).  For 32-bit MN-major operands the only
//            legal layout is SWIZZLE_128B_BASE32B (type 1: 32 B chunks XOR k%4, atom = 4 k-rows = 512 B; CUTLASS
//            sm100_common.inl:92 "for mn-major tf32 operands, SW128_32B is the only available smem layout"), written by
//            TMA with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B  -> LBO = 4096 (next 32 rows), SBO = 512 (next 4 k)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, bool mn_major) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
    d |= (uint64_t)(mn_major ? (4096u >> 4) : 1u) << 16;
    d |= (uint64_t)((mn_major ? 512u : 1024u) >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)(mn_major ? 1 : 2) << 61;
    return d;
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32=1 [4,6) | a/b_format TF32=2 [7,10)/[10,13) |
// a_major [15] | b_major [16] | N>>3 [17,23) | M>>4 [24,29)
__host__ __device__ constexpr uint32_t make_idesc(bool a_mn, bool b_mn, int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// kind::f16 instruction descriptor: a/b format F16 = 0, c format F32 = 1, both operands K-major
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

template <int ACT>
__device__ __forceinline__ float act_fwd_ct(float z) {
    if (ACT == SFB200_ACT_ELU) {
        // __expf(z) - 1 for z <= 0, computed unconditionally: __expf is ex2.approx(z * log2(e)) plus a rescaling branch for
        // results below 2^-126, which (e - 1) rounds to -1 either way -- same bits, half the instructions, no predication
        float e;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z * 1.4426950216293334961f));
        return z > 0.f ? z : e - 1.f;
    }
    if (ACT == SFB200_ACT_RELU) return fmaxf(z, 0.f);
    if (ACT == SFB200_ACT_TANH) return tanhf(z);
    return z;
}
template <int ACT>
__device__ __forceinline__ float act_bwd_ct(float h) {
    if (ACT == SFB200_ACT_ELU) return h > 0.f ? 1.f : h + 1.f;
    if (ACT == SFB200_ACT_RELU) return h > 0.f ? 1.f : 0.f;
    if (ACT == SFB200_ACT_TANH) return 1.f - h * h;
    return 1.f;
}

// host side (gemm_tc.cu): driver entry point for cuTensorMapEncodeTiled resolved at run time; 2-D fp32 tensor maps with
// the 128B swizzle (16 B chunks for K-major tiles, 32 B chunks for MN-major). dim0 = contiguous dimension.
bool tc_init();
bool make_tmap(CUtensorMap* out, const float* base, uint64_t dim0, uint64_t dim1, uint64_t stride1_elems, uint32_t box0,
               uint32_t box1, bool mn_major);
// 2-D fp16 tensor map, K-major rows of 64 halfs = 128 B, 128B swizzle
bool make_tmap_f16(CUtensorMap* out, const uint16_t* base, uint64_t dim0, uint64_t dim1, uint64_t stride1_elems, uint32_t box0,
                   uint32_t box1);

}  // namespace sfb
