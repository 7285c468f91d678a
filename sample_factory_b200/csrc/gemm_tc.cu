// tcgen05 / TMA GEMM engine for sm_100a (SFB200_GEMM_TC_3XTF32, SFB200_GEMM_TC_TF32).
//
//   C[m,n] = epilogue( sum_k A(m,k) * B(n,k) ),   fp32 in HBM, fp32 accumulate in TMEM.
//
// Precision: tcgen05 has no fp32 MMA. kind::tf32 keeps 10 mantissa bits, so a single pass is ~1e-3 relative -- not
// parity grade.  The 3xTF32 mode splits every operand element in shared memory into  hi = a & ~0x1fff  (exactly
// representable in tf32) and  lo = (a - hi) & ~0x1fff  and issues  hi*hi'  into one TMEM accumulator and
// hi*lo' + lo*hi'  into a second one (summed in the epilogue): each product is exact in fp32, the dropped lo*lo' term is
// 2^-22 relative, i.e. fp32-grade results.  (Two accumulators because the tensor core accumulates with truncation: keeping
// the 2^-11 smaller cross terms apart removes 2/3 of the roundings applied to the large partial sums -- measured 2.7e-5
// -> 9.8e-6 max error on a K=512 GEMM.)
//
// PERSISTENT kernel, one CTA per SM, 448 threads, static round-robin tile schedule (128 x BN output tiles):
//   warp 0      : TMA producer   (cp.async.bulk.tensor, 128B-swizzled boxes, mbarrier complete_tx), runs ahead across tiles
//   warp 1      : TMEM allocator + MMA issuer (one elected lane issues tcgen05.mma, tcgen05.commit frees the stage)
//   warps 2..5  : operand split: raw fp32 tile -> hi (in place) + lo (second buffer), fence.proxy.async, arrive
//   warps 6..13 : epilogue: tcgen05.ld both accumulators -> release the TMEM slot -> bias/activation -> global.
//                 The accumulator is double-buffered in TMEM, so the epilogue of tile i overlaps the main loop of tile i+1.
// Operands may be K-major ([rows, K], K contiguous) or MN-major ([K, rows], rows contiguous): the backward GEMMs
// (dX = dZ.W, dW = dZ^T.X) read the activations in the layout the forward pass wrote them -- no transposed copies.
// Split-K tiles write raw partial sums to a workspace that the SIMT engine's fixed-order reduce kernel sums.
#include <cuda.h>

#include <cstdlib>
#include <cudaTypedefs.h>

#include "common.cuh"
#include "gemm.h"
#include "tc_ptx.cuh"

namespace sfb {

// Passed to the kernels as a __grid_constant__ parameter: the epilogue reads its fields from the parameter bank where it
// uses them.  A by-value copy gets promoted into registers for the whole persistent tile loop, which makes the
// 128-register epilogue warps spill more (ptxas -v).
struct TcEpilogue {
    int mode;            // 0 plain, 1 act(acc + bias[n]), 2 acc * act'(aux[m,n])
    int act;
    const float* bias;
    const float* aux;
    int64_t ld_aux;
    // fused policy/value heads (mode 1 only): partial dot products of the activated output row with [Wv ; Wa] over this
    // thread's 64 columns -> head_part[(n_tile*2 + half)][m][kHeadPad]; C may be NULL (output row not stored)
    const float* head_wv;
    const float* head_wa;
    int head_A;
    float* head_part;
    // fused column sums of the OUTPUT (bias gradient of the previous layer = sum over rows of dX): one partial row per
    // (128-row tile, 32-row warp quadrant) -> colsum_part[(m_tile*4 + quadrant)][N]; requires M % 128 == 0, N % 128 == 0
    float* colsum_part;
};

constexpr int kHeadAP = 9;     // value + up to 8 action outputs
constexpr int kHeadPad = 12;   // floats per (partial, row): three 16 B stores

template <int BN, int STAGES>
struct TcSmem {
    // [stage][A hi | A lo | B hi | B lo]; every buffer is a multiple of 1024 B (swizzle-atom aligned)
    static constexpr int A_BYTES = TBM * TBK * 4;
    static constexpr int B_BYTES = BN * TBK * 4;
    static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
    static constexpr int NUM_BARS = 3 * STAGES + 4;
    static constexpr int BIAS_FLOATS = 2048;   // bias staged in smem when N <= this
    static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 512 /*barriers + tmem slot*/ + BIAS_FLOATS * 4;
};

// ELU via the fast exponential: |error| <= ~2.4e-7 absolute (2 ulp of exp on [0,1]) -- inside the 1e-5 parity budget;
// expm1f costs ~4x more instructions in the epilogue, which is the critical path of short-K tiles.
__device__ __forceinline__ float act_fwd_fast(float z, int act) {
    if (act == SFB200_ACT_ELU) return z > 0.f ? z : (__expf(z) - 1.f);
    return act_fwd(z, act);
}

// 256-bit global accesses (sm_100 LDG/STG.256): a lane of the epilogue owns a whole row segment, so a warp-wide 128-bit
// store touches 32 different 128 B lines with half a sector each -- every 32 B sector was written twice (ncu: 2x the
// ideal sector count on the store path, the limiter of the short-K layers).  One 32 B store per lane = one full sector.
__device__ __forceinline__ void st_global_v8(float* p, float a0, float a1, float a2, float a3, float a4, float a5, float a6,
                                             float a7) {
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(a0), "f"(a1), "f"(a2), "f"(a3), "f"(a4),
                 "f"(a5), "f"(a6), "f"(a7)
                 : "memory");
}
__device__ __forceinline__ void ld_global_v8(const float* p, float4& lo, float4& hi) {
    asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(lo.x), "=f"(lo.y), "=f"(lo.z), "=f"(lo.w), "=f"(hi.x), "=f"(hi.y), "=f"(hi.z), "=f"(hi.w)
                 : "l"(p));
}

// one output row segment (BN columns, fully in bounds, 16 B aligned) with the epilogue resolved at compile time
template <int MODE, int ACT, int BN>
__device__ __forceinline__ void write_row(float (&acc)[BN], float* __restrict__ dst, const float* bias_n0,
                                          const float4 (&auxv)[BN / 4], bool v8) {
#pragma unroll
    for (int j = 0; j < BN; j += 8) {
        float4 o[2];
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
            const int jj = j + 4 * hf;
            o[hf] = make_float4(acc[jj], acc[jj + 1], acc[jj + 2], acc[jj + 3]);
            if (MODE == 1) {
                if (bias_n0) {
                    const float4 b = *reinterpret_cast<const float4*>(bias_n0 + jj);   // shared (staged) or global
                    o[hf].x += b.x; o[hf].y += b.y; o[hf].z += b.z; o[hf].w += b.w;
                }
                o[hf].x = act_fwd_ct<ACT>(o[hf].x); o[hf].y = act_fwd_ct<ACT>(o[hf].y);
                o[hf].z = act_fwd_ct<ACT>(o[hf].z); o[hf].w = act_fwd_ct<ACT>(o[hf].w);
            } else if (MODE == 2) {
                const float4 h = auxv[jj / 4];
                o[hf].x *= act_bwd_ct<ACT>(h.x); o[hf].y *= act_bwd_ct<ACT>(h.y);
                o[hf].z *= act_bwd_ct<ACT>(h.z); o[hf].w *= act_bwd_ct<ACT>(h.w);
            }
        }
        if (v8) {
            st_global_v8(dst + j, o[0].x, o[0].y, o[0].z, o[0].w, o[1].x, o[1].y, o[1].z, o[1].w);
        } else {
            *reinterpret_cast<float4*>(dst + j) = o[0];
            *reinterpret_cast<float4*>(dst + j + 4) = o[1];
        }
        // keep the final values: the fused column-sum reduction reads them
        acc[j] = o[0].x; acc[j + 1] = o[0].y; acc[j + 2] = o[0].z; acc[j + 3] = o[0].w;
        acc[j + 4] = o[1].x; acc[j + 5] = o[1].y; acc[j + 6] = o[1].z; acc[j + 7] = o[1].w;
    }
}

// Sum 32 per-lane values over the 32 lanes of the warp so that lane j ends up with the total of v[j]: a transposing
// butterfly, 16 + 8 + 4 + 2 + 1 = 31 shuffles instead of 32 x 5.  (Fixed order -> deterministic.)
__device__ __forceinline__ float warp_transpose_sum32(float (&v)[32], int lane) {
#pragma unroll
    for (int half = 16; half >= 1; half >>= 1) {
        const bool upper = (lane & half) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const float send = upper ? v[i] : v[i + half];
            const float keep = upper ? v[i + half] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
        }
    }
    return v[0];
}

struct TileCoord {
    int64_t m0;
    int n0, k_begin, num_kb, z;
};

__device__ __forceinline__ TileCoord tile_coord(int tile, int tiles_n, int tiles_per_z, int BN, int K, int k_chunk) {
    TileCoord t;
    t.z = tile / tiles_per_z;
    const int r = tile - t.z * tiles_per_z;
    const int mb = r / tiles_n;
    t.m0 = (int64_t)mb * TBM;
    t.n0 = (r - mb * tiles_n) * BN;
    t.k_begin = t.z * k_chunk;
    const int k_end = (t.k_begin + k_chunk < K) ? t.k_begin + k_chunk : K;
    t.num_kb = (k_end - t.k_begin + TBK - 1) / TBK;
    return t;
}

struct EpiCtx {
    int lane_base, lane, col0, mode;
    bool vec_ok, aux_vec, bias_vec, st_v8, aux_v8;
    const float* bias_base;
    float out_scale;     // fp16-split engine: 2^-(operand shifts); 1 otherwise
};

// Epilogue warps 6..13: warp w may touch TMEM lanes [32*(w%4), 32*(w%4)+32); warps 6..9 take columns [0, BN/2) of their
// lane quadrant, warps 10..13 take [BN/2, BN).  One warp per scheduler was latency-bound (ncu: the epilogue warps were
// ~100% busy at IPC 0.12 and paced the whole kernel for short-K tiles).  The bias for ALL N columns is staged once per
// kernel in shared memory (persistent CTA).
template <int BN, int EPI_WARP0 = 6>
__device__ __forceinline__ EpiCtx make_epi_ctx(int warp, int lane, const float* C, int64_t ldc, int N, int splits,
                                               const TcEpilogue& epi, float* bias_s, int bias_floats) {
    EpiCtx ec;
    ec.lane_base = (warp & 3) * 32;
    ec.lane = lane;
    ec.col0 = ((warp - EPI_WARP0) >> 2) * (BN / 2);
    ec.vec_ok = (ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(C) & 15u) == 0);
    ec.aux_vec = epi.aux && (epi.ld_aux % 4 == 0) && ((reinterpret_cast<uintptr_t>(epi.aux) & 15u) == 0);
    ec.st_v8 = (ldc % 8 == 0) && ((reinterpret_cast<uintptr_t>(C) & 31u) == 0);
    ec.aux_v8 = epi.aux && (epi.ld_aux % 8 == 0) && ((reinterpret_cast<uintptr_t>(epi.aux) & 31u) == 0);
    const bool bias_smem = epi.bias != nullptr && N <= bias_floats;
    if (bias_smem) {
        for (int i = threadIdx.x - EPI_WARP0 * 32; i < N; i += 256) bias_s[i] = epi.bias[i];
        asm volatile("bar.sync 1, 256;" ::: "memory");
    }
    ec.bias_base = bias_smem ? bias_s : epi.bias;
    ec.bias_vec = epi.bias && (bias_smem || ((reinterpret_cast<uintptr_t>(epi.bias) & 15u) == 0));
    ec.mode = splits == 1 ? epi.mode : 0;
    ec.out_scale = 1.f;
    return ec;
}

// Whole accumulator row segment of this thread (CH columns, main + cross terms summed) -> registers, then the TMEM slot
// is handed back at once: all of the epilogue's arithmetic and global traffic overlaps the next tile's main loop (the
// TMEM-A kernel has a single accumulator slot, so whatever runs before the release is serialised with the MMAs).
// F16 (fp16-split engine): the cross columns hold the two hi x lo terms scaled by 2^11, and everything carries the
// operands' power-of-two shifts: acc = (main + cross * 2^-11) * out_scale, exact scalings.
template <int BN, int CH, bool SPLIT3, bool F16 = false>
__device__ __forceinline__ void tmem_drain(uint32_t t_main, float (&acc)[CH], uint64_t* acc_full_bar, uint32_t acc_ph,
                                           uint64_t* acc_empty_bar, float out_scale = 1.f) {
    mbar_wait(acc_full_bar, acc_ph);
    tc_fence_after();
#pragma unroll
    for (int c0 = 0; c0 < CH; c0 += 16) {
        uint32_t r[16];
        tmem_ld_32x32b_x16(t_main + (uint32_t)c0, r);
        if (SPLIT3) {
            uint32_t r2[16];
            tmem_ld_32x32b_x16(t_main + (uint32_t)(BN + c0), r2);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                if (F16) acc[c0 + j] = fmaf(__uint_as_float(r2[j]), 1.f / 2048.f, __uint_as_float(r[j])) * out_scale;
                else acc[c0 + j] = __uint_as_float(r[j]) + __uint_as_float(r2[j]);
            }
        } else {
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) acc[c0 + j] = __uint_as_float(r[j]);
        }
    }
    tc_fence_before();
    mbar_arrive(acc_empty_bar);
}

// One output tile: TMEM accumulator slot (main at column 0, cross terms at column BN) -> registers -> global.
template <int BN, bool SPLIT3, bool F16 = false>
__device__ __forceinline__ void tc_epilogue_tile(uint32_t tmem_slot_addr, uint64_t* acc_full_bar, uint32_t acc_ph,
                                                 uint64_t* acc_empty_bar, const TileCoord& tc, const EpiCtx& ec,
                                                 float* __restrict__ C, int64_t ldc, int64_t M, int N, int splits,
                                                 const TcEpilogue& epi) {
    constexpr int CH = BN / 2;                      // columns per thread
    const int lane_base = ec.lane_base, lane = ec.lane, col0 = ec.col0, mode = ec.mode;
    const bool vec_ok = ec.vec_ok, aux_vec = ec.aux_vec, bias_vec = ec.bias_vec;
    const float* bias_base = ec.bias_base;
    const int64_t m = tc.m0 + lane_base + lane;
    const int nbeg = tc.n0 + col0;
    const bool fast = (m < M) && (nbeg + CH <= N) && vec_ok &&
                      (mode == 0 || (mode == 1 && (bias_vec || !epi.bias)) || (mode == 2 && aux_vec));
    // mode 2: the activation-derivative operand of the first 32-column chunk is fetched BEFORE the accumulator is ready
    // (hides its HBM latency behind the main loop of this tile).
    const float* aux_row = (mode == 2 && fast) ? epi.aux + m * epi.ld_aux + nbeg : nullptr;
    float4 auxv[8];
    const bool aux_v8 = ec.aux_v8, st_v8 = ec.st_v8 && splits == 1;
    if (aux_row) {
        if (aux_v8) {
#pragma unroll
            for (int j = 0; j < 8; j += 2) ld_global_v8(aux_row + 4 * j, auxv[j], auxv[j + 1]);
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) auxv[j] = *reinterpret_cast<const float4*>(aux_row + 4 * j);
        }
    }
    float acc_all[CH];
    tmem_drain<BN, CH, SPLIT3, F16>(tmem_slot_addr + ((uint32_t)lane_base << 16) + (uint32_t)col0, acc_all, acc_full_bar, acc_ph,
                                    acc_empty_bar, ec.out_scale);
    if (m >= M) return;
    float* Cz = C + (splits > 1 ? (int64_t)tc.z * M * ldc : 0);
    float* dst_row = Cz + m * ldc + nbeg;
#pragma unroll
    for (int c0 = 0; c0 < CH; c0 += 32) {
        float (&acc)[32] = reinterpret_cast<float (&)[32]>(acc_all[c0]);
        if (c0 > 0 && aux_row) {
            if (aux_v8) {
#pragma unroll
                for (int j = 0; j < 8; j += 2) ld_global_v8(aux_row + c0 + 4 * j, auxv[j], auxv[j + 1]);
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) auxv[j] = *reinterpret_cast<const float4*>(aux_row + c0 + 4 * j);
            }
        }
        float* dst = dst_row + c0;
        if (fast) {
            // whole row segment in bounds, 128-bit everything; mode / activation resolved once per chunk into
            // a straight-line specialisation (a per-element switch cost 4x the instructions)
            const float* bias_n0 = epi.bias ? bias_base + nbeg + c0 : nullptr;
            if (mode == 1) {
                switch (epi.act) {
                    case SFB200_ACT_ELU: write_row<1, SFB200_ACT_ELU, 32>(acc, dst, bias_n0, auxv, st_v8); break;
                    case SFB200_ACT_RELU: write_row<1, SFB200_ACT_RELU, 32>(acc, dst, bias_n0, auxv, st_v8); break;
                    case SFB200_ACT_TANH: write_row<1, SFB200_ACT_TANH, 32>(acc, dst, bias_n0, auxv, st_v8); break;
                    default: write_row<1, SFB200_ACT_NONE, 32>(acc, dst, bias_n0, auxv, st_v8); break;
                }
            } else if (mode == 2) {
                switch (epi.act) {
                    case SFB200_ACT_ELU: write_row<2, SFB200_ACT_ELU, 32>(acc, dst, bias_n0, auxv, st_v8); break;
                    case SFB200_ACT_RELU: write_row<2, SFB200_ACT_RELU, 32>(acc, dst, bias_n0, auxv, st_v8); break;
                    case SFB200_ACT_TANH: write_row<2, SFB200_ACT_TANH, 32>(acc, dst, bias_n0, auxv, st_v8); break;
                    default: write_row<0, SFB200_ACT_NONE, 32>(acc, dst, bias_n0, auxv, st_v8); break;
                }
            } else {
                write_row<0, SFB200_ACT_NONE, 32>(acc, dst, bias_n0, auxv, st_v8);
            }
            if (epi.colsum_part) {   // (host guarantees full tiles: every lane of the warp is here)
                const float cs = warp_transpose_sum32(acc, lane);
                epi.colsum_part[((tc.m0 >> 5) + (lane_base >> 5)) * (int64_t)N + nbeg + c0 + lane] = cs;
            }
        } else {
#pragma unroll   // fully unrolled so that acc[] stays in registers (no dynamic indexing)
            for (int j = 0; j < 32; ++j) {
                const int n = nbeg + c0 + j;
                if (n < N) {
                    float v = acc[j];
                    if (mode == 1) v = act_fwd_fast(v + (epi.bias ? epi.bias[n] : 0.f), epi.act);
                    else if (mode == 2) v = v * act_bwd_from_out(epi.aux[m * epi.ld_aux + n], epi.act);
                    dst[j] = v;
                }
            }
        }
    }
}

// Epilogue with the policy/value heads folded in (forward layers feeding critic_linear / distribution_linear,
// actor_critic.py:171-186): y = act(acc + bias) is formed in registers, optionally stored, and immediately contracted
// with the (A+1) head weight rows staged in shared memory -- the separate heads kernel's re-read of y (4*N bytes per
// row) disappears, and in the sampler y is not written at all.  16-column chunks keep the live set (16 + 16 accumulator
// words, 9 partial sums) inside the 128-register budget.
template <int BN, bool SPLIT3, int ACT, bool F16 = false>
__device__ __forceinline__ void tc_epilogue_tile_heads(uint32_t tmem_slot_addr, uint64_t* acc_full_bar, uint32_t acc_ph,
                                                       uint64_t* acc_empty_bar, const TileCoord& tc, const EpiCtx& ec,
                                                       float* __restrict__ C, int64_t ldc, int64_t M, int N,
                                                       const TcEpilogue& epi, const float* __restrict__ headw_s) {
    constexpr int CH = BN / 2;
    const int64_t m = tc.m0 + ec.lane_base + ec.lane;
    const int nbeg = tc.n0 + ec.col0;
    float o[CH];
    tmem_drain<BN, CH, SPLIT3, F16>(tmem_slot_addr + ((uint32_t)ec.lane_base << 16) + (uint32_t)ec.col0, o, acc_full_bar, acc_ph,
                                    acc_empty_bar, ec.out_scale);
    if (m >= M) return;
    float hp[kHeadAP];
#pragma unroll
    for (int a = 0; a < kHeadAP; ++a) hp[a] = 0.f;
    float* dst_row = C ? C + m * ldc + nbeg : nullptr;
    const float* bias_n0 = ec.bias_base + nbeg;   // staged in shared memory (host guarantees N <= BIAS_FLOATS)
#pragma unroll
    for (int j = 0; j < CH; j += 8) {
#pragma unroll
        for (int jj = j; jj < j + 8; jj += 4) {
            const float4 b = *reinterpret_cast<const float4*>(bias_n0 + jj);
            o[jj] = act_fwd_ct<ACT>(o[jj] + b.x);
            o[jj + 1] = act_fwd_ct<ACT>(o[jj + 1] + b.y);
            o[jj + 2] = act_fwd_ct<ACT>(o[jj + 2] + b.z);
            o[jj + 3] = act_fwd_ct<ACT>(o[jj + 3] + b.w);
        }
        if (dst_row) {
            if (ec.st_v8) {
                st_global_v8(dst_row + j, o[j], o[j + 1], o[j + 2], o[j + 3], o[j + 4], o[j + 5], o[j + 6], o[j + 7]);
            } else {
                *reinterpret_cast<float4*>(dst_row + j) = make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]);
                *reinterpret_cast<float4*>(dst_row + j + 4) = make_float4(o[j + 4], o[j + 5], o[j + 6], o[j + 7]);
            }
        }
    }
#pragma unroll
    for (int a = 0; a < kHeadAP; ++a) {
        const float* w = headw_s + a * N + nbeg;   // warp-uniform address: shared-memory broadcast
        float s0 = 0.f, s1 = 0.f;                  // two chains per output: halves the dependent-FMA latency
#pragma unroll
        for (int j = 0; j < CH; j += 4) {
            const float4 wv = *reinterpret_cast<const float4*>(w + j);
            s0 = fmaf(o[j], wv.x, s0);
            s1 = fmaf(o[j + 1], wv.y, s1);
            s0 = fmaf(o[j + 2], wv.z, s0);
            s1 = fmaf(o[j + 3], wv.w, s1);
        }
        hp[a] = s0 + s1;
    }
    const int p = (tc.n0 / BN) * 2 + (ec.col0 ? 1 : 0);
    float4* dst = reinterpret_cast<float4*>(epi.head_part + ((int64_t)p * M + m) * kHeadPad);
    dst[0] = make_float4(hp[0], hp[1], hp[2], hp[3]);
    dst[1] = make_float4(hp[4], hp[5], hp[6], hp[7]);
    dst[2] = make_float4(hp[8], 0.f, 0.f, 0.f);
}

// ------------------------------------------------------------------------------------------------ the kernel
template <bool A_MN, bool B_MN, int BN, int STAGES, bool SPLIT3>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               float* __restrict__ C, int64_t ldc, int64_t M, int N, int K, int k_chunk, int splits,
               const __grid_constant__ TcEpilogue epi) {
    using S = TcSmem<BN, STAGES>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_align_1024(smem_raw);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * S::STAGE_BYTES);
    uint64_t* full = bars;                      // TMA bytes landed             (count 1 + tx)
    uint64_t* conv = bars + STAGES;             // operands split & visible      (count 128)
    uint64_t* empty = bars + 2 * STAGES;        // MMAs reading the stage done   (count 1, tcgen05.commit)
    uint64_t* acc_full = bars + 3 * STAGES;     // [2] accumulator slot complete (count 1, tcgen05.commit)
    uint64_t* acc_empty = bars + 3 * STAGES + 2;  // [2] accumulator slot drained  (count 128 epilogue threads)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + S::NUM_BARS);
    float* bias_s = reinterpret_cast<float*>(smem + STAGES * S::STAGE_BYTES + 512);

    constexpr uint32_t ACC_COLS = SPLIT3 ? 2 * BN : BN;   // columns per accumulator slot ([0,BN) main, [BN,2BN) cross)
    constexpr uint32_t TMEM_COLS = 2 * ACC_COLS;          // two slots: 256 (split) or 128

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles_n = (N + BN - 1) / BN;
    const int tiles_per_z = tiles_n * (int)((M + TBM - 1) / TBM);
    const int total_tiles = tiles_per_z * splits;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_b) : "memory");
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&conv[s], 128);
            mbar_init(&empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&acc_full[a], 1);
            mbar_init(&acc_empty[a], 256);
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // everything above is CTA-local setup (barriers, TMEM allocation, descriptor prefetch): under programmatic dependent
    // launch it overlaps the tail of the previous kernel; global memory is only touched after the wait
    pdl_wait();
    pdl_trigger();

    if (warp == 0) {
        // ===================================================== TMA producer
        if (lane == 0) {
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const TileCoord tc = tile_coord(tile, tiles_n, tiles_per_z, BN, K, k_chunk);
                for (int kb = 0; kb < tc.num_kb; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    mbar_wait(&empty[s], ph ^ 1);
                    uint8_t* st = smem + s * S::STAGE_BYTES;
                    mbar_expect_tx(&full[s], S::A_BYTES + S::B_BYTES);
                    const int k0 = tc.k_begin + kb * TBK;
                    if (A_MN) {
                        for (int j = 0; j < TBM / 32; ++j)
                            tma_load_2d(st + j * 4096, &tmap_a, &full[s], (int)tc.m0 + 32 * j, k0);
                    } else {
                        tma_load_2d(st, &tmap_a, &full[s], k0, (int)tc.m0);
                    }
                    uint8_t* sb = st + 2 * S::A_BYTES;
                    if (B_MN) {
                        for (int j = 0; j < BN / 32; ++j) tma_load_2d(sb + j * 4096, &tmap_b, &full[s], tc.n0 + 32 * j, k0);
                    } else {
                        tma_load_2d(sb, &tmap_b, &full[s], k0, tc.n0);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================================================== MMA issuer
        constexpr uint32_t idesc = make_idesc(A_MN, B_MN, TBM, BN);
        constexpr uint32_t A_KSTEP = A_MN ? (1024u >> 4) : (UMMA_K * 4u >> 4);   // descriptor start advance per k8
        constexpr uint32_t B_KSTEP = B_MN ? (1024u >> 4) : (UMMA_K * 4u >> 4);
        uint32_t it = 0, tile_iter = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++tile_iter) {
            const TileCoord tc = tile_coord(tile, tiles_n, tiles_per_z, BN, K, k_chunk);
            const uint32_t slot = tile_iter & 1, acc_ph = (tile_iter >> 1) & 1;
            mbar_wait(&acc_empty[slot], acc_ph ^ 1);   // epilogue has drained this accumulator slot
            tc_fence_after();
            const uint32_t d_main = tmem_base + slot * ACC_COLS;
            for (int kb = 0; kb < tc.num_kb; ++kb, ++it) {
                const int s = it % STAGES;
                const uint32_t ph = (it / STAGES) & 1;
                mbar_wait(&conv[s], ph);
                tc_fence_after();
                if (lane == 0) {
                    const uint32_t a_hi = smem_u32(smem + s * S::STAGE_BYTES);
                    const uint32_t a_lo = a_hi + S::A_BYTES;
                    const uint32_t b_hi = a_hi + 2 * S::A_BYTES;
                    const uint32_t b_lo = b_hi + S::B_BYTES;
                    const uint64_t da_hi = make_smem_desc(a_hi, A_MN), da_lo = make_smem_desc(a_lo, A_MN);
                    const uint64_t db_hi = make_smem_desc(b_hi, B_MN), db_lo = make_smem_desc(b_lo, B_MN);
#pragma unroll
                    for (int k = 0; k < TBK / UMMA_K; ++k) {
                        const uint64_t ao = (uint64_t)(k * A_KSTEP), bo = (uint64_t)(k * B_KSTEP);
                        umma_tf32(d_main, da_hi + ao, db_hi + bo, idesc, (kb | k) != 0);
                        if (SPLIT3) {
                            umma_tf32(d_main + BN, da_hi + ao, db_lo + bo, idesc, (kb | k) != 0);
                            umma_tf32(d_main + BN, da_lo + ao, db_hi + bo, idesc, 1);
                        }
                    }
                    umma_commit(&empty[s]);                                  // stage reusable once these MMAs have read it
                    if (kb == tc.num_kb - 1) umma_commit(&acc_full[slot]);   // accumulator slot final
                }
                __syncwarp();
            }
        }
    } else if (warp < 6) {
        // ===================================================== operand split (per stage)
        const int ct = threadIdx.x - 64;   // 0..127
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const TileCoord tc = tile_coord(tile, tiles_n, tiles_per_z, BN, K, k_chunk);
            for (int kb = 0; kb < tc.num_kb; ++kb, ++it) {
                const int s = it % STAGES;
                const uint32_t ph = (it / STAGES) & 1;
                mbar_wait(&full[s], ph);
                if (SPLIT3) {
                    uint8_t* st = smem + s * S::STAGE_BYTES;
                    // elementwise, hence layout-agnostic: hi in place, lo at the same (swizzled) offset of the lo buffer
                    auto split = [&](uint8_t* hi_buf, uint8_t* lo_buf, int n16) {
                        uint4* h4 = reinterpret_cast<uint4*>(hi_buf);
                        uint4* l4 = reinterpret_cast<uint4*>(lo_buf);
#pragma unroll 4
                        for (int i = ct; i < n16; i += 128) {
                            const uint4 v = h4[i];
                            uint4 h, l;
                            h.x = v.x & 0xffffe000u; h.y = v.y & 0xffffe000u; h.z = v.z & 0xffffe000u; h.w = v.w & 0xffffe000u;
                            l.x = __float_as_uint(__uint_as_float(v.x) - __uint_as_float(h.x)) & 0xffffe000u;
                            l.y = __float_as_uint(__uint_as_float(v.y) - __uint_as_float(h.y)) & 0xffffe000u;
                            l.z = __float_as_uint(__uint_as_float(v.z) - __uint_as_float(h.z)) & 0xffffe000u;
                            l.w = __float_as_uint(__uint_as_float(v.w) - __uint_as_float(h.w)) & 0xffffe000u;
                            h4[i] = h;
                            l4[i] = l;
                        }
                    };
                    split(st, st + S::A_BYTES, S::A_BYTES / 16);
                    split(st + 2 * S::A_BYTES, st + 2 * S::A_BYTES + S::B_BYTES, S::B_BYTES / 16);
                }
                fence_proxy_async_smem();   // generic-proxy writes -> visible to the tensor core (async proxy)
                mbar_arrive(&conv[s]);
            }
        }
    } else {
        // ===================================================== epilogue: TMEM -> registers -> global
        // 8 warps: warp w may touch TMEM lanes [32*(w%4), 32*(w%4)+32); warps 6..9 take columns [0, BN/2) of their
        // lane quadrant, warps 10..13 take [BN/2, BN).  One warp per scheduler was latency-bound (ncu: the epilogue
        // warps were ~100% busy at IPC 0.12 and paced the whole kernel for short-K tiles).
        const EpiCtx ec = make_epi_ctx<BN>(warp, lane, C, ldc, N, splits, epi, bias_s, S::BIAS_FLOATS);
        uint32_t tile_iter = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++tile_iter) {
            const TileCoord tc = tile_coord(tile, tiles_n, tiles_per_z, BN, K, k_chunk);
            const uint32_t slot = tile_iter & 1, acc_ph = (tile_iter >> 1) & 1;
            tc_epilogue_tile<BN, SPLIT3>(tmem_base + slot * ACC_COLS, &acc_full[slot], acc_ph, &acc_empty[slot], tc, ec, C, ldc, M,
                                         N, splits, epi);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------------ kernel, A in TMEM
// Variant for a K-major A operand (forward layers, dX).  TMA still stages the raw A tile in shared memory (deep pipeline
// = HBM/L2 latency hidden), but the four operand warps read it ONCE (each thread owns one of the 128 tile rows = one TMEM
// lane; the 128B swizzle makes the row-per-thread reads conflict-free), split it in registers and tcgen05.st the hi / lo
// halves into a TMEM stage; the MMAs take A from TMEM ("TS" form) and only B from shared memory.  Per k-block this
// removes the two split writes and the three MMA operand reads of A from the shared-memory pipe (224 KB -> 144 KB of
// smem traffic per k-block: the 3xTF32 main loop was smem-bound).  (Reading A straight from global into registers was
// tried first and lost: one k-block of register prefetch cannot cover the L2/HBM latency.)
// The two MMAs of the 3x scheme are issued as  A_hi x [B_hi ; B_lo]  (N = 256: main and cross accumulators are adjacent
// TMEM columns, B_hi and B_lo adjacent smem tiles) and  A_lo x B_hi  (N = 128 into the cross columns).
// TMEM budget (512 columns): accumulator [0,256) (single slot), A stages [256, 256 + 64*STAGES).
constexpr int TA_STAGES = 4;
constexpr uint32_t TA_ACOL0 = 256;
// Operand warps of the TMEM-A kernel.  With 4 (one per TMEM lane quadrant, each thread converting a whole 32-column row of
// the k-block) the conversion paced the main loop: one warp per SM sub-partition cannot overlap its own shared-memory /
// tcgen05.st / mbarrier latencies.  8 warps = two per quadrant, each thread converts 16 columns.
// Instantiated for the dW GEMM only (both operands are MN-major activations: 32-bit shared-memory reads for A and an
// in-kernel split of B; 576 threads leave 96 registers per thread, which makes the epilogue spill -- tolerable there
// because a dW tile runs ~100 k-blocks per epilogue).  Opt-in, see dw_operand_warps().
constexpr int ta_threads(int opw) { return 32 * (2 + opw + 8); }   // 448 (4 operand warps) or 576 (8)

// F16 (fp16-split engine): a stage covers 64 k: B tiles are [128][64] fp16 (the same 16 KB), A is two fp32 boxes of 32 k
constexpr int TA_F16_STAGES = 3;
template <int STAGES, bool F16 = false>
struct TaSmem {
    static constexpr int B_BYTES = 128 * TBK * 4;
    static constexpr int A_BYTES = TBM * TBK * 4 * (F16 ? 2 : 1);
    static constexpr int STAGE_BYTES = 2 * B_BYTES + A_BYTES;   // [B hi | B lo | A raw]
    static constexpr int NUM_BARS = 3 * STAGES + 2;
    static constexpr int BIAS_FLOATS = 2048;
    static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 + 512 + BIAS_FLOATS * 4;
    static constexpr int HEADW_FLOATS = kHeadAP * 512;   // fused heads: (A+1) x N weights, N <= 512
    static constexpr int TOTAL_HEADS = TOTAL + HEADW_FLOATS * 4;
};

// BLO: the B operand is a registered weight buffer whose low tf32 halves sit in a second array (tmap_b_lo): TMA fills the
// B_hi (raw weights; the tensor core ignores the 13 low mantissa bits) and B_lo tiles directly and the operand warps do
// no shared-memory work for B at all.
// (Tried and dropped: two extra warps taking over the B-tile split of the dW-type GEMM so that A and B work of a stage
// proceed in parallel -- 230.6 vs 232.4 us for dW + dX at M=32768, N=K=512, i.e. the B split is not what paces that GEMM.)
// F16: the fp16-split engine (A K-major fp32 with a known bound -> scaled fp16 hi/lo pairs in TMEM; B = registered fp16
// twins of a weight matrix by TMA; kind::f16 MMAs; see common.cuh "fp16 operand split").  Same roles and barriers.
template <bool A_MN, bool B_MN, bool SPLIT3, bool HEADS, bool BLO, int TA_OPW, bool F16 = false>
__global__ void __launch_bounds__(ta_threads(TA_OPW), 1)
gemm_tc_ta_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                  const __grid_constant__ CUtensorMap tmap_b_lo, float* __restrict__ C, int64_t ldc, int64_t M, int N,
                  int K, int k_chunk, int splits, const __grid_constant__ TcEpilogue epi, const float* __restrict__ a_bound) {
    static_assert(!F16 || (!A_MN && !B_MN && SPLIT3 && BLO && TA_OPW == 4), "fp16-split engine: K-major operands, weight twins");
    constexpr int BN = 128, STAGES = F16 ? TA_F16_STAGES : TA_STAGES;
    constexpr int KB_K = F16 ? 64 : TBK;                    // k per pipeline stage
    constexpr int TA_EPI_WARP0 = 2 + TA_OPW;                // first of the 8 epilogue warps
    using S = TaSmem<STAGES, F16>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_align_1024(smem_raw);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * S::STAGE_BYTES);
    uint64_t* full = bars;                  // A and B tiles landed (TMA)
    uint64_t* conv = bars + STAGES;         // A in TMEM + B split, visible to the tensor core (count 128)
    uint64_t* empty = bars + 2 * STAGES;    // MMAs of the stage retired: smem B stage and TMEM A stage reusable
    uint64_t* acc_full = bars + 3 * STAGES;
    uint64_t* acc_empty = bars + 3 * STAGES + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + S::NUM_BARS);
    float* bias_s = reinterpret_cast<float*>(smem + STAGES * S::STAGE_BYTES + 512);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles_n = (N + BN - 1) / BN;
    const int tiles_per_z = tiles_n * (int)((M + TBM - 1) / TBM);
    const int total_tiles = tiles_per_z * splits;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_b) : "memory");
        if (BLO) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_b_lo) : "memory");
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&conv[s], 32 * TA_OPW);
            mbar_init(&empty[s], 1);
        }
        mbar_init(acc_full, 1);
        mbar_init(acc_empty, 256);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // everything above is CTA-local setup (barriers, TMEM allocation, descriptor prefetch): under programmatic dependent
    // launch it overlaps the tail of the previous kernel; global memory is only touched after the wait
    pdl_wait();
    pdl_trigger();
    // fp16-split engine: binary shift of the A operand from its bound (written by an earlier kernel of the stream)
    const int a_shift = F16 ? f16_shift_for_bound(a_bound[0]) : 0;

    if (warp == 0) {
        // ===================================================== TMA producer
        if (lane == 0) {
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const TileCoord tc = tile_coord(tile, tiles_n, tiles_per_z, BN, K, k_chunk);
                const int nkb = F16 ? tc.num_kb / 2 : tc.num_kb;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % STAGES;
                    mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
                    uint8_t* sb = smem + s * S::STAGE_BYTES;
                    mbar_expect_tx(&full[s], (BLO ? 2 : 1) * S::B_BYTES + S::A_BYTES);
                    const int k0 = tc.k_begin + kb * KB_K;
                    if (F16) {
                        tma_load_2d(sb + 2 * S::B_BYTES, &tmap_a, &full[s], k0, (int)tc.m0);
                        tma_load_2d(sb + 2 * S::B_BYTES + 16384, &tmap_a, &full[s], k0 + 32, (int)tc.m0);
                        tma_load_2d(sb, &tmap_b, &full[s], k0, tc.n0);                    // hi16 [128 n][64 k]
                        tma_load_2d(sb + S::B_BYTES, &tmap_b_lo, &full[s], k0, tc.n0);    // lo16
                        continue;
                    }
                    if (A_MN) {
                        for (int j = 0; j < TBM / 32; ++j)
                            tma_load_2d(sb + 2 * S::B_BYTES + j * 4096, &tmap_a, &full[s], (int)tc.m0 + 32 * j, k0);
                    } else {
                        tma_load_2d(sb + 2 * S::B_BYTES, &tmap_a, &full[s], k0, (int)tc.m0);
                    }
                    if (B_MN) {
                        for (int j = 0; j < BN / 32; ++j) tma_load_2d(sb + j * 4096, &tmap_b, &full[s], tc.n0 + 32 * j, k0);
                        if (BLO)
                            for (int j = 0; j < BN / 32; ++j)
                                tma_load_2d(sb + S::B_BYTES + j * 4096, &tmap_b_lo, &full[s], tc.n0 + 32 * j, k0);
                    } else {
                        tma_load_2d(sb, &tmap_b, &full[s], k0, tc.n0);
                        if (BLO) tma_load_2d(sb + S::B_BYTES, &tmap_b_lo, &full[s], k0, tc.n0);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================================================== MMA issuer
        constexpr uint32_t idesc_wide = F16 ? make_idesc_f16(TBM, 2 * BN) : make_idesc(false, B_MN, TBM, SPLIT3 ? 2 * BN : BN);
        constexpr uint32_t idesc_cross = F16 ? make_idesc_f16(TBM, BN) : make_idesc(false, B_MN, TBM, BN);
        constexpr uint32_t B_KSTEP = B_MN ? (1024u >> 4) : (UMMA_K * 4u >> 4);     // 32 B per k-step (8 tf32 = 16 fp16)
        uint32_t it = 0, tile_iter = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++tile_iter) {
            const TileCoord tc = tile_coord(tile, tiles_n, tiles_per_z, BN, K, k_chunk);
            const int nkb = F16 ? tc.num_kb / 2 : tc.num_kb;
            mbar_wait(acc_empty, (tile_iter & 1) ^ 1);
            tc_fence_after();
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int s = it % STAGES;
                if (BLO) mbar_wait(&full[s], (it / STAGES) & 1);   // B tiles come straight from TMA: observe their barrier here too
                mbar_wait(&conv[s], (it / STAGES) & 1);
                tc_fence_after();
                if (lane == 0) {
                    const uint64_t db_hi = make_smem_desc(smem_u32(smem + s * S::STAGE_BYTES), B_MN);
                    const uint32_t a_hi = tmem_base + TA_ACOL0 + (uint32_t)s * 64u;
#pragma unroll
                    for (int k = 0; k < TBK / UMMA_K; ++k) {
                        const uint64_t bo = (uint64_t)(k * B_KSTEP);
                        if (F16) {
                            // 16 k per instruction = 8 TMEM columns of packed pairs; A_hi at +0, A_lo at +32 of the stage
                            umma_f16_ts(tmem_base, a_hi + k * 8, db_hi + bo, idesc_wide, (kb | k) != 0);
                            umma_f16_ts(tmem_base + BN, a_hi + 32 + k * 8, db_hi + bo, idesc_cross, 1);
                            continue;
                        }
                        // [main | cross] (+)= A_hi x [B_hi ; B_lo]   (plain tf32 mode: main (+)= A x B)
                        umma_tf32_ts(tmem_base, a_hi + k * UMMA_K, db_hi + bo, idesc_wide, (kb | k) != 0);
                        if (SPLIT3) umma_tf32_ts(tmem_base + BN, a_hi + 32 + k * UMMA_K, db_hi + bo, idesc_cross, 1);
                    }
                    umma_commit(&empty[s]);
                    if (kb == nkb - 1) umma_commit(acc_full);
                }
                __syncwarp();
            }
        }
    } else if (warp < TA_EPI_WARP0) {
        // ===================================================== operand warps: A smem -> registers -> TMEM, B split in smem
        constexpr int NCT = 32 * TA_OPW;                       // operand threads
        constexpr int CPT = 128 * TBK / NCT;                   // k-columns of its row a thread converts per k-block: 32 or 16
        const int ct = threadIdx.x - 64;                       // 0..NCT-1
        const int row = (warp & 3) * 32 + lane;                // tile row == TMEM lane this thread may access
        const int c0 = ((warp - 2) >> 2) * CPT;                // first k-column of this thread
        const uint32_t lane_addr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + TA_ACOL0 + (uint32_t)c0;
        const int sw = row & 7;                                // 128B swizzle: 16 B chunk index XOR (row % 8)
        uint32_t it = 0;
        const float a_scale = pow2f_int(a_shift);
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const TileCoord tc = tile_coord(tile, tiles_n, tiles_per_z, BN, K, k_chunk);
            const int nkb = F16 ? tc.num_kb / 2 : tc.num_kb;
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int s = it % STAGES;
                const uint32_t ph = (it / STAGES) & 1;
                // full[s] of this phase implies empty[s] of the previous one: the MMAs that read TMEM stage s have retired
                mbar_wait(&full[s], ph);
                tc_fence_after();
                uint8_t* sb = smem + s * S::STAGE_BYTES;
                if constexpr (F16) {
                    // 64 k of a tile row = two 128 B swizzled rows (one per 32-k box) -> 32 + 32 packed half2 words of TMEM;
                    // a thread converts both boxes of its row.
                    uint32_t h16[32], l16[32];
#pragma unroll
                    for (int bx = 0; bx < 2; ++bx) {
                        const uint4* arow = reinterpret_cast<const uint4*>(sb + 2 * S::B_BYTES + bx * 16384 + row * 128);
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const uint4 q = arow[j ^ sw];
                            f16_split2(__uint_as_float(q.x) * a_scale, __uint_as_float(q.y) * a_scale, h16[bx * 16 + 2 * j],
                                       l16[bx * 16 + 2 * j]);
                            f16_split2(__uint_as_float(q.z) * a_scale, __uint_as_float(q.w) * a_scale, h16[bx * 16 + 2 * j + 1],
                                       l16[bx * 16 + 2 * j + 1]);
                        }
                    }
                    const uint32_t st_addr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + TA_ACOL0 + (uint32_t)s * 64u;
                    tmem_st_cols<32>(st_addr, h16);
                    tmem_st_cols<32>(st_addr + 32u, l16);
                    tmem_st_wait();
                    tc_fence_before();
                    mbar_arrive(&conv[s]);
                    continue;
                }
                // hi = the raw fp32 word: the tensor core reads only the top 19 bits of a tf32 operand (truncation), so
                // only lo has to be formed
                uint32_t hi[CPT], lo[CPT];
                if (A_MN) {
                    // MN-major tile: box (row/32) of [32 k][32 rows], k-rows 128 B apart, 32 B chunks XOR (k % 4)
                    // (SWIZZLE_128B_ATOM_32B).  A warp reads one whole 128 B k-row per instruction: conflict-free.
                    const uint8_t* abox = sb + 2 * S::B_BYTES + (row >> 5) * 4096 + (lane & 7) * 4;
                    const int chunk = lane >> 3;
#pragma unroll
                    for (int kk = 0; kk < CPT; ++kk) {
                        const int kabs = c0 + kk;
                        const uint32_t v = *reinterpret_cast<const uint32_t*>(abox + kabs * 128 + ((chunk ^ (kabs & 3)) << 5));
                        hi[kk] = v;
                        if (SPLIT3) lo[kk] = __float_as_uint(__uint_as_float(v) - __uint_as_float(v & 0xffffe000u)) & 0xffffe000u;
                    }
                } else {
                    const uint4* arow = reinterpret_cast<const uint4*>(sb + 2 * S::B_BYTES + row * 128);
#pragma unroll
                    for (int j = 0; j < CPT / 4; ++j) {
                        const uint4 q = arow[(c0 / 4 + j) ^ sw];
                        const uint32_t v[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            hi[4 * j + e] = v[e];
                            if (SPLIT3)
                                lo[4 * j + e] =
                                    __float_as_uint(__uint_as_float(v[e]) - __uint_as_float(v[e] & 0xffffe000u)) & 0xffffe000u;
                        }
                    }
                }
                tmem_st_cols<CPT>(lane_addr + (uint32_t)s * 64u, hi);
                if (SPLIT3) tmem_st_cols<CPT>(lane_addr + (uint32_t)s * 64u + 32u, lo);
                if (SPLIT3 && !BLO) {
                    // B hi stays the raw tile in place (see above); only the lo tile is written
                    const uint4* h4 = reinterpret_cast<const uint4*>(sb);
                    uint4* l4 = reinterpret_cast<uint4*>(sb + S::B_BYTES);
#pragma unroll 4
                    for (int i = ct; i < S::B_BYTES / 16; i += NCT) {
                        const uint4 v = h4[i];
                        uint4 l;
                        l.x = __float_as_uint(__uint_as_float(v.x) - __uint_as_float(v.x & 0xffffe000u)) & 0xffffe000u;
                        l.y = __float_as_uint(__uint_as_float(v.y) - __uint_as_float(v.y & 0xffffe000u)) & 0xffffe000u;
                        l.z = __float_as_uint(__uint_as_float(v.z) - __uint_as_float(v.z & 0xffffe000u)) & 0xffffe000u;
                        l.w = __float_as_uint(__uint_as_float(v.w) - __uint_as_float(v.w & 0xffffe000u)) & 0xffffe000u;
                        l4[i] = l;
                    }
                }
                tmem_st_wait();
                if (!BLO) fence_proxy_async_smem();   // (BLO: these warps wrote nothing to shared memory)
                tc_fence_before();
                mbar_arrive(&conv[s]);
            }
        }
    } else {
        // ===================================================== epilogue (single accumulator slot)
        float* headw_s = bias_s + S::BIAS_FLOATS;
        if (HEADS) {
            // [kHeadAP][N]: row 0 = critic weights, rows 1..A = distribution_linear rows, the rest zero
            for (int i = threadIdx.x - TA_EPI_WARP0 * 32; i < kHeadAP * N; i += 256) {
                const int a = i / N, n = i - a * N;
                headw_s[i] = (a == 0) ? epi.head_wv[n] : (a <= epi.head_A ? epi.head_wa[(int64_t)(a - 1) * N + n] : 0.f);
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");
        }
        EpiCtx ec = make_epi_ctx<BN, TA_EPI_WARP0>(warp, lane, C, ldc, N, splits, epi, bias_s, S::BIAS_FLOATS);
        if (F16) ec.out_scale = pow2f_int(-(a_shift + kF16WShift));
        uint32_t tile_iter = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++tile_iter) {
            const TileCoord tc = tile_coord(tile, tiles_n, tiles_per_z, BN, K, k_chunk);
            if (HEADS) {
                switch (epi.act) {
                    case SFB200_ACT_ELU:
                        tc_epilogue_tile_heads<BN, SPLIT3, SFB200_ACT_ELU, F16>(tmem_base, acc_full, tile_iter & 1, acc_empty, tc, ec, C,
                                                                           ldc, M, N, epi, headw_s);
                        break;
                    case SFB200_ACT_RELU:
                        tc_epilogue_tile_heads<BN, SPLIT3, SFB200_ACT_RELU, F16>(tmem_base, acc_full, tile_iter & 1, acc_empty, tc, ec,
                                                                            C, ldc, M, N, epi, headw_s);
                        break;
                    case SFB200_ACT_TANH:
                        tc_epilogue_tile_heads<BN, SPLIT3, SFB200_ACT_TANH, F16>(tmem_base, acc_full, tile_iter & 1, acc_empty, tc, ec,
                                                                            C, ldc, M, N, epi, headw_s);
                        break;
                    default:
                        tc_epilogue_tile_heads<BN, SPLIT3, SFB200_ACT_NONE, F16>(tmem_base, acc_full, tile_iter & 1, acc_empty, tc, ec,
                                                                            C, ldc, M, N, epi, headw_s);
                        break;
                }
            } else {
                tc_epilogue_tile<BN, SPLIT3, F16>(tmem_base, acc_full, tile_iter & 1, acc_empty, tc, ec, C, ldc, M, N, splits, epi);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ------------------------------------------------------------------------------------------------ host side
static PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;
static int g_tc_state = 0;   // 0 unknown, 1 ok, -1 unavailable

bool tc_init() {
    if (g_tc_state != 0) return g_tc_state > 0;
    g_tc_state = -1;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
        qres != cudaDriverEntryPointSuccess) {
        cudaGetLastError();
        return false;
    }
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess ||
        major != 10) {
        cudaGetLastError();
        return false;
    }
    g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
    g_tc_state = 1;
    return true;
}

// 2-D fp32 tensor map, 128B swizzle (16 B chunks for K-major tiles, 32 B chunks for MN-major). dim0 = contiguous dim.
bool make_tmap(CUtensorMap* out, const float* base, uint64_t dim0, uint64_t dim1, uint64_t stride1_elems,
                      uint32_t box0, uint32_t box1, bool mn_major) {
    cuuint64_t gdim[2] = {dim0, dim1};
    cuuint64_t gstride[1] = {stride1_elems * sizeof(float)};
    cuuint32_t box[2] = {box0, box1};
    cuuint32_t estride[2] = {1, 1};
    CUresult r = g_encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstride, box, estride,
                          CU_TENSOR_MAP_INTERLEAVE_NONE,
                          mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

static bool operand_ok(const float* p, int64_t ld) {
    return ((reinterpret_cast<uintptr_t>(p) & 15u) == 0) && (ld % 4 == 0) && ld > 0;
}

// shared-memory-A kernel: N < 128 (every N >= 128 shape runs on the TMEM-A kernel)
template <bool A_MN, bool B_MN, bool SPLIT3>
static int launch_tc(const CUtensorMap& ta, const CUtensorMap& tb, float* C, int64_t ldc, int64_t M, int N, int K,
                     int k_chunk, int splits, const TcEpilogue& epi, cudaStream_t st) {
    constexpr int BN = 64, STAGES = 4;
    using S = TcSmem<BN, STAGES>;
    auto kern = gemm_tc_kernel<A_MN, B_MN, BN, STAGES, SPLIT3>;
    static bool attr_set = false;
    if (!attr_set) {
        SFB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
        attr_set = true;
    }
    const int64_t tiles = ceil_div(N, BN) * ceil_div(M, TBM) * splits;
    const int64_t grid = tiles < sm_count() ? tiles : sm_count();   // persistent: one CTA per SM
    SFB_CUDA_OK(launch_pdl(kern, dim3((unsigned)grid), dim3(TC_THREADS), (size_t)S::TOTAL, st, ta, tb, C, ldc, M, N, K, k_chunk,
                           splits, epi));
    SFB_LAUNCH_OK();
    return 0;
}

// SFB200_TA_DW_OPW=8 runs the dW-type GEMM (both operands MN-major) with eight operand warps instead of four: 120.8 vs 128.0 us
// at 32768 x 512 x 512 (tools/dw_bench.py, call r02_y; before the shared-memory address-space fix the two were equal).  Opt-in:
// the round's GPU budget ended before the full parity suite could be re-run with it as the default.
static int dw_operand_warps() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("SFB200_TA_DW_OPW");
        v = (e && e[0] == '8') ? 8 : 4;
    }
    return v;
}

template <bool A_MN, bool B_MN, bool SPLIT3, bool HEADS, bool BLO, int OPW, bool F16 = false>
static int launch_tc_ta_opw(const CUtensorMap& ta, const CUtensorMap& tb, float* C, int64_t ldc, int64_t M, int N, int K,
                            int k_chunk, int splits, const TcEpilogue& epi, cudaStream_t st, const CUtensorMap* tb_lo,
                            const float* a_bound = nullptr) {
    using S = TaSmem<F16 ? TA_F16_STAGES : TA_STAGES, F16>;
    auto kern = gemm_tc_ta_kernel<A_MN, B_MN, SPLIT3, HEADS, BLO, OPW, F16>;
    constexpr int SMEM = HEADS ? S::TOTAL_HEADS : S::TOTAL;
    static bool attr_set = false;
    if (!attr_set) {
        SFB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
        attr_set = true;
    }
    const int64_t tiles = ceil_div(N, 128) * ceil_div(M, TBM) * splits;
    const int64_t grid = tiles < sm_count() ? tiles : sm_count();
    SFB_CUDA_OK(launch_pdl(kern, dim3((unsigned)grid), dim3(ta_threads(OPW)), (size_t)SMEM, st, ta, tb, tb_lo ? *tb_lo : tb, C, ldc, M,
                           N, K, k_chunk, splits, epi, a_bound));
    SFB_LAUNCH_OK();
    return 0;
}

template <bool A_MN, bool B_MN, bool SPLIT3, bool HEADS = false, bool BLO = false>
static int launch_tc_ta(const CUtensorMap& ta, const CUtensorMap& tb, float* C, int64_t ldc, int64_t M, int N, int K,
                        int k_chunk, int splits, const TcEpilogue& epi, cudaStream_t st, const CUtensorMap* tb_lo = nullptr) {
    if constexpr (A_MN && B_MN) {
        if (dw_operand_warps() == 8)
            return launch_tc_ta_opw<A_MN, B_MN, SPLIT3, HEADS, BLO, 8>(ta, tb, C, ldc, M, N, K, k_chunk, splits, epi, st, tb_lo);
    }
    return launch_tc_ta_opw<A_MN, B_MN, SPLIT3, HEADS, BLO, 4>(ta, tb, C, ldc, M, N, K, k_chunk, splits, epi, st, tb_lo);
}

bool make_tmap_f16(CUtensorMap* out, const uint16_t* base, uint64_t dim0, uint64_t dim1, uint64_t stride1_elems, uint32_t box0,
                   uint32_t box1) {
    cuuint64_t gdim[2] = {dim0, dim1};
    cuuint64_t gstride[1] = {stride1_elems * sizeof(uint16_t)};
    cuuint32_t box[2] = {box0, box1};
    cuuint32_t estride[2] = {1, 1};
    CUresult r = g_encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<uint16_t*>(base), gdim, gstride, box, estride,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

// SFB200_CHECK_F16=1: verify registered fp16 twins against the weights on the device before every use (debugging aid, like
// SFB200_CHECK_LO for the tf32 twins)
bool f16_check_enabled() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("SFB200_CHECK_F16");
        v = (e && e[0] == '1') ? 1 : 0;
    }
    return v == 1;
}

// C[M,N] = epi( sum_k A(m,k) B(n,k) ). Returns SFB_TC_UNSUPPORTED when the shape/alignment is not covered.
static int gemm_tc(bool a_mn, const float* A, int64_t lda, bool b_mn, const float* B, int64_t ldb, float* C, int64_t ldc,
                   int64_t M, int N, int K, int splits, const TcEpilogue& epi, float* ws, bool split3, cudaStream_t st) {
    if (!tc_init()) return SFB_TC_UNSUPPORTED;
    if (!operand_ok(A, lda) || !operand_ok(B, ldb) || M < 1 || N < 8 || K < 8) return SFB_TC_UNSUPPORTED;
    if (M > 0x7fffffff || ceil_div(M, TBM) * ceil_div(N, 64) * 64 > 0x7fffffff) return SFB_TC_UNSUPPORTED;
    // (A MN-major, B K-major) has no caller and is not instantiated
    if (a_mn && !b_mn) return SFB_TC_UNSUPPORTED;
    const int BN = (N >= 128) ? 128 : 64;
    CUtensorMap ta, tb;
    bool ok;
    if (a_mn) ok = make_tmap(&ta, A, (uint64_t)M, (uint64_t)K, (uint64_t)lda, 32, TBK, true);
    else ok = make_tmap(&ta, A, (uint64_t)K, (uint64_t)M, (uint64_t)lda, TBK, TBM, false);
    if (b_mn) ok = ok && make_tmap(&tb, B, (uint64_t)N, (uint64_t)K, (uint64_t)ldb, 32, TBK, true);
    else ok = ok && make_tmap(&tb, B, (uint64_t)K, (uint64_t)N, (uint64_t)ldb, TBK, (uint32_t)BN, false);
    if (!ok) return SFB_TC_UNSUPPORTED;

    int k_chunk = K;
    if (splits > 1) {
        k_chunk = (int)(ceil_div(ceil_div(K, splits), TBK) * TBK);
        splits = (int)ceil_div(K, k_chunk);
    }
    if (splits > 1 && !ws) return SFB_TC_UNSUPPORTED;
    float* out = splits > 1 ? ws : C;
    const int64_t ld_out = splits > 1 ? N : ldc;

    if (epi.head_part && !(BN == 128 && !a_mn && !b_mn && splits == 1)) return SFB_TC_UNSUPPORTED;
    // fp16-split engine: A is a K-major activation buffer with a registered bound, B a weight matrix with registered fp16
    // twins (the transposed twins when B is read MN-major, i.e. dX = dz . W), K a multiple of the 64-k stage
    if (BN == 128 && !a_mn && split3 && splits == 1 && K % 64 == 0) {
        const float* a_bound = operand_bound_lookup(A, ((int64_t)(M - 1) * lda + K) * (int64_t)sizeof(float));
        F16Twin tw{nullptr, nullptr};
        if (a_bound) {
            if (!b_mn && ldb == K) tw = f16_twin_lookup(B, (int64_t)N * K);
            else if (b_mn && ldb == N) tw = f16_twinT_lookup(B, K, N);      // B = W[K][N] row-major, twins stored as [N][K]
        }
        if (tw.hi) {
            if (f16_check_enabled()) {
                // B = W[N][K] row-major (forward) or W[K][N] row-major read along its other axis (dX: twins transposed)
                const int rc_chk = b_mn ? f16_twins_check(B, tw, K, N, true, st) : f16_twins_check(B, tw, N, K, false, st);
                if (rc_chk) return rc_chk;
            }
            CUtensorMap tb_hi, tb_lo16;
            if (!make_tmap_f16(&tb_hi, tw.hi, (uint64_t)K, (uint64_t)N, (uint64_t)K, 64, 128) ||
                !make_tmap_f16(&tb_lo16, tw.lo, (uint64_t)K, (uint64_t)N, (uint64_t)K, 64, 128))
                return SFB_TC_UNSUPPORTED;
            if (epi.head_part)
                return launch_tc_ta_opw<false, false, true, true, true, 4, true>(ta, tb_hi, out, ld_out, M, N, K, k_chunk, splits,
                                                                                 epi, st, &tb_lo16, a_bound);
            return launch_tc_ta_opw<false, false, true, false, true, 4, true>(ta, tb_hi, out, ld_out, M, N, K, k_chunk, splits, epi,
                                                                              st, &tb_lo16, a_bound);
        }
    }
    int rc;
    if (BN == 128) {
        // A operand from TMEM (gemm_tc_ta_kernel)
        // weight operand with a registered tf32-lo twin (forward layers and dX: B is the weight matrix)
        const int64_t b_extent = b_mn ? (int64_t)(K - 1) * ldb + N : (int64_t)(N - 1) * ldb + K;
        const float* B_lo = (split3 && !a_mn) ? tf32_lo_lookup(B, b_extent) : nullptr;
        if (B_lo) {
            CUtensorMap tb_lo;
            bool ok_lo;
            if (b_mn) ok_lo = make_tmap(&tb_lo, B_lo, (uint64_t)N, (uint64_t)K, (uint64_t)ldb, 32, TBK, true);
            else ok_lo = make_tmap(&tb_lo, B_lo, (uint64_t)K, (uint64_t)N, (uint64_t)ldb, TBK, 128, false);
            if (!ok_lo) return SFB_TC_UNSUPPORTED;
            if (tf32_lo_check_enabled()) {
                int rcc = tf32_lo_check(B, B_lo, b_extent, st);
                if (rcc) return rcc;
            }
            if (epi.head_part) rc = launch_tc_ta<false, false, true, true, true>(ta, tb, out, ld_out, M, N, K, k_chunk, splits, epi, st, &tb_lo);
            else if (!b_mn) rc = launch_tc_ta<false, false, true, false, true>(ta, tb, out, ld_out, M, N, K, k_chunk, splits, epi, st, &tb_lo);
            else rc = launch_tc_ta<false, true, true, false, true>(ta, tb, out, ld_out, M, N, K, k_chunk, splits, epi, st, &tb_lo);
        } else {
#define SFB_TA(AM, BM_)                                                                                                \
    (split3 ? launch_tc_ta<AM, BM_, true>(ta, tb, out, ld_out, M, N, K, k_chunk, splits, epi, st)                     \
            : launch_tc_ta<AM, BM_, false>(ta, tb, out, ld_out, M, N, K, k_chunk, splits, epi, st))
            if (epi.head_part) {
                rc = split3 ? launch_tc_ta<false, false, true, true>(ta, tb, out, ld_out, M, N, K, k_chunk, splits, epi, st)
                            : launch_tc_ta<false, false, false, true>(ta, tb, out, ld_out, M, N, K, k_chunk, splits, epi, st);
            } else if (!a_mn && !b_mn) rc = SFB_TA(false, false);
            else if (!a_mn && b_mn) rc = SFB_TA(false, true);
            else rc = SFB_TA(true, true);
#undef SFB_TA
        }
    } else {
#define SFB_TC(AM, BM_)                                                                                                \
    (split3 ? launch_tc<AM, BM_, true>(ta, tb, out, ld_out, M, N, K, k_chunk, splits, epi, st)                         \
            : launch_tc<AM, BM_, false>(ta, tb, out, ld_out, M, N, K, k_chunk, splits, epi, st))
        if (!a_mn && !b_mn) rc = SFB_TC(false, false);
        else if (!a_mn && b_mn) rc = SFB_TC(false, true);
        else rc = SFB_TC(true, true);
#undef SFB_TC
    }
    if (rc) return rc;
    if (splits > 1) return splitk_reduce(ws, splits, M, N, C, ldc, st);
    return 0;
}

int tc_linear_act_forward(const float* x, int64_t ldx, const float* W, const float* b, float* y, int64_t ldy, int64_t M,
                          int N, int K, int act, int engine, cudaStream_t st) {
    TcEpilogue epi{1, act, b, nullptr, 0};
    return gemm_tc(false, x, ldx, false, W, K, y, ldy, M, N, K, 1, epi, nullptr, engine == SFB200_GEMM_TC_3XTF32, st);
}

// Number of head partials the fused forward produces per row for an N-wide layer, or 0 when the fused path does not
// cover the shape (callers then run the layer and the heads kernel separately).
int tc_linear_heads_partials(int N, int A, int engine) {
    if (engine == SFB200_GEMM_SIMT_FP32 || !tc_init()) return 0;
    if (N % 128 != 0 || N > 512 || A < 1 || A + 1 > kHeadAP) return 0;
    return 2 * (N / 128);
}

int tc_linear_act_heads_forward(const float* x, int64_t ldx, const float* W, const float* b, float* y, int64_t ldy,
                                int64_t M, int N, int K, int act, int engine, const float* Wv, const float* Wa, int A,
                                float* head_part, cudaStream_t st) {
    if (tc_linear_heads_partials(N, A, engine) == 0 || !b) return SFB_TC_UNSUPPORTED;
    if (y && (ldy % 4 != 0 || (reinterpret_cast<uintptr_t>(y) & 15u))) return SFB_TC_UNSUPPORTED;
    if (reinterpret_cast<uintptr_t>(head_part) & 15u) return SFB_TC_UNSUPPORTED;
    TcEpilogue epi{1, act, b, nullptr, 0, Wv, Wa, A, head_part};
    return gemm_tc(false, x, ldx, false, W, K, y, y ? ldy : N, M, N, K, 1, epi, nullptr, engine == SFB200_GEMM_TC_3XTF32, st);
}

int tc_linear_backward(const float* dz, int64_t lddz, const float* x, int64_t ldx, const float* W, int64_t M, int N, int K,
                       int act_prev, float* dW, float* dx, int64_t lddx, int engine, float* ws, cudaStream_t st,
                       float* colsum_part, int* colsum_fused) {
    const bool split3 = engine == SFB200_GEMM_TC_3XTF32;
    // dW[n,k] = sum_m dz[m,n] x[m,k]: both operands are stored with the reduced index m as the row -> MN-major
    TcEpilogue none{0, 0, nullptr, nullptr, 0};
    const int splits = choose_splits(N, K, (int)M);
    int rc = dW ? gemm_tc(true, dz, lddz, true, x, ldx, dW, K, N, K, (int)M, splits, none, ws, split3, st) : 0;
    if (rc) return rc;
    if (dx) {
        // dx[m,k] = (sum_n dz[m,n] W[n,k]) * act_prev'(x[m,k]): A = dz K-major, B(k, n) = W[n,k] MN-major
        TcEpilogue e{act_prev == SFB200_ACT_NONE ? 0 : 2, act_prev, nullptr, x, ldx};
        // db_prev = column sums of dx, folded into this GEMM's epilogue when every tile is full (TMEM-A kernel, BN = 128)
        const bool fuse_cs = colsum_part && M % 128 == 0 && K % 128 == 0 && lddx % 4 == 0 &&
                             (act_prev == SFB200_ACT_NONE || (ldx % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15u) == 0)) &&
                             (reinterpret_cast<uintptr_t>(dx) & 15u) == 0;
        if (fuse_cs) e.colsum_part = colsum_part;
        if (colsum_fused) *colsum_fused = fuse_cs ? 1 : 0;
        rc = gemm_tc(false, dz, lddz, true, W, K, dx, lddx, M, K, N, 1, e, nullptr, split3, st);
        if (rc) return rc;
    }
    return 0;
}

}  // namespace sfb

extern "C" int sfb200_tc_available(void) { return sfb::tc_init() ? 1 : 0; }
