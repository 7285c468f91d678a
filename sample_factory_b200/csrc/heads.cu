// Policy/value heads: critic_linear + distribution_linear (N = 1 + A output columns, far too narrow for a
// tensor-core tile) fused with the categorical distribution math, forward and backward.  Both kernels stream h once
// (HBM-bound: 4*H bytes per row read, backward also writes 4*H).
#include "gemm.h"
#include "heads_tail.cuh"

namespace sfb {

constexpr int kHeadsMaxGroups = 1024;


// Heads from the partial dot products left by the fused GEMM epilogue (gemm_tc.cu, tc_epilogue_tile_heads):
// part[p][row][kPad], summed over p in fixed order (deterministic).  One warp per row, lane a = output a.
__global__ void __launch_bounds__(256) heads_from_partials_kernel(const float* __restrict__ part, int P, int64_t rows,
                                                                  const HeadsFinish f) {
    pdl_wait();
    pdl_trigger();
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float pv = f.pv_scalar ? *f.pv_scalar : 0.f;
    const uint64_t offset = f.offset_host + (f.offset_dev ? (uint64_t)*f.offset_dev : 0ull);
    for (int64_t row = warp; row < rows; row += nwarps) heads_finish_row(part, P, rows, row, lane, f, pv, offset);
}

// ---------------------------------------------------------------------------------------------------------------------
// forward (+ optional sampling).  One warp handles RPW rows at a time; lane l owns columns l, l+32, ...
// Wcat (smem): row 0 = Wv, rows 1..A = Wa.  AP = compile-time bound on A+1.
// ---------------------------------------------------------------------------------------------------------------------
template <int AP, int RPW, bool VEC>
__global__ void __launch_bounds__(256) heads_forward_kernel(
    const float* __restrict__ h, int64_t ldh, int64_t rows, int H, int A, const float* __restrict__ Wv,
    const float* __restrict__ bv, const float* __restrict__ Wa, const float* __restrict__ ba, const HeadsOut out,
    const float* __restrict__ noise, uint64_t seed, uint64_t offset_host, const int64_t* __restrict__ offset_dev,
    const float* __restrict__ pv_scalar) {
    extern __shared__ float wcat[];   // [(A+1)][H]
    pdl_wait();
    pdl_trigger();
    const int n_out = A + 1;
    for (int i = threadIdx.x; !VEC && i < n_out * H; i += blockDim.x) {
        const int a = i / H, j = i - a * H;
        wcat[i] = (a == 0) ? Wv[j] : Wa[(int64_t)(a - 1) * H + j];
    }
    if (!VEC) __syncthreads();

    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float pv = pv_scalar ? *pv_scalar : 0.f;
    const uint64_t offset = offset_host + (offset_dev ? (uint64_t)*offset_dev : 0ull);
    const float my_bias = (lane == 0) ? bv[0] : (lane <= A ? ba[lane - 1] : 0.f);

    for (int64_t r0 = warp * RPW; r0 < rows; r0 += nwarps * RPW) {
        float acc[RPW][AP];
#pragma unroll
        for (int r = 0; r < RPW; ++r)
#pragma unroll
            for (int a = 0; a < AP; ++a) acc[r][a] = 0.f;

        if (VEC) {
            // 128-bit path: lane owns 4 consecutive columns; the (A+1) x H weights (18 KB for cfg-2) are read through
            // L1 with __ldg -- every warp of the SM reads the same lines, so no shared-memory staging is needed
            for (int j = lane * 4; j < H; j += 128) {
                float4 hv[RPW];
#pragma unroll
                for (int r = 0; r < RPW; ++r)
                    hv[r] = (r0 + r < rows) ? *reinterpret_cast<const float4*>(h + (r0 + r) * ldh + j)
                                            : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int a = 0; a < AP; ++a) {
                    if (a < n_out) {
                        const float4 w = __ldg(reinterpret_cast<const float4*>((a == 0 ? Wv : Wa + (int64_t)(a - 1) * H) + j));
#pragma unroll
                        for (int r = 0; r < RPW; ++r) {
                            acc[r][a] = fmaf(hv[r].x, w.x, acc[r][a]);
                            acc[r][a] = fmaf(hv[r].y, w.y, acc[r][a]);
                            acc[r][a] = fmaf(hv[r].z, w.z, acc[r][a]);
                            acc[r][a] = fmaf(hv[r].w, w.w, acc[r][a]);
                        }
                    }
                }
            }
        } else {
            for (int j = lane; j < H; j += 32) {
                float hv[RPW];
#pragma unroll
                for (int r = 0; r < RPW; ++r) hv[r] = (r0 + r < rows) ? h[(r0 + r) * ldh + j] : 0.f;
#pragma unroll
                for (int a = 0; a < AP; ++a) {
                    if (a < n_out) {
                        const float w = wcat[a * H + j];
#pragma unroll
                        for (int r = 0; r < RPW; ++r) acc[r][a] = fmaf(hv[r], w, acc[r][a]);
                    }
                }
            }
        }
#pragma unroll
        for (int r = 0; r < RPW; ++r) {
            const int64_t row = r0 + r;
            if (row >= rows) break;   // warp-uniform
            // lane a ends up with output a (0 = value, 1..A = logits)
            float mine = 0.f;
#pragma unroll
            for (int a = 0; a < AP; ++a) {
                if (a < n_out) {
                    const float s = warp_sum(acc[r][a]);
                    if (lane == a) mine = s;
                }
            }
            mine += my_bias;
            heads_row_tail(mine, lane, A, row, out, noise, seed, offset, pv);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// backward.  grid = row groups; block = 256 threads, thread owns column j of the current 256-wide strip.
// g[b][0] = dvalues[b], g[b][1..A] = dlogits[b][:].
//   dz[b][j]      = (sum_a g[b][a] * Wcat[a][j]) * act'(h[b][j])
//   dWcat[a][j]  += g[b][a] * h[b][j] ;  db_prev[j] += dz[b][j] ;  dbcat[a] += g[b][a]
// per-block partial sums go to the workspace, a second kernel reduces them in fixed order (deterministic).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kHbTile = 32;   // rows of coefficients staged in smem per iteration

template <int AP>
__global__ void __launch_bounds__(256) heads_backward_kernel(
    const float* __restrict__ h, int64_t ldh, int64_t rows, int H, int A, const float* __restrict__ Wv,
    const float* __restrict__ Wa, const float* __restrict__ dlogits, const float* __restrict__ dvalues, int act,
    float* __restrict__ dz, int64_t lddz, float* __restrict__ part, int64_t rows_per_group) {
    __shared__ float g_s[kHbTile][AP];
    const int n_out = A + 1;
    const int tid = threadIdx.x;
    const int64_t r_begin = blockIdx.x * rows_per_group;
    const int64_t r_end = (r_begin + rows_per_group < rows) ? r_begin + rows_per_group : rows;
    const int64_t part_stride = (int64_t)(A + 2) * H + n_out;
    float* my_part = part + blockIdx.x * part_stride;

    float acc_g = 0.f;   // dbcat partial, threads tid < n_out (strip 0 only)
    const int nstrips = (H + 255) / 256;
    for (int strip = 0; strip < nstrips; ++strip) {
        const int j = strip * 256 + tid;
        const bool col_ok = j < H;
        float w[AP], accw[AP];
#pragma unroll
        for (int a = 0; a < AP; ++a) {
            accw[a] = 0.f;
            w[a] = (col_ok && a < n_out) ? (a == 0 ? Wv[j] : Wa[(int64_t)(a - 1) * H + j]) : 0.f;
        }
        float acc_db = 0.f;
        for (int64_t b0 = r_begin; b0 < r_end; b0 += kHbTile) {
            const int nb = (int)((r_end - b0 < kHbTile) ? (r_end - b0) : kHbTile);
            __syncthreads();
            for (int i = tid; i < kHbTile * n_out; i += 256) {
                const int bb = i / n_out, a = i - bb * n_out;
                float v = 0.f;
                if (bb < nb) v = (a == 0) ? dvalues[b0 + bb] : dlogits[(b0 + bb) * A + (a - 1)];
                g_s[bb][a] = v;
            }
            __syncthreads();
            if (strip == 0 && tid < n_out) {
                for (int bb = 0; bb < nb; ++bb) acc_g += g_s[bb][tid];
            }
            if (col_ok) {
#pragma unroll 4
                for (int bb = 0; bb < nb; ++bb) {
                    const float hv = h[(b0 + bb) * ldh + j];
                    float s = 0.f;
#pragma unroll
                    for (int a = 0; a < AP; ++a) {
                        if (a < n_out) {
                            const float g = g_s[bb][a];
                            s = fmaf(g, w[a], s);
                            accw[a] = fmaf(g, hv, accw[a]);
                        }
                    }
                    const float d = s * act_bwd_from_out(hv, act);
                    dz[(b0 + bb) * lddz + j] = d;
                    acc_db += d;
                }
            }
        }
        if (col_ok) {
#pragma unroll
            for (int a = 0; a < AP; ++a)
                if (a < n_out) my_part[(int64_t)a * H + j] = accw[a];
            my_part[(int64_t)n_out * H + j] = acc_db;
        }
    }
    if (tid < n_out) my_part[(int64_t)(A + 2) * H + tid] = acc_g;
}

// Vectorised variant: a thread owns VW (4 or 2) consecutive columns (128- / 64-bit loads and stores) and every RPB-th
// row of the group; row-lane partials are combined through shared memory at the end.  VW = 2 halves the per-thread
// register state (weights + 9 weight-gradient accumulators per column), which lets four blocks reside per SM with eight
// row loads in flight per thread: this kernel is HBM-latency bound (reads h, writes dz: 8*H bytes per row).
template <int AP, int VW, int UNROLL, int MINB>
__global__ void __launch_bounds__(256, MINB) heads_backward_vec_kernel(
    const float* __restrict__ h, int64_t ldh, int64_t rows, int H, int A, const float* __restrict__ Wv,
    const float* __restrict__ Wa, const float* __restrict__ dlogits, const float* __restrict__ dvalues, int act,
    float* __restrict__ dz, int64_t lddz, float* __restrict__ part, int64_t rows_per_group) {
    __shared__ float g_s[kHbTile][AP];
    extern __shared__ float red_s[];   // [(A+2)][H] cross-row-lane reduction
    const int n_out = A + 1;
    const int tid = threadIdx.x;
    const int TPR = H / VW, RPB = 256 / TPR;
    const int cv = tid % TPR, rl = tid / TPR;
    const int j = cv * VW;
    const int64_t r_begin = blockIdx.x * rows_per_group;
    const int64_t r_end = (r_begin + rows_per_group < rows) ? r_begin + rows_per_group : rows;
    const int64_t part_stride = (int64_t)(A + 2) * H + n_out;
    float* my_part = part + blockIdx.x * part_stride;

    float w[AP][VW], accw[AP][VW];
#pragma unroll
    for (int a = 0; a < AP; ++a) {
#pragma unroll
        for (int c = 0; c < VW; ++c) {
            accw[a][c] = 0.f;
            w[a][c] = (a < n_out) ? (a == 0 ? Wv[j + c] : Wa[(int64_t)(a - 1) * H + j + c]) : 0.f;
        }
    }
    float acc_db[VW];
#pragma unroll
    for (int c = 0; c < VW; ++c) acc_db[c] = 0.f;
    float acc_g = 0.f;
    for (int64_t b0 = r_begin; b0 < r_end; b0 += kHbTile) {
        const int nb = (int)((r_end - b0 < kHbTile) ? (r_end - b0) : kHbTile);
        __syncthreads();
        for (int i = tid; i < kHbTile * n_out; i += 256) {
            const int bb = i / n_out, a = i - bb * n_out;
            float v = 0.f;
            if (bb < nb) v = (a == 0) ? dvalues[b0 + bb] : dlogits[(b0 + bb) * A + (a - 1)];
            g_s[bb][a] = v;
        }
        __syncthreads();
        if (tid < n_out)
            for (int bb = 0; bb < nb; ++bb) acc_g += g_s[bb][tid];
#pragma unroll UNROLL
        for (int bb = rl; bb < nb; bb += RPB) {
            float hv[VW];
            if (VW == 4) {
                const float4 q = *reinterpret_cast<const float4*>(h + (b0 + bb) * ldh + j);
                hv[0] = q.x; hv[1] = q.y; hv[VW - 2] = q.z; hv[VW - 1] = q.w;
            } else {
                const float2 q = *reinterpret_cast<const float2*>(h + (b0 + bb) * ldh + j);
                hv[0] = q.x; hv[1] = q.y;
            }
            float sacc[VW];
#pragma unroll
            for (int c = 0; c < VW; ++c) sacc[c] = 0.f;
#pragma unroll
            for (int a = 0; a < AP; ++a) {
                if (a < n_out) {
                    const float g = g_s[bb][a];
#pragma unroll
                    for (int c = 0; c < VW; ++c) {
                        sacc[c] = fmaf(g, w[a][c], sacc[c]);
                        accw[a][c] = fmaf(g, hv[c], accw[a][c]);
                    }
                }
            }
            float d[VW];
#pragma unroll
            for (int c = 0; c < VW; ++c) {
                d[c] = sacc[c] * act_bwd_from_out(hv[c], act);
                acc_db[c] += d[c];
            }
            if (VW == 4) *reinterpret_cast<float4*>(dz + (b0 + bb) * lddz + j) = make_float4(d[0], d[1], d[VW - 2], d[VW - 1]);
            else *reinterpret_cast<float2*>(dz + (b0 + bb) * lddz + j) = make_float2(d[0], d[1]);
        }
    }
    // combine the RPB row lanes (fixed order -> deterministic)
    for (int r = 0; r < RPB; ++r) {
        __syncthreads();
        if (rl == r) {
#pragma unroll
            for (int a = 0; a < AP; ++a) {
                if (a < n_out) {
#pragma unroll
                    for (int c = 0; c < VW; ++c) {
                        float v = accw[a][c];
                        if (r > 0) v += red_s[a * H + j + c];
                        red_s[a * H + j + c] = v;
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < VW; ++c) {
                float v = acc_db[c];
                if (r > 0) v += red_s[n_out * H + j + c];
                red_s[n_out * H + j + c] = v;
            }
        }
    }
    __syncthreads();
    for (int i = tid; i < (A + 2) * H; i += 256) my_part[i] = red_s[i];
    if (tid < n_out) my_part[(int64_t)(A + 2) * H + tid] = acc_g;
}

// Software-pipelined variant for the learner-sized case (two columns per thread).  Two things bound the kernel above
// (ncu, profiles/r01_m_ncu_heads_backward.md): the compiler keeps ONE row load in flight per thread (load -> 36 FMAs ->
// store, serially: ~2 TB/s), and once that is fixed, instruction issue (123 instructions per row and warp, 2/3 of them
// address arithmetic, guards and scalar shared-memory loads).  Here the row loads run U rows ahead of the arithmetic
// through a register queue with static slots, all pointers advance by increments, full batches run unguarded, the
// coefficients of a row come as three 128-bit shared loads, and the activation is a template parameter.
// Row k of a thread is r_begin + rl + k*RPB; a staged coefficient tile covers kpt = kHbTile/RPB consecutive k, a
// multiple of U.
constexpr int kHbGP = 20;   // floats per staged coefficient row: 9 duplicated pairs (g, g) + padding to 5 x 16 bytes

// packed fp32 pairs (sm_100 FFMA2: two IEEE fma.rn per instruction -- same results as the scalar form, half the issue slots)
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ float2 unpack2(uint64_t v) {
    float2 r;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
    return r;
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

// one row of the pipelined kernel: hq = the thread's two h values, gp = the row's duplicated coefficient pairs in smem.
// All nine outputs are always computed (unused ones have zero coefficients and zero weights and are never written).
template <int ACT>
__device__ __forceinline__ void hb_row(const uint64_t hq, const float* __restrict__ gp, const uint64_t (&w)[9],
                                       uint64_t (&accw)[9], float (&acc_db)[2], float* __restrict__ dzk) {
    const ulonglong2* g2 = reinterpret_cast<const ulonglong2*>(gp);
    const ulonglong2 p0 = g2[0], p1 = g2[1], p2 = g2[2], p3 = g2[3];
    const uint64_t p8 = *reinterpret_cast<const uint64_t*>(gp + 16);
    const uint64_t g[9] = {p0.x, p0.y, p1.x, p1.y, p2.x, p2.y, p3.x, p3.y, p8};
    uint64_t sacc = 0ull;    // (+0.f, +0.f)
#pragma unroll
    for (int a = 0; a < 9; ++a) {
        sacc = fma2(g[a], w[a], sacc);
        accw[a] = fma2(g[a], hq, accw[a]);
    }
    const float2 hv = unpack2(hq), sv = unpack2(sacc);
    const float d0 = sv.x * act_bwd_from_out(hv.x, ACT), d1 = sv.y * act_bwd_from_out(hv.y, ACT);
    acc_db[0] += d0;
    acc_db[1] += d1;
    *reinterpret_cast<float2*>(dzk) = make_float2(d0, d1);
}

template <int U, int MINB, int ACT>
__global__ void __launch_bounds__(256, MINB) heads_backward_pipe_kernel(
    const float* __restrict__ h, int64_t ldh, int64_t rows, int H, int A, const float* __restrict__ Wv,
    const float* __restrict__ Wa, const float* __restrict__ dlogits, const float* __restrict__ dvalues,
    float* __restrict__ dz, int64_t lddz, float* __restrict__ part, int64_t rows_per_group) {
    constexpr int VW = 2, AP = 9;
    __shared__ __align__(16) float g_s[kHbTile][kHbGP];
    extern __shared__ float red_s[];   // [(A+2)][H] cross-row-lane reduction
    const int n_out = A + 1;
    const int tid = threadIdx.x;
    const int TPR = H / VW, RPB = 256 / TPR;
    const int cv = tid % TPR, rl = tid / TPR;
    const int j = cv * VW;
    const int64_t r_begin = blockIdx.x * rows_per_group;
    const int64_t r_end = (r_begin + rows_per_group < rows) ? r_begin + rows_per_group : rows;
    const int64_t part_stride = (int64_t)(A + 2) * H + n_out;
    float* my_part = part + blockIdx.x * part_stride;

    uint64_t w[AP], accw[AP];
#pragma unroll
    for (int a = 0; a < AP; ++a) {
        accw[a] = 0ull;
        const float* src = (a == 0) ? Wv : Wa + (int64_t)(a - 1) * H;
        w[a] = (a < n_out) ? pack2(src[j], src[j + 1]) : 0ull;
    }
    float acc_db[VW] = {0.f, 0.f};
    float acc_g = 0.f;
    const int kpt = kHbTile / RPB;                                              // k per coefficient tile
    const int K = (int)((r_end - r_begin - rl + RPB - 1) / RPB);                // rows of this thread (may be <= 0)
    const int64_t hstep = (int64_t)RPB * ldh, dstep = (int64_t)RPB * lddz;
    const float* hnext = h + (r_begin + rl) * ldh + j;                          // next row to prefetch
    float* dzk = dz + (r_begin + rl) * lddz + j;                                // next row to write
    uint64_t q[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        q[u] = (u < K) ? __ldg(reinterpret_cast<const unsigned long long*>(hnext)) : 0ull;
        hnext += hstep;
    }

    // (staging one 32-row coefficient tile at a time keeps the resident blocks out of phase; staging a whole row group up
    //  front, with or without L2 prefetches further ahead, measured slower: 54-60 vs 50 us, profiles/r01_m_ncu_heads_backward.md)
    int k = 0;
    for (int64_t b0 = r_begin; b0 < r_end; b0 += kHbTile) {
        const int nb = (int)((r_end - b0 < kHbTile) ? (r_end - b0) : kHbTile);
        __syncthreads();
        for (int i = tid; i < kHbTile * (kHbGP / 2); i += 256) {
            const int bb = i / (kHbGP / 2), a = i - bb * (kHbGP / 2);
            float v = 0.f;
            if (bb < nb && a < n_out) v = (a == 0) ? dvalues[b0 + bb] : dlogits[(b0 + bb) * A + (a - 1)];
            *reinterpret_cast<float2*>(&g_s[bb][2 * a]) = make_float2(v, v);
        }
        __syncthreads();
        if (tid < n_out)
            for (int bb = 0; bb < nb; ++bb) acc_g += g_s[bb][2 * tid];
        const float* gp = &g_s[rl][0];
        for (int kk = 0; kk < kpt; kk += U, k += U) {
            if (k + 2 * U <= K) {          // a full batch whose prefetches are all in range: no guards
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const uint64_t hq = q[u];
                    q[u] = __ldg(reinterpret_cast<const unsigned long long*>(hnext));
                    hb_row<ACT>(hq, gp, w, accw, acc_db, dzk);
                    hnext += hstep; dzk += dstep; gp += RPB * kHbGP;
                }
            } else {
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (k + u < K) {
                        const uint64_t hq = q[u];
                        if (k + u + U < K) q[u] = __ldg(reinterpret_cast<const unsigned long long*>(hnext));
                        hb_row<ACT>(hq, gp, w, accw, acc_db, dzk);
                    }
                    hnext += hstep; dzk += dstep; gp += RPB * kHbGP;
                }
            }
        }
    }
    // combine the RPB row lanes (fixed order -> deterministic)
    for (int r = 0; r < RPB; ++r) {
        __syncthreads();
        if (rl == r) {
#pragma unroll
            for (int a = 0; a < AP; ++a) {
                if (a < n_out) {
                    float2 v = unpack2(accw[a]);
                    if (r > 0) { v.x += red_s[a * H + j]; v.y += red_s[a * H + j + 1]; }
                    red_s[a * H + j] = v.x;
                    red_s[a * H + j + 1] = v.y;
                }
            }
#pragma unroll
            for (int c = 0; c < VW; ++c) {
                float v = acc_db[c];
                if (r > 0) v += red_s[n_out * H + j + c];
                red_s[n_out * H + j + c] = v;
            }
        }
    }
    __syncthreads();
    for (int i = tid; i < (A + 2) * H; i += 256) my_part[i] = red_s[i];
    if (tid < n_out) my_part[(int64_t)(A + 2) * H + tid] = acc_g;
}

static void launch_heads_backward_pipe(int act, unsigned groups, size_t red_bytes, cudaStream_t st, const float* h,
                                       int64_t ldh, int64_t rows, int H, int A, const float* Wv, const float* Wa,
                                       const float* dlogits, const float* dvalues, float* dz, int64_t lddz, float* part,
                                       int64_t rpg) {
#define SFB_HBP(ACT)                                                                                                      \
    heads_backward_pipe_kernel<8, 3, ACT><<<groups, 256, red_bytes, st>>>(h, ldh, rows, H, A, Wv, Wa, dlogits, dvalues, dz,  \
                                                                          lddz, part, rpg)
    switch (act) {
        case SFB200_ACT_ELU: SFB_HBP(SFB200_ACT_ELU); break;
        case SFB200_ACT_RELU: SFB_HBP(SFB200_ACT_RELU); break;
        case SFB200_ACT_TANH: SFB_HBP(SFB200_ACT_TANH); break;
        default: SFB_HBP(SFB200_ACT_NONE); break;
    }
#undef SFB_HBP
}

__global__ void heads_backward_reduce_kernel(const float* __restrict__ part, int groups, int H, int A,
                                             float* __restrict__ dWv, float* __restrict__ dbv, float* __restrict__ dWa,
                                             float* __restrict__ dba, float* __restrict__ db_prev) {
    // one warp per output element, lanes stride over the row groups (fixed mapping + butterfly -> deterministic)
    const int64_t part_stride = (int64_t)(A + 2) * H + (A + 1);
    const int lane = threadIdx.x & 31;
    const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (i >= part_stride) return;
    float s = 0.f;
    for (int g = lane; g < groups; g += 32) s += part[g * part_stride + i];
    s = warp_sum(s);
    if (lane != 0) return;
    const int64_t wsz = (int64_t)(A + 1) * H;
    if (i < H) dWv[i] = s;
    else if (i < wsz) dWa[i - H] = s;
    else if (i < wsz + H) { if (db_prev) db_prev[i - wsz] = s; }
    else {
        const int a = (int)(i - wsz - H);
        if (a == 0) dbv[0] = s; else dba[a - 1] = s;
    }
}

// sampling mode of the calling host thread (sfb200_set_sampling_mode), read by every heads entry that samples actions
static thread_local const uint8_t* g_action_mask = nullptr;
static thread_local int64_t g_mask_stride = 0;
static thread_local int g_deterministic = 0;

static int apply_sampling_mode(HeadsOut& out, int A) {
    if (out.actions_f32 == nullptr) return 0;     // values / distribution parameters only: nothing is sampled
    out.deterministic = g_deterministic;
    if (g_action_mask) {
        SFB_CHECK_ARG(out.dist == 0 && out.num_seg <= 1,
                      "action masks are supported for a plain Discrete action space only (the reference indexes a Tuple's "
                      "mask by head along the batch axis, action_distributions.py:224)");
        SFB_CHECK_ARG(g_mask_stride >= A, "action mask: row stride %lld < %d actions", (long long)g_mask_stride, A);
        out.action_mask = g_action_mask;
        out.mask_stride = g_mask_stride;
    }
    return 0;
}

template <int AP, int RPW, bool VEC>
static int launch_heads_forward(const float* h, int64_t ldh, int64_t rows, int H, int A, const float* Wv,
                                const float* bv, const float* Wa, const float* ba, const HeadsOut& out,
                                const float* noise, uint64_t seed, uint64_t offset, const int64_t* offset_dev,
                                const float* pv_scalar, cudaStream_t st) {
    const size_t smem = VEC ? 0 : (size_t)(A + 1) * H * sizeof(float);
    auto kern = heads_forward_kernel<AP, RPW, VEC>;
    if (smem > 48 * 1024) SFB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t blocks = ceil_div(ceil_div(rows, RPW), 8);
    const int64_t cap = (int64_t)sm_count() * 4;
    if (blocks > cap) blocks = cap;
    SFB_CUDA_OK(launch_pdl(kern, dim3((unsigned)blocks), dim3(256), smem, st, h, ldh, rows, H, A, Wv, bv, Wa, ba, out, noise,
                           seed, offset, offset_dev, pv_scalar));
    SFB_LAUNCH_OK();
    return 0;
}

// A = rows of distribution_linear (n for Discrete(n); 2*act_dim or act_dim for a Box action space)
static int heads_forward_impl(const float* h, int64_t ldh, int64_t rows, int H, int A, const float* Wv, const float* bv,
                              const float* Wa, const float* ba, const HeadsOut& out_in, const float* noise, uint64_t seed,
                              uint64_t offset, const int64_t* offset_dev, const float* pv_scalar, cudaStream_t st) {
    HeadsOut out = out_in;
    if (int rc = apply_sampling_mode(out, A)) return rc;
    SFB_CHECK_ARG(h && Wv && bv && Wa && ba && out.values && rows >= 0 && H > 0, "heads_forward: bad arguments");
    SFB_CHECK_ARG(A >= 1 && A <= 31, "heads_forward: supports 1 <= distribution_linear rows <= 31, got %d", A);
    SFB_CHECK_ARG((size_t)(A + 1) * H * sizeof(float) <= 200 * 1024, "heads_forward: (A+1)*H too large for smem");
    if (rows == 0) return 0;
#define SFB_HF(AP, RPW, VEC)                                                                                          \
    return launch_heads_forward<AP, RPW, VEC>(h, ldh, rows, H, A, Wv, bv, Wa, ba, out, noise, seed, offset, offset_dev, \
                                              pv_scalar, st)
    auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
    const bool vec = (H % 4 == 0) && (ldh % 4 == 0) && al16(h) && al16(Wv) && al16(Wa);
    if (A + 1 <= 9) {
        if (vec && rows <= 8192) SFB_HF(9, 2, true);   // sampler-sized batch: more, smaller warps-of-work
        if (vec) SFB_HF(9, 4, true);
        SFB_HF(9, 4, false);
    }
    if (A + 1 <= 17) {
        if (vec) SFB_HF(17, 2, true);
        SFB_HF(17, 2, false);
    }
    if (vec) SFB_HF(32, 1, true);
    SFB_HF(32, 1, false);
#undef SFB_HF
}

static int heads_from_partials_impl(const float* head_partials, int P, int64_t rows, int A, const float* bv,
                                    const float* ba, const HeadsOut& out_in, const float* noise, uint64_t seed,
                                    uint64_t offset, const int64_t* offset_dev, const float* pv_scalar, cudaStream_t st) {
    HeadsOut out = out_in;
    if (int rc = apply_sampling_mode(out, A)) return rc;
    SFB_CHECK_ARG(head_partials && bv && ba && out.values && rows >= 0 && P >= 1, "heads_from_partials: bad arguments");
    SFB_CHECK_ARG(A >= 1 && A + 1 <= kHeadPartPad, "heads_from_partials: supports 1 <= A <= %d, got %d", kHeadPartPad - 1, A);
    if (rows == 0) return 0;
    int64_t blocks = ceil_div(rows, 8);
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    const HeadsFinish fin{out, bv, ba, noise, seed, offset, offset_dev, pv_scalar, A};
    SFB_CUDA_OK(launch_pdl(heads_from_partials_kernel, dim3((unsigned)blocks), dim3(256), 0, st, head_partials, P, rows, fin));
    SFB_LAUNCH_OK();
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// The rest of a sampler step after the policy GEMMs, for the synthetic tape env (envs.TapeVecEnv, BASELINE config 2), in
// ONE launch: finish the heads + sample (heads_finish_row) -> env step (the rules of tape_env_kernel, elementwise.cu)
// -> advance_rollouts part 2 (post_step_body: reward scale / clip, dones, episode accounting, batched_sampling.py:319-357)
// -> generate_policy_request + normalisation of step t+1 (normalize_body).  Everything is per env, so one warp walks one
// env through all four stages; the three kernel boundaries (and two of the five launches of a policy step) disappear.
// Same device functions / same arithmetic as the separate kernels -> identical trajectories.
struct TapeStepArgs {
    const float* tape; int64_t tape_len; int dim; int num_actions; int64_t env_off; int term_period, trunc_period;
    int64_t* env_step;                                   // [0] env step, [1] block ticket
    float* env_obs; float* env_rew; uint8_t* env_term; uint8_t* env_trunc;
    float reward_scale, reward_clip; int32_t policy_id;
    float* t_rew; uint8_t* t_done; uint8_t* t_to; int32_t* t_pid; int64_t stride;
    float* ep_ret; int32_t* ep_len; float* ep_min; float* ep_max; int32_t len_inc; double* stats;
    int64_t* sampler_step; float* fin_ret; int32_t* fin_len;
    float* traj_obs_next; int64_t traj_obs_stride; float* x_norm; const double* mean; const double* var;
    float sub, inv_scale; int do_sub, do_scale; float eps, clip;
    const float* rnn; int rnn_dim; float* traj_rnn_next; int64_t traj_rnn_stride;
};

__global__ void __launch_bounds__(256) sampler_tail_tape_kernel(const float* __restrict__ part, int P, int64_t rows,
                                                                const HeadsFinish f, const TapeStepArgs a) {
    // per-column normaliser constants once per block (instead of a double load + sqrt + divide per element)
    extern __shared__ float cstat[];   // [2][dim]: mu, 1 / sigma
    const bool do_rms = a.mean != nullptr && a.x_norm != nullptr;
    pdl_wait();
    pdl_trigger();
    if (do_rms) {
        for (int c = threadIdx.x; c < a.dim; c += blockDim.x) col_stats(a.mean, a.var, c, a.eps, cstat[c], cstat[a.dim + c]);
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float pv = f.pv_scalar ? *f.pv_scalar : 0.f;
    const uint64_t offset = f.offset_host + (f.offset_dev ? (uint64_t)*f.offset_dev : 0ull);
    const int64_t step = a.env_step[0];
    const float* src_step = a.tape + ((step + 1) % a.tape_len) * rows * a.dim;
    const bool two = (a.dim == 64);    // the common case: one float2 per lane, issued before the heads math
    for (int64_t row = warp; row < rows; row += nwarps) {
        // ---- everything that does not depend on the sampled action is loaded first (the next observation comes from the
        //      tape whatever the action is; the episode accumulators are lane 0's)
        const float* src = src_step + row * a.dim;
        float2 o2 = make_float2(0.f, 0.f);
        if (two) o2 = *reinterpret_cast<const float2*>(src + 2 * lane);
        float er0 = 0.f, mn0 = 0.f, mx0 = 0.f;
        int32_t el0 = 0;
        if (lane == 0 && a.ep_ret) { er0 = a.ep_ret[row]; el0 = a.ep_len[row]; mn0 = a.ep_min[row]; mx0 = a.ep_max[row]; }
        const int act = heads_finish_row(part, P, rows, row, lane, f, pv, offset);
        // ---- env step
        const int64_t env = a.env_off + row;
        const float r_raw = (float)act / (float)a.num_actions;
        const bool tm = ((step * 7 + env * 13) % a.term_period) == 0;
        const bool tr = (((step + env) % a.trunc_period) == 0) && !tm;
        // ---- next observation: env buffer, trajectory slot t+1, normalised policy input
        if (two) {
            const int c = 2 * lane;
            *reinterpret_cast<float2*>(a.env_obs + row * a.dim + c) = o2;
            *reinterpret_cast<float2*>(a.traj_obs_next + row * a.traj_obs_stride + c) = o2;
            if (a.x_norm) {
                float2 y;
                y.x = norm_one(o2.x, a.sub, a.inv_scale, a.do_sub, a.do_scale, do_rms, do_rms ? cstat[c] : 0.f, do_rms ? cstat[a.dim + c] : 1.f, a.clip);
                y.y = norm_one(o2.y, a.sub, a.inv_scale, a.do_sub, a.do_scale, do_rms, do_rms ? cstat[c + 1] : 0.f, do_rms ? cstat[a.dim + c + 1] : 1.f, a.clip);
                *reinterpret_cast<float2*>(a.x_norm + row * a.dim + c) = y;
            }
        } else {
            for (int c = lane; c < a.dim; c += 32) {
                const float v = src[c];
                a.env_obs[row * a.dim + c] = v;
                a.traj_obs_next[row * a.traj_obs_stride + c] = v;
                if (a.x_norm)
                    a.x_norm[row * a.dim + c] = norm_one(v, a.sub, a.inv_scale, a.do_sub, a.do_scale, do_rms,
                                                         do_rms ? cstat[c] : 0.f, do_rms ? cstat[a.dim + c] : 1.f, a.clip);
            }
        }
        if (a.rnn)
            for (int j = lane; j < a.rnn_dim; j += 32) a.traj_rnn_next[row * a.traj_rnn_stride + j] = a.rnn[row * a.rnn_dim + j];
        // ---- post step (lane 0 owns the env's scalars)
        if (lane == 0) {
            a.env_rew[row] = r_raw;
            a.env_term[row] = tm;
            a.env_trunc[row] = tr;
            const bool done = tm || tr;                                     // batched_sampling.py:317
            float r = __fmul_rn(r_raw, a.reward_scale);                     // :209
            r = clampf(r, -a.reward_clip, a.reward_clip);                   // :210
            a.t_rew[row * a.stride] = r;
            a.t_done[row * a.stride] = done ? 1 : 0;
            a.t_to[row * a.stride] = tr ? 1 : 0;                            // :328
            a.t_pid[row * a.stride] = a.policy_id;
            if (a.ep_ret) {                                                 // _process_env_step :215-287 (raw reward)
                float er = er0 + r_raw;
                int32_t el = el0 + a.len_inc;
                float mn = fminf(mn0, r_raw), mx = fmaxf(mx0, r_raw);
                if (a.fin_ret) {
                    a.fin_ret[row * a.stride] = done ? er : __int_as_float(0x7fc00000);
                    a.fin_len[row * a.stride] = done ? el : -1;
                }
                if (done) {
                    if (a.stats) {
                        atomicAdd(a.stats + 0, 1.0); atomicAdd(a.stats + 1, (double)er); atomicAdd(a.stats + 2, (double)el);
                        atomicAdd(a.stats + 3, (double)mn); atomicAdd(a.stats + 4, (double)mx);
                    }
                    er = 0.f; el = 0; mn = INFINITY; mx = -INFINITY;
                }
                a.ep_ret[row] = er; a.ep_len[row] = el; a.ep_min[row] = mn; a.ep_max[row] = mx;
            }
        }
    }
    // every block has read both counters before taking its ticket, so the last ticket holder may advance them
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        unsigned long long* ticket = reinterpret_cast<unsigned long long*>(a.env_step + 1);
        if (atomicAdd(ticket, 1ull) == (unsigned long long)gridDim.x - 1ull) {
            *ticket = 0ull;
            a.env_step[0] = step + 1;
            if (a.sampler_step) *a.sampler_step += 1;
        }
    }
}

static int make_gaussian_out(HeadsOut& out, int act_dim, int adaptive_stddev, const float* learned_log_std,
                             float tanh_scale, float* values, int64_t values_stride, float* params,
                             int64_t params_stride, float* actions_f32, int64_t actions_stride, float* env_actions_f32,
                             float* log_prob, int64_t log_prob_stride, float* pv_out, int64_t pv_stride) {
    SFB_CHECK_ARG(act_dim >= 1 && (adaptive_stddev ? 2 * act_dim : act_dim) <= 31,
                  "heads (continuous): act_dim %d needs more than 31 distribution_linear rows", act_dim);
    SFB_CHECK_ARG(adaptive_stddev || learned_log_std, "heads (continuous): learned_log_std is required when adaptive_stddev=0");
    out = HeadsOut{values, values_stride, params, params_stride, actions_f32, actions_stride, nullptr, log_prob,
                   log_prob_stride, pv_out, pv_stride, adaptive_stddev ? 1 : 2, act_dim, learned_log_std, tanh_scale,
                   env_actions_f32};
    return 0;
}

}  // namespace sfb

using namespace sfb;

extern "C" {

int sfb200_set_sampling_mode(const uint8_t* action_mask, int64_t mask_row_stride, int deterministic) {
    SFB_CHECK_ARG(action_mask == nullptr || mask_row_stride >= 1, "set_sampling_mode: bad mask stride");
    g_action_mask = action_mask;
    g_mask_stride = action_mask ? mask_row_stride : 0;
    g_deterministic = deterministic ? 1 : 0;
    return 0;
}

int sfb200_heads_forward(const float* h, int64_t ldh, int64_t rows, int H, int A, const float* Wv, const float* bv,
                         const float* Wa, const float* ba, float* values, int64_t values_stride, float* logits,
                         int64_t logits_stride, const float* noise, uint64_t philox_seed, uint64_t philox_offset,
                         const int64_t* philox_offset_dev, float* actions_f32, int64_t actions_stride, int32_t* env_actions_i32, float* log_prob,
                         int64_t log_prob_stride, const float* policy_version_scalar, float* policy_version_out,
                         int64_t pv_stride, void* stream) {
    const HeadsOut out{values, values_stride, logits, logits_stride, actions_f32, actions_stride, env_actions_i32,
                       log_prob, log_prob_stride, policy_version_out, pv_stride, 0, 0, nullptr, 0.f, nullptr};
    return heads_forward_impl(h, ldh, rows, H, A, Wv, bv, Wa, ba, out, noise, philox_seed, philox_offset,
                              philox_offset_dev, policy_version_scalar, (cudaStream_t)stream);
}

int sfb200_heads_from_partials(const float* head_partials, int P, int64_t rows, int A, const float* bv, const float* ba,
                               float* values, int64_t values_stride, float* logits, int64_t logits_stride,
                               const float* noise, uint64_t philox_seed, uint64_t philox_offset,
                               const int64_t* philox_offset_dev, float* actions_f32, int64_t actions_stride,
                               int32_t* env_actions_i32, float* log_prob, int64_t log_prob_stride,
                               const float* policy_version_scalar, float* policy_version_out, int64_t pv_stride,
                               void* stream) {
    const HeadsOut out{values, values_stride, logits, logits_stride, actions_f32, actions_stride, env_actions_i32,
                       log_prob, log_prob_stride, policy_version_out, pv_stride, 0, 0, nullptr, 0.f, nullptr};
    return heads_from_partials_impl(head_partials, P, rows, A, bv, ba, out, noise, philox_seed, philox_offset,
                                    philox_offset_dev, policy_version_scalar, (cudaStream_t)stream);
}

int sfb200_sampler_tail_tape_step(const float* head_partials, int P, int64_t n_envs, int A, const float* bv, const float* ba,
                                  float* values_t, int64_t values_stride, float* logits_t, int64_t logits_stride,
                                  const float* noise, uint64_t philox_seed, int64_t* sampler_step, float* actions_t,
                                  int64_t actions_stride, int32_t* env_actions, float* log_prob_t, int64_t log_prob_stride,
                                  const float* policy_version_scalar, float* policy_version_t, int64_t pv_stride,
                                  const float* tape, int64_t tape_len, int dim, int64_t env_index_offset, int term_period,
                                  int trunc_period, int64_t* env_step_counter, float* env_obs, float* env_rew,
                                  uint8_t* env_terminated, uint8_t* env_truncated, float reward_scale, float reward_clip,
                                  int32_t policy_id, float* traj_rewards_t, uint8_t* traj_dones_t, uint8_t* traj_time_outs_t,
                                  int32_t* traj_policy_id_t, int64_t traj_stride, float* ep_return, int32_t* ep_len,
                                  float* ep_min_raw, float* ep_max_raw, int32_t len_increment, double* stats,
                                  float* fin_return_t, int32_t* fin_len_t, float* traj_obs_next, int64_t traj_obs_stride,
                                  const float* rnn, int rnn_dim, float* traj_rnn_next, int64_t traj_rnn_stride, float* x_norm,
                                  const double* mean, const double* var, float sub_mean, float inv_scale, float eps,
                                  float clip, void* stream) {
    HeadsOut out{values_t, values_stride, logits_t, logits_stride, actions_t, actions_stride, env_actions,
                 log_prob_t, log_prob_stride, policy_version_t, pv_stride, 0, 0, nullptr, 0.f, nullptr};
    if (int rc = apply_sampling_mode(out, A)) return rc;
    SFB_CHECK_ARG(head_partials && bv && ba && values_t && actions_t && env_actions && n_envs >= 0 && P >= 1 && A >= 1 &&
                      A + 1 <= kHeadPartPad, "sampler_tail_tape_step: bad heads arguments");
    SFB_CHECK_ARG(tape && tape_len > 0 && dim > 0 && term_period > 0 && trunc_period > 0 && env_step_counter && env_obs &&
                      env_rew && env_terminated && env_truncated, "sampler_tail_tape_step: bad env arguments");
    SFB_CHECK_ARG(traj_rewards_t && traj_dones_t && traj_time_outs_t && traj_policy_id_t && traj_obs_next,
                  "sampler_tail_tape_step: bad trajectory arguments");
    SFB_CHECK_ARG((mean == nullptr) == (var == nullptr), "sampler_tail_tape_step: mean/var must both be set or both NULL");
    SFB_CHECK_ARG((ep_return == nullptr) == (ep_len == nullptr) && (ep_return == nullptr) == (ep_min_raw == nullptr) &&
                      (ep_return == nullptr) == (ep_max_raw == nullptr), "sampler_tail_tape_step: episode buffers all or none");
    if (n_envs == 0) return 0;
    const bool with_rnn = rnn && traj_rnn_next && rnn_dim > 0;
    const TapeStepArgs a{tape, tape_len, dim, A, env_index_offset, term_period, trunc_period, env_step_counter, env_obs, env_rew,
                         env_terminated, env_truncated, reward_scale, reward_clip, policy_id, traj_rewards_t, traj_dones_t,
                         traj_time_outs_t, traj_policy_id_t, traj_stride, ep_return, ep_len, ep_min_raw, ep_max_raw,
                         len_increment, stats, sampler_step, fin_return_t, fin_len_t, traj_obs_next, traj_obs_stride, x_norm,
                         mean, var, sub_mean, inv_scale, fabsf(sub_mean) > 1e-8f ? 1 : 0, fabsf(inv_scale - 1.0f) > 1e-8f ? 1 : 0,
                         eps, clip, with_rnn ? rnn : nullptr, rnn_dim, traj_rnn_next, traj_rnn_stride};
    const HeadsFinish fin{out, bv, ba, noise, philox_seed, 0ull, sampler_step, policy_version_scalar, A};
    int64_t blocks = ceil_div(n_envs, 8);
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    SFB_CHECK_ARG(dim <= 4096, "sampler_tail_tape_step: observation rows of up to 4096 floats");
    SFB_CUDA_OK(launch_pdl(sampler_tail_tape_kernel, dim3((unsigned)blocks), dim3(256), (size_t)(2 * dim * sizeof(float)),
                           (cudaStream_t)stream, head_partials, P, n_envs, fin, a));
    SFB_LAUNCH_OK();
    return 0;
}

static int make_tuple_out(HeadsOut& out, int A, int num_seg, const int32_t* seg_lens) {
    SFB_CHECK_ARG(num_seg >= 1 && num_seg <= 8 && seg_lens, "heads (tuple): 1 <= number of heads <= 8");
    int tot = 0;
    for (int k = 0; k < num_seg; ++k) {
        SFB_CHECK_ARG(seg_lens[k] >= 1, "heads (tuple): empty head");
        out.seg_len[k] = seg_lens[k];
        tot += seg_lens[k];
    }
    SFB_CHECK_ARG(tot == A, "heads (tuple): the heads' sizes sum to %d but distribution_linear has %d rows", tot, A);
    out.num_seg = num_seg;
    return 0;
}

int sfb200_heads_forward_tuple(const float* h, int64_t ldh, int64_t rows, int H, int A, int num_heads,
                               const int32_t* head_sizes_host, const float* Wv, const float* bv, const float* Wa,
                               const float* ba, float* values, int64_t values_stride, float* logits,
                               int64_t logits_stride, const float* noise, uint64_t philox_seed, uint64_t philox_offset,
                               const int64_t* philox_offset_dev, float* actions_f32, int64_t actions_stride,
                               int32_t* env_actions_i32, float* log_prob, int64_t log_prob_stride,
                               const float* policy_version_scalar, float* policy_version_out, int64_t pv_stride,
                               void* stream) {
    HeadsOut out{values, values_stride, logits, logits_stride, actions_f32, actions_stride, env_actions_i32,
                 log_prob, log_prob_stride, policy_version_out, pv_stride, 0, 0, nullptr, 0.f, nullptr};
    if (int rc = make_tuple_out(out, A, num_heads, head_sizes_host)) return rc;
    return heads_forward_impl(h, ldh, rows, H, A, Wv, bv, Wa, ba, out, noise, philox_seed, philox_offset,
                              philox_offset_dev, policy_version_scalar, (cudaStream_t)stream);
}

int sfb200_heads_from_partials_tuple(const float* head_partials, int P, int64_t rows, int A, int num_heads,
                                     const int32_t* head_sizes_host, const float* bv, const float* ba, float* values,
                                     int64_t values_stride, float* logits, int64_t logits_stride, const float* noise,
                                     uint64_t philox_seed, uint64_t philox_offset, const int64_t* philox_offset_dev,
                                     float* actions_f32, int64_t actions_stride, int32_t* env_actions_i32,
                                     float* log_prob, int64_t log_prob_stride, const float* policy_version_scalar,
                                     float* policy_version_out, int64_t pv_stride, void* stream) {
    HeadsOut out{values, values_stride, logits, logits_stride, actions_f32, actions_stride, env_actions_i32,
                 log_prob, log_prob_stride, policy_version_out, pv_stride, 0, 0, nullptr, 0.f, nullptr};
    if (int rc = make_tuple_out(out, A, num_heads, head_sizes_host)) return rc;
    return heads_from_partials_impl(head_partials, P, rows, A, bv, ba, out, noise, philox_seed, philox_offset,
                                    philox_offset_dev, policy_version_scalar, (cudaStream_t)stream);
}

int sfb200_heads_forward_continuous(const float* h, int64_t ldh, int64_t rows, int H, int act_dim, int adaptive_stddev,
                                    const float* Wv, const float* bv, const float* Wa, const float* ba,
                                    const float* learned_log_std, float tanh_scale, float* values,
                                    int64_t values_stride, float* params, int64_t params_stride, const float* noise,
                                    uint64_t philox_seed, uint64_t philox_offset, const int64_t* philox_offset_dev,
                                    float* actions_f32, int64_t actions_stride, float* env_actions_f32, float* log_prob,
                                    int64_t log_prob_stride, const float* policy_version_scalar,
                                    float* policy_version_out, int64_t pv_stride, void* stream) {
    HeadsOut out;
    if (int rc = make_gaussian_out(out, act_dim, adaptive_stddev, learned_log_std, tanh_scale, values, values_stride, params,
                                   params_stride, actions_f32, actions_stride, env_actions_f32, log_prob, log_prob_stride,
                                   policy_version_out, pv_stride))
        return rc;
    return heads_forward_impl(h, ldh, rows, H, adaptive_stddev ? 2 * act_dim : act_dim, Wv, bv, Wa, ba, out, noise,
                              philox_seed, philox_offset, philox_offset_dev, policy_version_scalar, (cudaStream_t)stream);
}

int sfb200_heads_from_partials_continuous(const float* head_partials, int P, int64_t rows, int act_dim,
                                          int adaptive_stddev, const float* bv, const float* ba,
                                          const float* learned_log_std, float tanh_scale, float* values,
                                          int64_t values_stride, float* params, int64_t params_stride,
                                          const float* noise, uint64_t philox_seed, uint64_t philox_offset,
                                          const int64_t* philox_offset_dev, float* actions_f32, int64_t actions_stride,
                                          float* env_actions_f32, float* log_prob, int64_t log_prob_stride,
                                          const float* policy_version_scalar, float* policy_version_out,
                                          int64_t pv_stride, void* stream) {
    HeadsOut out;
    if (int rc = make_gaussian_out(out, act_dim, adaptive_stddev, learned_log_std, tanh_scale, values, values_stride, params,
                                   params_stride, actions_f32, actions_stride, env_actions_f32, log_prob, log_prob_stride,
                                   policy_version_out, pv_stride))
        return rc;
    return heads_from_partials_impl(head_partials, P, rows, adaptive_stddev ? 2 * act_dim : act_dim, bv, ba, out, noise,
                                    philox_seed, philox_offset, philox_offset_dev, policy_version_scalar,
                                    (cudaStream_t)stream);
}

int64_t sfb200_heads_backward_workspace_bytes(int H, int A) {
    return (int64_t)kHeadsMaxGroups * ((int64_t)(A + 2) * H + (A + 1)) * (int64_t)sizeof(float);
}

int sfb200_heads_backward(const float* h, int64_t ldh, int64_t rows, int H, int A, const float* Wv, const float* Wa,
                          const float* dlogits, const float* dvalues, int act, float* dz, int64_t lddz, float* dWv,
                          float* dbv, float* dWa, float* dba, float* db_prev, void* workspace, void* stream) {
    SFB_CHECK_ARG(h && Wv && Wa && dlogits && dvalues && dz && dWv && dbv && dWa && dba && workspace && rows > 0 && H > 0,
                  "heads_backward: bad arguments");
    SFB_CHECK_ARG(A >= 1 && A <= 31, "heads_backward: supports 1 <= A <= 31, got %d", A);
    cudaStream_t st = (cudaStream_t)stream;
    auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
    const size_t red_bytes = (size_t)(A + 2) * H * sizeof(float);
    const bool vec_common = (ldh % 4 == 0) && (lddz % 4 == 0) && al16(h) && al16(dz) && al16(Wv) && al16(Wa) &&
                            red_bytes <= 40 * 1024 && A + 1 <= 9;
    // two columns per thread (64 registers, 4 blocks per SM) when a row fills a whole block, else four
    const bool vec2 = vec_common && (H % 2 == 0) && (H / 2 <= 256) && (256 % (H / 2) == 0) && rows >= 16384;
    const bool vec4 = vec_common && (H % 4 == 0) && (H / 4 <= 256) && (256 % (H / 4) == 0);
    // pipelined row loads (see heads_backward_pipe_kernel): rows per thread and tile must be a multiple of the queue depth
    const bool pipe = vec2 && (kHbTile / (256 / (H / 2))) % 8 == 0;
    int64_t groups = (int64_t)sm_count() * (pipe ? 3 : (vec2 ? 4 : 2));
    if (groups > kHeadsMaxGroups) groups = kHeadsMaxGroups;
    int64_t rpg = ceil_div(rows, groups);
    if (!pipe) rpg = ceil_div(rpg, kHbTile) * kHbTile;     // (the pipelined kernel fills exactly one wave instead)
    groups = ceil_div(rows, rpg);
    float* part = (float*)workspace;
    if (pipe)
        launch_heads_backward_pipe(act, (unsigned)groups, red_bytes, st, h, ldh, rows, H, A, Wv, Wa, dlogits, dvalues, dz, lddz,
                                   part, rpg);
    else if (vec2)
        heads_backward_vec_kernel<9, 2, 8, 4><<<(unsigned)groups, 256, red_bytes, st>>>(h, ldh, rows, H, A, Wv, Wa, dlogits,
                                                                                        dvalues, act, dz, lddz, part, rpg);
    else if (vec4)
        heads_backward_vec_kernel<9, 4, 4, 2><<<(unsigned)groups, 256, red_bytes, st>>>(h, ldh, rows, H, A, Wv, Wa, dlogits,
                                                                                        dvalues, act, dz, lddz, part, rpg);
    else if (A + 1 <= 9)
        heads_backward_kernel<9><<<(unsigned)groups, 256, 0, st>>>(h, ldh, rows, H, A, Wv, Wa, dlogits, dvalues, act, dz,
                                                                   lddz, part, rpg);
    else if (A + 1 <= 17)
        heads_backward_kernel<17><<<(unsigned)groups, 256, 0, st>>>(h, ldh, rows, H, A, Wv, Wa, dlogits, dvalues, act,
                                                                    dz, lddz, part, rpg);
    else
        heads_backward_kernel<32><<<(unsigned)groups, 256, 0, st>>>(h, ldh, rows, H, A, Wv, Wa, dlogits, dvalues, act,
                                                                    dz, lddz, part, rpg);
    SFB_LAUNCH_OK();
    const int64_t total = (int64_t)(A + 2) * H + (A + 1);
    heads_backward_reduce_kernel<<<(unsigned)ceil_div(total * 32, 256), 256, 0, st>>>(part, (int)groups, H, A, dWv, dbv, dWa,
                                                                                 dba, db_prev);
    SFB_LAUNCH_OK();
    return 0;
}

}  // extern "C"
