// A whole rollout of the cfg-2 class of policies (two-layer MLP, Discrete actions, synthetic tape env) as ONE persistent
// kernel: `T` env steps x { layer-1 GEMM, layer-2 GEMM + head partials, heads finish + sampling + env step + post-step +
// pre-step of the next step } without leaving the SMs (batched_sampling.py:298-388 + inference_worker.py:313-341 +
// actor_critic.py:160-195 for every step of the rollout).
//
// Decomposition: all data dependencies of a step stay inside a 128-row block of envs -- layer 2 needs all H1 columns of the
// block's h1, the heads need all H2 columns of its h2, the next step's layer 1 needs the block's new observations -- so a
// thread-block CLUSTER of CX = H2/128 CTAs owns a row block for the whole rollout and the only synchronisation is the
// cluster barrier (three per step); there is no grid-wide barrier and no kernel boundary.  CTA c of the cluster computes
// columns [128c, 128c+128) of h1, then of h2 (partial head products), then finishes rows [32c.., ) of the block.
// h1 and the head partials cross between the CTAs of a cluster through global memory (L2-resident: 256 KB per block);
// DSMEM would move ~21 B/clk (B300_MICROARCH), the L2 path is a TMA load like any other A operand.
//
// Each GEMM tile is the TMEM-A pipeline of gemm_tc.cu (A raw via TMA -> operand warps split it into tensor memory; B =
// registered weights, hi and lo tiles straight from TMA; 3xTF32 with main | cross accumulators), the step tail is the code of
// sampler_tail_tape_kernel (heads.cu).  What the persistent form removes per step: two kernel launches + their prologues
// (TMEM allocation, barrier init, descriptor prefetch, bias / head-weight staging) and the launch-to-launch dependency gaps.
//
//   warp 0      TMA producer            warp 1      MMA issuer (+ TMEM allocation)
//   warps 2-5   operand warps           warps 6-13  epilogues (h1 tile store; h2 -> head partials)
//   warps 6-13  the step tail (an 8-lane group per row: four rows per warp, the CTA's 32 rows in one pass)
#include <cuda.h>

#include "common.cuh"
#include "gemm.h"
#include "heads_tail.cuh"
#include "tc_ptx.cuh"

namespace sfb {

constexpr int RF_THREADS = 448;
constexpr int RF_TILE_BYTES = 128 * TBK * 4;          // 16 KB: one [128 rows][32 fp32] (or [128][64 fp16]) K-major swizzled tile
// tf32 split: 4 stages of 32 k, [B hi | B lo | A raw].  fp16 split (F16): 3 stages of 64 k, [B hi16 | B lo16 | A raw x 2]
template <bool F16> struct RfPipe {
    static constexpr int STAGES = F16 ? 3 : 4;
    static constexpr int KB_K = F16 ? 64 : 32;
    static constexpr int STAGE_BYTES = (F16 ? 4 : 3) * RF_TILE_BYTES;
};
constexpr int RF_MAX_STAGES = 4;
constexpr uint32_t RF_ACOL0 = 256;                    // TMEM: accumulator [0,256) (main | cross), A stages [256, 512)
constexpr int RF_HEAD_AP = 9;
constexpr int RF_MAX_DIM = 128;

struct RfSmem {
    static constexpr int OFF_BARS = 4 * 3 * RF_TILE_BYTES;      // == 3 * 4 * RF_TILE_BYTES: both pipelines fill 192 KB
    static constexpr int OFF_B1 = OFF_BARS + 256;
    static constexpr int OFF_B2 = OFF_B1 + 128 * 4;
    static constexpr int OFF_HEADW = OFF_B2 + 128 * 4;
    static constexpr int OFF_CSTAT = OFF_HEADW + RF_HEAD_AP * 128 * 4;
    static constexpr int TOTAL = OFF_CSTAT + 2 * RF_MAX_DIM * 4 + 1024 /*align slack*/;
};

struct RolloutArgs {
    int64_t N; int T, K1, H1, H2;
    const float* b1; const float* b2; const float* wv; const float* wa; int A; const float* bv; const float* ba;
    float* h1; float* part; float* x_norm;
    // trajectory slots of step 0 (slot t = + t * per-step element count), row strides in elements
    float* values; int64_t values_rs; float* logits; int64_t logits_rs; float* actions; int64_t actions_rs;
    int32_t* env_actions; float* log_prob; int64_t lp_rs; float* pv_out; int64_t pv_rs; const float* pv_scalar;
    const float* noise; uint64_t seed; int64_t* sampler_step;
    // tape env
    const float* tape; int64_t tape_len; int64_t env_off; int term_period, trunc_period; int64_t* env_step;
    float* env_obs; float* env_rew; uint8_t* env_term; uint8_t* env_trunc;
    // post step
    float reward_scale, reward_clip; int32_t policy_id; float* t_rew; uint8_t* t_done; uint8_t* t_to; int32_t* t_pid; int64_t stride;
    float* ep_ret; int32_t* ep_len; float* ep_min; float* ep_max; int32_t len_inc; double* stats; float* fin_ret; int32_t* fin_len;
    // pre step
    float* traj_obs; int64_t traj_obs_rs; const float* rnn; int rnn_dim; float* traj_rnn; int64_t traj_rnn_rs;
    const double* mean; const double* var; float sub, inv_scale; int do_sub, do_scale; float eps, clip;
    unsigned int* ticket;
    unsigned long long* trace;   // debug: [T][16] globaltimer stamps of CTA (0,0)'s first epilogue thread, or NULL
    const float* bound_x; const float* bound_h1;   // fp16-split form: bounds of |x_norm| and |h1| (device floats), else NULL
};

__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// generic-proxy global stores -> async-proxy (TMA) loads: the .global form is a single FENCE.VIEW.ASYNC.G; the unqualified
// form adds a MEMBAR.ALL.GPU (the cluster barrier's release already carries one)
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ unsigned long long rf_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}

// bounded spin: a protocol bug traps instead of hanging the GPU
__device__ __forceinline__ void rf_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done = 0;
    uint64_t t0 = 0;
    for (uint32_t spins = 0; !done; ++spins) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if ((spins & 1023u) == 1023u) {
            uint64_t now;
            asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 2000000000ull) __trap();
        }
    }
}

template <int ACT, bool F16>
__global__ void __launch_bounds__(RF_THREADS, 1)
rollout_mlp2_tape_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w1,
                         const __grid_constant__ CUtensorMap tmap_w1lo, const __grid_constant__ CUtensorMap tmap_h1,
                         const __grid_constant__ CUtensorMap tmap_w2, const __grid_constant__ CUtensorMap tmap_w2lo,
                         const RolloutArgs a) {
    using S = RfSmem;
    constexpr int RF_STAGES = RfPipe<F16>::STAGES, RF_STAGE_BYTES = RfPipe<F16>::STAGE_BYTES, KB_K = RfPipe<F16>::KB_K;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_align_1024(smem_raw);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BARS);
    uint64_t* full = bars;                       // [stages] A and B tiles landed (TMA)
    uint64_t* conv = bars + RF_MAX_STAGES;       // [stages] A in TMEM (128 operand threads)
    uint64_t* empty = bars + 2 * RF_MAX_STAGES;  // [stages] MMAs of the stage retired
    uint64_t* acc_full = bars + 3 * RF_MAX_STAGES;
    uint64_t* acc_empty = bars + 3 * RF_MAX_STAGES + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * RF_MAX_STAGES + 2);
    float* b1_s = reinterpret_cast<float*>(smem + S::OFF_B1);         // this CTA's 128 columns of b1
    float* b2_s = reinterpret_cast<float*>(smem + S::OFF_B2);
    float* headw_s = reinterpret_cast<float*>(smem + S::OFF_HEADW);   // [9][128]
    float* cstat = reinterpret_cast<float*>(smem + S::OFF_CSTAT);     // [2][K1]: mu, 1 / sigma of the observation normaliser

    // episode statistics of finished episodes: accumulated per CTA over the WHOLE rollout in shared memory, five global
    // atomics per CTA at the end (the per-step launches issue them per finished episode: ~370 per step on five addresses --
    // inside this kernel every cluster barrier's release would have to wait for those same-address atomics to drain)
    __shared__ double s_stats[5];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x < 5) s_stats[threadIdx.x] = 0.0;
    const int cx = (int)cluster_ctarank();           // == blockIdx.x (cluster spans the x dimension)
    const int CX = gridDim.x;
    const int n0 = cx * 128;
    const int64_t m0 = (int64_t)blockIdx.y * 128;
    const int KB1 = a.K1 / KB_K, KB2 = a.H1 / KB_K;
    const int P = 2 * CX;
    const bool do_rms = a.mean != nullptr;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_x) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_w1) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_w1lo) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_h1) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_w2) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_w2lo) : "memory");
        for (int s = 0; s < RF_STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&conv[s], 128);
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
    pdl_wait();
    pdl_trigger();
    // constants of the whole rollout -> shared memory (epilogue warps)
    if (warp >= 6) {
        const int et = threadIdx.x - 192;   // 0..255
        if (et < 128) { b1_s[et] = a.b1[n0 + et]; b2_s[et] = a.b2[n0 + et]; }
        for (int i = et; i < RF_HEAD_AP * 128; i += 256) {
            const int r = i >> 7, n = i & 127;
            headw_s[i] = (r == 0) ? a.wv[n0 + n] : (r <= a.A ? a.wa[(int64_t)(r - 1) * a.H2 + n0 + n] : 0.f);
        }
        if (do_rms)
            for (int c = et; c < a.K1; c += 256) col_stats(a.mean, a.var, c, a.eps, cstat[c], cstat[a.K1 + c]);
    }
    __syncthreads();
    // fp16-split form: binary shifts of the two activation operands from their bounds (constant over the rollout: the
    // weights, hence the bounds, do not change inside a rollout)
    const int shift_x = F16 ? f16_shift_for_bound(a.bound_x[0]) : 0;
    const int shift_h = F16 ? f16_shift_for_bound(a.bound_h1[0]) : 0;
    const int64_t env_step0 = a.env_step[0];
    const uint64_t philox0 = a.sampler_step ? (uint64_t)*a.sampler_step : 0ull;
    const float pv = a.pv_scalar ? *a.pv_scalar : 0.f;

    int pref = 0;             // producer: stages of the current tile already armed + weight tiles requested
    const bool tracer = a.trace != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 192;
#define RF_TRACE(slot) do { if (tracer) a.trace[(int64_t)t * 16 + (slot)] = rf_now(); } while (0)
    uint32_t it = 0;          // stage use counter (every role advances it identically)
    uint32_t tile_iter = 0;   // accumulator use counter

    for (int t = 0; t < a.T; ++t) {
        RF_TRACE(0);
#pragma unroll 1
        for (int layer = 0; layer < 2; ++layer) {
            const int num_kb = layer == 0 ? KB1 : KB2;
            if (warp == 0) {
                // ===================================================== TMA producer
                if (lane == 0) {
                    if (layer == 1 || t > 0) fence_proxy_async_all();   // peers' generic-proxy writes (h1 / x_norm) -> TMA reads
                    const CUtensorMap* ta = layer == 0 ? &tmap_x : &tmap_h1;
                    const CUtensorMap* tb = layer == 0 ? &tmap_w1 : &tmap_w2;
                    const CUtensorMap* tbl = layer == 0 ? &tmap_w1lo : &tmap_w2lo;
                    for (int kb = 0; kb < num_kb; ++kb) {
                        const uint32_t i = it + kb;
                        const int s = i % RF_STAGES;
                        uint8_t* sb = smem + s * RF_STAGE_BYTES;
                        if (kb >= pref) {      // (the first `pref` stages were armed and their weight tiles requested before the barrier)
                            rf_wait(&empty[s], ((i / RF_STAGES) & 1) ^ 1);
                            mbar_expect_tx(&full[s], RF_STAGE_BYTES);
                            tma_load_2d(sb, tb, &full[s], kb * KB_K, n0);
                            tma_load_2d(sb + RF_TILE_BYTES, tbl, &full[s], kb * KB_K, n0);
                        }
                        tma_load_2d(sb + 2 * RF_TILE_BYTES, ta, &full[s], kb * KB_K, (int)m0);
                        if (F16) tma_load_2d(sb + 3 * RF_TILE_BYTES, ta, &full[s], kb * KB_K + 32, (int)m0);
                    }
                    // weight tiles of the NEXT tile do not depend on the cluster barrier: request them now, so that only the
                    // activation tiles' latency is exposed after it
                    pref = 0;
                    const bool has_next = (layer == 0) || (t + 1 < a.T);
                    if (has_next) {
                        const int nkb = layer == 0 ? KB2 : KB1;
                        const CUtensorMap* nb = layer == 0 ? &tmap_w2 : &tmap_w1;
                        const CUtensorMap* nbl = layer == 0 ? &tmap_w2lo : &tmap_w1lo;
                        pref = nkb < RF_STAGES ? nkb : RF_STAGES;
                        for (int kb = 0; kb < pref; ++kb) {
                            const uint32_t i = it + num_kb + kb;
                            const int s = i % RF_STAGES;
                            uint8_t* sb = smem + s * RF_STAGE_BYTES;
                            rf_wait(&empty[s], ((i / RF_STAGES) & 1) ^ 1);
                            mbar_expect_tx(&full[s], RF_STAGE_BYTES);
                            tma_load_2d(sb, nb, &full[s], kb * KB_K, n0);
                            tma_load_2d(sb + RF_TILE_BYTES, nbl, &full[s], kb * KB_K, n0);
                        }
                    }
                }
                __syncwarp();
            } else if (warp == 1) {
                // ===================================================== MMA issuer
                constexpr uint32_t idesc_wide = F16 ? make_idesc_f16(TBM, 256) : make_idesc(false, false, TBM, 256);
                constexpr uint32_t idesc_cross = F16 ? make_idesc_f16(TBM, 128) : make_idesc(false, false, TBM, 128);
                rf_wait(acc_empty, (tile_iter & 1) ^ 1);
                tc_fence_after();
                for (int kb = 0; kb < num_kb; ++kb) {
                    const uint32_t i = it + kb;
                    const int s = i % RF_STAGES;
                    rf_wait(&full[s], (i / RF_STAGES) & 1);    // B tiles come straight from TMA
                    rf_wait(&conv[s], (i / RF_STAGES) & 1);    // A halves are in tensor memory
                    tc_fence_after();
                    if (lane == 0) {
                        const uint64_t db = make_smem_desc(smem_u32(smem + s * RF_STAGE_BYTES), false);
                        const uint32_t a_hi = tmem_base + RF_ACOL0 + (uint32_t)s * 64u;
#pragma unroll
                        for (int k = 0; k < TBK / UMMA_K; ++k) {
                            const uint64_t bo = (uint64_t)(k * (UMMA_K * 4 >> 4));     // 32 B per k-step: 8 tf32 or 16 fp16
                            if (F16) {
                                umma_f16_ts(tmem_base, a_hi + k * 8, db + bo, idesc_wide, (kb | k) != 0);
                                umma_f16_ts(tmem_base + 128, a_hi + 32 + k * 8, db + bo, idesc_cross, 1);
                                continue;
                            }
                            umma_tf32_ts(tmem_base, a_hi + k * UMMA_K, db + bo, idesc_wide, (kb | k) != 0);
                            umma_tf32_ts(tmem_base + 128, a_hi + 32 + k * UMMA_K, db + bo, idesc_cross, 1);
                        }
                        umma_commit(&empty[s]);
                        if (kb == num_kb - 1) umma_commit(acc_full);
                    }
                    __syncwarp();
                }
            } else if (warp < 6) {
                // ===================================================== operand warps: A smem -> (hi, lo) -> TMEM
                const int row = (warp & 3) * 32 + lane;
                const uint32_t lane_addr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + RF_ACOL0;
                const int sw = row & 7;
                for (int kb = 0; kb < num_kb; ++kb) {
                    const uint32_t i = it + kb;
                    const int s = i % RF_STAGES;
                    rf_wait(&full[s], (i / RF_STAGES) & 1);
                    tc_fence_after();
                    const uint4* arow = reinterpret_cast<const uint4*>(smem + s * RF_STAGE_BYTES + 2 * RF_TILE_BYTES + row * 128);
                    uint32_t hi[32], lo[32];
                    if constexpr (F16) {
                        // 64 k of this thread's row (two 32-k boxes) -> scaled fp16 (hi, lo) pairs, two k per TMEM column
                        const float a_scale = pow2f_int(layer == 0 ? shift_x : shift_h);
#pragma unroll
                        for (int bx = 0; bx < 2; ++bx) {
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const uint4 q = arow[bx * (RF_TILE_BYTES / 16) + (j ^ sw)];
                                f16_split2(__uint_as_float(q.x) * a_scale, __uint_as_float(q.y) * a_scale, hi[bx * 16 + 2 * j],
                                           lo[bx * 16 + 2 * j]);
                                f16_split2(__uint_as_float(q.z) * a_scale, __uint_as_float(q.w) * a_scale, hi[bx * 16 + 2 * j + 1],
                                           lo[bx * 16 + 2 * j + 1]);
                            }
                        }
                    } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const uint4 q = arow[j ^ sw];
                        hi[4 * j] = q.x; hi[4 * j + 1] = q.y; hi[4 * j + 2] = q.z; hi[4 * j + 3] = q.w;   // raw word = hi operand
                        lo[4 * j] = tf32_lo_bits(q.x); lo[4 * j + 1] = tf32_lo_bits(q.y);
                        lo[4 * j + 2] = tf32_lo_bits(q.z); lo[4 * j + 3] = tf32_lo_bits(q.w);
                    }
                    }
                    tmem_st_32x32b_x32(lane_addr + (uint32_t)s * 64u, hi);
                    tmem_st_32x32b_x32(lane_addr + (uint32_t)s * 64u + 32u, lo);
                    tmem_st_wait();
                    tc_fence_before();
                    mbar_arrive(&conv[s]);
                }
            } else {
                // ===================================================== epilogue: accumulator -> act(. + bias) -> h1 tile | head partials
                const int quad = warp & 3;
                const int half = (warp - 6) >> 2;                  // columns [64*half, 64*half + 64) of the 128-column tile
                const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(half * 64);
                const float out_scale = F16 ? pow2f_int(-((layer == 0 ? shift_x : shift_h) + kF16WShift)) : 1.f;
                rf_wait(acc_full, tile_iter & 1);
                RF_TRACE(1 + 4 * layer);          // accumulator complete
                tc_fence_after();
                float o[64];
#pragma unroll
                for (int c0 = 0; c0 < 64; c0 += 16) {
                    uint32_t r[16], r2[16];
                    tmem_ld_32x32b_x16(taddr + (uint32_t)c0, r);
                    tmem_ld_32x32b_x16(taddr + 128u + (uint32_t)c0, r2);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        if (F16) o[c0 + j] = fmaf(__uint_as_float(r2[j]), 1.f / 2048.f, __uint_as_float(r[j])) * out_scale;
                        else o[c0 + j] = __uint_as_float(r[j]) + __uint_as_float(r2[j]);
                    }
                }
                tc_fence_before();
                mbar_arrive(acc_empty);
                RF_TRACE(2 + 4 * layer);          // drained
                const float* bias = (layer == 0 ? b1_s : b2_s) + half * 64;
#pragma unroll
                for (int j = 0; j < 64; ++j) o[j] = act_fwd_ct<ACT>(o[j] + bias[j]);
                RF_TRACE(11 + layer);             // bias + activation done
                const int64_t m = m0 + quad * 32 + lane;
                if (m < a.N) {
                    if (layer == 0) {
                        float4* dst = reinterpret_cast<float4*>(a.h1 + m * a.H1 + n0 + half * 64);
#pragma unroll
                        for (int j = 0; j < 16; ++j) dst[j] = make_float4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
                    } else {
                        float hp[RF_HEAD_AP];
#pragma unroll
                        for (int r = 0; r < RF_HEAD_AP; ++r) {
                            const float* w = headw_s + r * 128 + half * 64;   // warp-uniform: shared-memory broadcast
                            float s0 = 0.f, s1 = 0.f;
#pragma unroll
                            for (int j = 0; j < 64; j += 4) {
                                const float4 wv4 = *reinterpret_cast<const float4*>(w + j);
                                s0 = fmaf(o[j], wv4.x, s0);
                                s1 = fmaf(o[j + 1], wv4.y, s1);
                                s0 = fmaf(o[j + 2], wv4.z, s0);
                                s1 = fmaf(o[j + 3], wv4.w, s1);
                            }
                            hp[r] = s0 + s1;
                        }
                        RF_TRACE(13);             // head partial dot products done
                        float4* dst = reinterpret_cast<float4*>(a.part + ((int64_t)(cx * 2 + half) * a.N + m) * kHeadPartPad);
                        dst[0] = make_float4(hp[0], hp[1], hp[2], hp[3]);
                        dst[1] = make_float4(hp[4], hp[5], hp[6], hp[7]);
                        dst[2] = make_float4(hp[8], 0.f, 0.f, 0.f);
                    }
                }
                if (layer == 0) fence_proxy_async_all();   // h1 stores -> the peers' TMA loads
                RF_TRACE(3 + 4 * layer);          // epilogue stores issued
            }
            it += (uint32_t)num_kb;
            ++tile_iter;
            cluster_sync_all();   // h1 of the row block complete (layer 0) / all head partials of the row block written (layer 1)
            RF_TRACE(4 + 4 * layer);              // past the cluster barrier
        }

        // ===================================================== step tail: this CTA's share of the block's rows.
        // FOUR rows per warp at a time: an 8-lane group owns a row (one lane per action logit, the group leader also the value
        // and the env's scalars), so the 32 rows of a CTA are ONE pass of eight warps -- the per-row dependency chain (partial
        // sums from L2 -> softmax -> Philox -> argmax -> env rule -> stores, ~4.7 us measured) is paid once per step, not once
        // per row a warp owns.  Bit-identical to heads_row_tail: logit a sits at group position (a + 1) % 8, which reproduces
        // the association order of the 32-lane butterfly sums there (lanes 1..8 after the xor-16 / xor-8 steps).
        if (warp >= 6) {
            const int g = lane & 7;                       // position inside the 8-lane group
            const int grp = lane >> 3;                    // which of the warp's four rows
            const int act_idx = (g + 7) & 7;              // action index held by this lane (position (a + 1) % 8)
            const bool has_logit = act_idx < a.A;
            const bool leader = g == 0;
            const bool last = (t + 1 == a.T);
            const int64_t step = env_step0 + t;
            const uint64_t offset = philox0 + (uint64_t)t;
            const float* src_step = a.tape + ((step + 1) % a.tape_len) * a.N * a.K1;
            const float* noise_t = a.noise ? a.noise + (int64_t)t * a.N * a.A : nullptr;
            const int rpc = 128 / CX;                     // rows of the block this CTA finishes
            const unsigned gmask = 0xffu << (grp * 8);
            for (int base = 0; base < rpc; base += 32) {
                const int rr = base + (warp - 6) * 4 + grp;
                const int64_t row = m0 + cx * rpc + rr;
                const bool ok = rr < rpc && row < a.N;
                // ---- loads first: head partials, next observation (K1 / 8 floats per lane), episode accumulators
                float x = 0.f, val = 0.f;
                float ob[RF_MAX_DIM / 8];
                float er0 = 0.f, mn0 = 0.f, mx0 = 0.f;
                int32_t el0 = 0;
                const int cpl = a.K1 >> 3;                // observation columns per lane (K1 is a multiple of 32)
                if (ok) {
                    if (has_logit)
                        for (int p = 0; p < P; ++p) x += a.part[((int64_t)p * a.N + row) * kHeadPartPad + 1 + act_idx];
                    if (leader)
                        for (int p = 0; p < P; ++p) val += a.part[((int64_t)p * a.N + row) * kHeadPartPad];
                    const float4* src4 = reinterpret_cast<const float4*>(src_step + row * a.K1 + g * cpl);
#pragma unroll
                    for (int q = 0; q < RF_MAX_DIM / 32; ++q)
                        if (4 * q < cpl) {
                            const float4 f4 = src4[q];
                            ob[4 * q] = f4.x; ob[4 * q + 1] = f4.y; ob[4 * q + 2] = f4.z; ob[4 * q + 3] = f4.w;
                        }
                    if (leader && a.ep_ret) { er0 = a.ep_ret[row]; el0 = a.ep_len[row]; mn0 = a.ep_min[row]; mx0 = a.ep_max[row]; }
                }
                // ---- CategoricalActionDistribution on the group (action_distributions.py:110-148), as heads_row_tail
                x += has_logit ? a.ba[act_idx] : 0.f;
                val += a.bv[0];
                const float xl = has_logit ? x : -INFINITY;
                float m = xl;
#pragma unroll
                for (int o = 4; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
                const float ex = has_logit ? expf(xl - m) : 0.f;
                float ssum = ex;
#pragma unroll
                for (int o = 4; o > 0; o >>= 1) ssum += __shfl_xor_sync(0xffffffffu, ssum, o);
                const float pr = __fdiv_rn(ex, ssum);                       // softmax :116
                const float logp = (xl - m) - logf(ssum);                   // log_softmax :125
                float q = 1.f;
                if (ok && has_logit) {
                    if (noise_t) q = noise_t[row * a.A + act_idx];
                    else {
                        curandStatePhilox4_32_10_t st;
                        curand_init(a.seed, (unsigned long long)(row * a.A + act_idx), offset, &st);
                        q = fmaxf(-logf(curand_uniform(&st)), 1.0e-30f);    // Exp(1)
                    }
                }
                float best = has_logit ? __fdiv_rn(pr, q) : -INFINITY;      // multinomial == argmax(p / q), first index on ties
                int idx = has_logit ? act_idx : 0x7fffffff;
#pragma unroll
                for (int o = 4; o > 0; o >>= 1) {
                    const float ob_ = __shfl_xor_sync(0xffffffffu, best, o);
                    const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
                    if (ob_ > best || (ob_ == best && oi < idx)) { best = ob_; idx = oi; }
                }
                const float lp = __shfl_sync(0xffffffffu, logp, (grp << 3) | ((idx + 1) & 7));   // log_prob :145-148
                (void)gmask;
                if (!ok) continue;
                // ---- trajectory slot t, env step, post step, pre step of t + 1
                if (has_logit) a.logits[row * a.logits_rs + (int64_t)t * a.A + act_idx] = x;
                const int64_t env = a.env_off + row;
                const float r_raw = (float)idx / (float)a.A;
                const bool tm = ((step * 7 + env * 13) % a.term_period) == 0;
                const bool tr = (((step + env) % a.trunc_period) == 0) && !tm;
                float* obs_next = a.traj_obs + row * a.traj_obs_rs + (int64_t)(t + 1) * a.K1 + g * cpl;
                float* env_o = a.env_obs + row * a.K1 + g * cpl;
                float* xn = a.x_norm + row * a.K1 + g * cpl;
#pragma unroll
                for (int q4 = 0; q4 < RF_MAX_DIM / 32; ++q4)
                    if (4 * q4 < cpl) {
                        const float4 f4 = make_float4(ob[4 * q4], ob[4 * q4 + 1], ob[4 * q4 + 2], ob[4 * q4 + 3]);
                        reinterpret_cast<float4*>(env_o)[q4] = f4;
                        reinterpret_cast<float4*>(obs_next)[q4] = f4;
                        if (!last) {
                            const int c = g * cpl + 4 * q4;
                            float4 y;
                            y.x = norm_one(f4.x, a.sub, a.inv_scale, a.do_sub, a.do_scale, do_rms, do_rms ? cstat[c] : 0.f, do_rms ? cstat[a.K1 + c] : 1.f, a.clip);
                            y.y = norm_one(f4.y, a.sub, a.inv_scale, a.do_sub, a.do_scale, do_rms, do_rms ? cstat[c + 1] : 0.f, do_rms ? cstat[a.K1 + c + 1] : 1.f, a.clip);
                            y.z = norm_one(f4.z, a.sub, a.inv_scale, a.do_sub, a.do_scale, do_rms, do_rms ? cstat[c + 2] : 0.f, do_rms ? cstat[a.K1 + c + 2] : 1.f, a.clip);
                            y.w = norm_one(f4.w, a.sub, a.inv_scale, a.do_sub, a.do_scale, do_rms, do_rms ? cstat[c + 3] : 0.f, do_rms ? cstat[a.K1 + c + 3] : 1.f, a.clip);
                            reinterpret_cast<float4*>(xn)[q4] = y;
                        }
                    }
                if (a.rnn)
                    for (int j = g; j < a.rnn_dim; j += 8)
                        a.traj_rnn[row * a.traj_rnn_rs + (int64_t)(t + 1) * a.rnn_dim + j] = a.rnn[row * a.rnn_dim + j];
                if (leader) {
                    a.values[row * a.values_rs + t] = val;
                    a.actions[row * a.actions_rs + t] = (float)idx;
                    a.env_actions[row] = idx;
                    a.log_prob[row * a.lp_rs + t] = lp;
                    a.pv_out[row * a.pv_rs + t] = pv;
                    a.env_rew[row] = r_raw;
                    a.env_term[row] = tm;
                    a.env_trunc[row] = tr;
                    const bool done = tm || tr;                                     // batched_sampling.py:317
                    float r = __fmul_rn(r_raw, a.reward_scale);                     // :209
                    r = clampf(r, -a.reward_clip, a.reward_clip);                   // :210
                    a.t_rew[row * a.stride + t] = r;
                    a.t_done[row * a.stride + t] = done ? 1 : 0;
                    a.t_to[row * a.stride + t] = tr ? 1 : 0;                        // :328
                    a.t_pid[row * a.stride + t] = a.policy_id;
                    if (a.ep_ret) {                                                 // _process_env_step :215-287 (raw reward)
                        float er = er0 + r_raw;
                        int32_t el = el0 + a.len_inc;
                        float mn = fminf(mn0, r_raw), mx = fmaxf(mx0, r_raw);
                        if (a.fin_ret) {
                            a.fin_ret[row * a.stride + t] = done ? er : __int_as_float(0x7fc00000);
                            a.fin_len[row * a.stride + t] = done ? el : -1;
                        }
                        if (done) {
                            if (a.stats) {
                                atomicAdd(&s_stats[0], 1.0); atomicAdd(&s_stats[1], (double)er); atomicAdd(&s_stats[2], (double)el);
                                atomicAdd(&s_stats[3], (double)mn); atomicAdd(&s_stats[4], (double)mx);
                            }
                            er = 0.f; el = 0; mn = INFINITY; mx = -INFINITY;
                        }
                        a.ep_ret[row] = er; a.ep_len[row] = el; a.ep_min[row] = mn; a.ep_max[row] = mx;
                    }
                }
            }
            fence_proxy_async_all();   // x_norm stores -> the peers' TMA loads of the next step
            RF_TRACE(9);                          // tail done
        }
        cluster_sync_all();   // the row block's next policy input is complete; nobody still reads this step's partials
        RF_TRACE(10);
    }
#undef RF_TRACE

    // every block has read the two step counters at its start; the last one to finish advances them by T
    __syncthreads();
    if (threadIdx.x < 5 && a.stats && s_stats[0] > 0.0) atomicAdd(a.stats + threadIdx.x, s_stats[threadIdx.x]);
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(a.ticket, 1u) == gridDim.x * gridDim.y - 1u) {
            *a.ticket = 0u;
            a.env_step[0] = env_step0 + a.T;
            if (a.sampler_step) *a.sampler_step = (int64_t)philox0 + a.T;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

template <int ACT, bool F16>
static int launch_rollout(const CUtensorMap* tm, const RolloutArgs& a, int CX, cudaStream_t st) {
    auto kern = rollout_mlp2_tape_kernel<ACT, F16>;
    static bool attr_set = false;
    if (!attr_set) {
        SFB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, RfSmem::TOTAL));
        attr_set = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)CX, (unsigned)ceil_div(a.N, 128));
    cfg.blockDim = dim3(RF_THREADS);
    cfg.dynamicSmemBytes = RfSmem::TOTAL;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)CX;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 2 : 1;
    SFB_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, tm[0], tm[1], tm[2], tm[3], tm[4], tm[5], a));
    SFB_LAUNCH_OK();
    return 0;
}

int tc_rollout_mlp2_supported(const float* W1, const float* W2, int K1, int H1, int H2, int A, int engine) {
    if (engine != SFB200_GEMM_TC_3XTF32 || !tc_init()) return 0;
    if (!(K1 == 32 || K1 == 64 || K1 == 96 || K1 == 128) || H1 != H2 || !(H2 == 128 || H2 == 256 || H2 == 512)) return 0;
    if (A < 1 || A + 1 > RF_HEAD_AP) return 0;
    if (!tf32_lo_lookup(W1, (int64_t)H1 * K1) || !tf32_lo_lookup(W2, (int64_t)H2 * H1)) return 0;
    return 2 * (H2 / 128);
}

// fp16-split form (common.cuh): taken when the weights have registered fp16 twins and both activation buffers (x_norm, the
// h1 scratch) have registered bounds
int tc_rollout_mlp2_tape(const float* W1, const float* W2, int act, int engine, const RolloutArgs& a_in, cudaStream_t st) {
    if (!tc_rollout_mlp2_supported(W1, W2, a_in.K1, a_in.H1, a_in.H2, a_in.A, engine)) return SFB_TC_UNSUPPORTED;
    RolloutArgs a = a_in;
    if (a.K1 % 64 == 0 && a.H1 % 64 == 0) {
        const F16Twin t1 = f16_twin_lookup(W1, (int64_t)a.H1 * a.K1), t2 = f16_twin_lookup(W2, (int64_t)a.H2 * a.H1);
        const float* bx = operand_bound_lookup(a.x_norm, a.N * a.K1 * (int64_t)sizeof(float));
        const float* bh = operand_bound_lookup(a.h1, a.N * a.H1 * (int64_t)sizeof(float));
        if (t1.hi && t2.hi && bx && bh) {
            if (f16_check_enabled()) {
                int rc = f16_twins_check(W1, t1, a.H1, a.K1, false, st);
                if (!rc) rc = f16_twins_check(W2, t2, a.H2, a.H1, false, st);
                if (rc) return rc;
            }
            a.bound_x = bx;
            a.bound_h1 = bh;
            CUtensorMap tm[6];
            bool ok = make_tmap(&tm[0], a.x_norm, (uint64_t)a.K1, (uint64_t)a.N, (uint64_t)a.K1, 32, 128, false);
            ok = ok && make_tmap_f16(&tm[1], t1.hi, (uint64_t)a.K1, (uint64_t)a.H1, (uint64_t)a.K1, 64, 128);
            ok = ok && make_tmap_f16(&tm[2], t1.lo, (uint64_t)a.K1, (uint64_t)a.H1, (uint64_t)a.K1, 64, 128);
            ok = ok && make_tmap(&tm[3], a.h1, (uint64_t)a.H1, (uint64_t)a.N, (uint64_t)a.H1, 32, 128, false);
            ok = ok && make_tmap_f16(&tm[4], t2.hi, (uint64_t)a.H1, (uint64_t)a.H2, (uint64_t)a.H1, 64, 128);
            ok = ok && make_tmap_f16(&tm[5], t2.lo, (uint64_t)a.H1, (uint64_t)a.H2, (uint64_t)a.H1, 64, 128);
            if (!ok) return SFB_TC_UNSUPPORTED;
            const int CX = a.H2 / 128;
            switch (act) {
                case SFB200_ACT_ELU: return launch_rollout<SFB200_ACT_ELU, true>(tm, a, CX, st);
                case SFB200_ACT_RELU: return launch_rollout<SFB200_ACT_RELU, true>(tm, a, CX, st);
                case SFB200_ACT_TANH: return launch_rollout<SFB200_ACT_TANH, true>(tm, a, CX, st);
                default: return launch_rollout<SFB200_ACT_NONE, true>(tm, a, CX, st);
            }
        }
    }
    const float* W1lo = tf32_lo_lookup(W1, (int64_t)a.H1 * a.K1);
    const float* W2lo = tf32_lo_lookup(W2, (int64_t)a.H2 * a.H1);
    if (tf32_lo_check_enabled()) {
        int rc = tf32_lo_check(W1, W1lo, (int64_t)a.H1 * a.K1, st);
        if (!rc) rc = tf32_lo_check(W2, W2lo, (int64_t)a.H2 * a.H1, st);
        if (rc) return rc;
    }
    CUtensorMap tm[6];
    bool ok = make_tmap(&tm[0], a.x_norm, (uint64_t)a.K1, (uint64_t)a.N, (uint64_t)a.K1, 32, 128, false);
    ok = ok && make_tmap(&tm[1], W1, (uint64_t)a.K1, (uint64_t)a.H1, (uint64_t)a.K1, 32, 128, false);
    ok = ok && make_tmap(&tm[2], W1lo, (uint64_t)a.K1, (uint64_t)a.H1, (uint64_t)a.K1, 32, 128, false);
    ok = ok && make_tmap(&tm[3], a.h1, (uint64_t)a.H1, (uint64_t)a.N, (uint64_t)a.H1, 32, 128, false);
    ok = ok && make_tmap(&tm[4], W2, (uint64_t)a.H1, (uint64_t)a.H2, (uint64_t)a.H1, 32, 128, false);
    ok = ok && make_tmap(&tm[5], W2lo, (uint64_t)a.H1, (uint64_t)a.H2, (uint64_t)a.H1, 32, 128, false);
    if (!ok) return SFB_TC_UNSUPPORTED;
    const int CX = a.H2 / 128;
    switch (act) {
        case SFB200_ACT_ELU: return launch_rollout<SFB200_ACT_ELU, false>(tm, a, CX, st);
        case SFB200_ACT_RELU: return launch_rollout<SFB200_ACT_RELU, false>(tm, a, CX, st);
        case SFB200_ACT_TANH: return launch_rollout<SFB200_ACT_TANH, false>(tm, a, CX, st);
        default: return launch_rollout<SFB200_ACT_NONE, false>(tm, a, CX, st);
    }
}

}  // namespace sfb

using namespace sfb;

extern "C" {

static unsigned long long* g_rollout_trace = nullptr;
/* debug: device buffer of T x 12 uint64 that the next rollouts fill with phase time stamps (NULL switches it off) */
int sfb200_rollout_set_trace(void* trace_dev) {
    g_rollout_trace = (unsigned long long*)trace_dev;
    return 0;
}

int sfb200_rollout_mlp2_partials(const float* W1, const float* W2, int K1, int H1, int H2, int A, int engine) {
    return tc_rollout_mlp2_supported(W1, W2, K1, H1, H2, A, engine);
}

int sfb200_rollout_mlp2_tape(int64_t n_envs, int T, int K1, const float* W1, const float* b1, int H1, const float* W2,
                             const float* b2, int H2, int act, int engine, const float* Wv, const float* bv, const float* Wa,
                             const float* ba, int A, float* h1_scratch, float* head_partials, float* x_norm,
                             float* values_0, int64_t values_stride, float* logits_0, int64_t logits_stride,
                             const float* noise, uint64_t philox_seed, int64_t* sampler_step, float* actions_0,
                             int64_t actions_stride, int32_t* env_actions, float* log_prob_0, int64_t log_prob_stride,
                             const float* policy_version_scalar, float* policy_version_0, int64_t pv_stride,
                             const float* tape, int64_t tape_len, int64_t env_index_offset, int term_period, int trunc_period,
                             int64_t* env_step_counter, float* env_obs, float* env_rew, uint8_t* env_terminated,
                             uint8_t* env_truncated, float reward_scale, float reward_clip, int32_t policy_id,
                             float* traj_rewards_0, uint8_t* traj_dones_0, uint8_t* traj_time_outs_0, int32_t* traj_policy_id_0,
                             int64_t traj_stride, float* ep_return, int32_t* ep_len, float* ep_min_raw, float* ep_max_raw,
                             int32_t len_increment, double* stats, float* fin_return_0, int32_t* fin_len_0, float* traj_obs_0,
                             int64_t traj_obs_stride, const float* rnn, int rnn_dim, float* traj_rnn_0, int64_t traj_rnn_stride,
                             const double* mean, const double* var, float sub_mean, float inv_scale, float eps, float clip,
                             void* stream) {
    SFB_CHECK_ARG(n_envs > 0 && T > 0 && W1 && b1 && W2 && b2 && Wv && bv && Wa && ba && h1_scratch && head_partials && x_norm,
                  "rollout_mlp2_tape: bad model arguments");
    SFB_CHECK_ARG(values_0 && logits_0 && actions_0 && env_actions && log_prob_0 && policy_version_0 && policy_version_scalar,
                  "rollout_mlp2_tape: bad heads arguments");
    SFB_CHECK_ARG(tape && tape_len > 0 && term_period > 0 && trunc_period > 0 && env_step_counter && env_obs && env_rew &&
                      env_terminated && env_truncated, "rollout_mlp2_tape: bad env arguments");
    SFB_CHECK_ARG(traj_rewards_0 && traj_dones_0 && traj_time_outs_0 && traj_policy_id_0 && traj_obs_0,
                  "rollout_mlp2_tape: bad trajectory arguments");
    SFB_CHECK_ARG((mean == nullptr) == (var == nullptr), "rollout_mlp2_tape: mean/var must both be set or both NULL");
    SFB_CHECK_ARG(K1 <= RF_MAX_DIM, "rollout_mlp2_tape: observation rows of up to %d floats", RF_MAX_DIM);
    SFB_CHECK_ARG((reinterpret_cast<uintptr_t>(h1_scratch) & 15u) == 0 && (reinterpret_cast<uintptr_t>(x_norm) & 15u) == 0 &&
                      (reinterpret_cast<uintptr_t>(head_partials) & 15u) == 0, "rollout_mlp2_tape: scratch buffers must be 16-byte aligned");
    const bool with_rnn = rnn && traj_rnn_0 && rnn_dim > 0;
    // the block ticket lives in the second word pair of the env's step counter (int64 [2]: step, ticket)
    unsigned int* ticket = reinterpret_cast<unsigned int*>(env_step_counter + 1);
    const RolloutArgs a{n_envs, T, K1, H1, H2, b1, b2, Wv, Wa, A, bv, ba, h1_scratch, head_partials, x_norm,
                        values_0, values_stride, logits_0, logits_stride, actions_0, actions_stride, env_actions, log_prob_0,
                        log_prob_stride, policy_version_0, pv_stride, policy_version_scalar, noise, philox_seed, sampler_step,
                        tape, tape_len, env_index_offset, term_period, trunc_period, env_step_counter, env_obs, env_rew,
                        env_terminated, env_truncated, reward_scale, reward_clip, policy_id, traj_rewards_0, traj_dones_0,
                        traj_time_outs_0, traj_policy_id_0, traj_stride, ep_return, ep_len, ep_min_raw, ep_max_raw, len_increment,
                        stats, fin_return_0, fin_len_0, traj_obs_0, traj_obs_stride, with_rnn ? rnn : nullptr, rnn_dim, traj_rnn_0,
                        traj_rnn_stride, mean, var, sub_mean, inv_scale, fabsf(sub_mean) > 1e-8f ? 1 : 0,
                        fabsf(inv_scale - 1.0f) > 1e-8f ? 1 : 0, eps, clip, ticket, g_rollout_trace, nullptr, nullptr};
    const int rc = tc_rollout_mlp2_tape(W1, W2, act, engine, a, (cudaStream_t)stream);
    SFB_CHECK_ARG(rc != SFB_TC_UNSUPPORTED, "rollout_mlp2_tape: model not covered (K1=%d H1=%d H2=%d A=%d engine=%d); "
                  "sfb200_rollout_mlp2_partials() tells when to use the per-step calls", K1, H1, H2, A, engine);
    return rc;
}

}  // extern "C"
