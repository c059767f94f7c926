// K5 -- whole-rollout cost normalisation (SURVEY §8 (f1)): replaces the per-step host arithmetic of
// VecNormalizeWithCost.step_wait / _update_cost / normalize_cost (stable_baselines3/common/vec_env/vec_normalize.py:
// 232-257) and RunningMeanStd.update (common/running_mean_std.py:19-39) for a [T, E] rollout that K1 has just
// relabelled, so that collection no longer needs T tiny cost_function calls.
//
// The reference's statistics are float64 numpy; the result is required to be BIT-EXACT (the normalised costs feed
// K3 and K4), so every operation is an explicit round-to-nearest double intrinsic (no FMA contraction) in numpy's
// evaluation order, and the batch mean / variance over the E environments use numpy's pairwise summation.
//
//   E <= 64 (every named workload): ONE launch of one CTA, cost_norm_fused_kernel, walking the rollout in tiles of TT steps
//   staged in shared memory.  Only loop-carried arithmetic stays serial; per tile:
//     load (coalesced; costs widened to double once)  ->  return chain per env (E threads) || count chain (1 thread)
//     ->  batch moments, tot = count + n, RN(1 / tot)   (parallel over t)
//     ->  Chan merge as a three-stage pipeline on three warps, progress published through shared memory:
//           mean chain (8 dependent FP64 ops / step) -> cross term (4 independent divisions per block) -> variance chain
//     ->  normalise + store (parallel)
//   Measured on B200 (tools/micro/fp64_bench.cu): DFMA/DADD/DMUL issue at 64 lanes/cycle/SM with 8.5-cycle latency, but
//   float<->double conversions (F2F) run at ~16 lanes/cycle/SM with ~22-cycle latency, hence no conversion on a chain.
//   E > 64, or no training: three launches (without training: A, then C when norm_cost) --
//   A  cost_ret_kernel    one thread per environment: ret <- ret * gamma + c[t], store, zero at episode ends   (T-serial)
//   B  cost_rms_kernel    one CTA: per-step batch mean/var (parallel over t), then the Chan merge chain on thread 0
//   C  cost_apply_kernel  c / sqrt(var_t + eps), clip, -> float32                                              (parallel)
#include <stdlib.h>

#include "common.cuh"

namespace icrl {

// numpy's pairwise summation (numpy/core/src/umath/loops_utils.h.src, @TYPE@_pairwise_sum) over f(a[i]).
// The recursion for n > 128 is bounded at compile time (DEPTH levels, each a real call) so that the stack is sized
// statically; pw_max_n(DEPTH) below is how many elements DEPTH levels cover.
template <int DEPTH, class F>
__device__ __noinline__ double np_pairwise_sum(const double* a, int n, F f) {
    if (n < 8) {
        double res = 0.0;
        for (int i = 0; i < n; ++i) res = __dadd_rn(res, f(a[i]));
        return res;
    }
    if (n <= 128) {
        double r[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = f(a[j]);
        int i = 8;
        for (; i < n - (n % 8); i += 8) {
#pragma unroll
            for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], f(a[i + j]));
        }
        double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                               __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
        for (; i < n; ++i) res = __dadd_rn(res, f(a[i]));
        return res;
    }
    if constexpr (DEPTH > 0) {
        int n2 = n / 2;
        n2 -= n2 % 8;
        return __dadd_rn(np_pairwise_sum<DEPTH - 1>(a, n2, f), np_pairwise_sum<DEPTH - 1>(a + n2, n - n2, f));
    } else {
        return __longlong_as_double(0x7ff8000000000000LL);   // unreachable for n <= pw_max_n(DEPTH): see kMaxEnvs
    }
}
// The largest m such that every n <= m reaches blocks of at most 128 within `depth` splits.  numpy's split of
// n = 16k + r (0 <= r < 16) is n2 = 8k, so the larger half is 8k + r and the halves are uneven: the first n whose larger
// half exceeds p = pw_max_n(depth - 1) is p + 1 + 8 * ceil((p - 14) / 8), well below 128 * 2^depth (491 529 needs 13
// levels, not 12).  Not monotone above that bound (256 needs one level, 249 two), hence "every n <= m".
constexpr int pw_max_n(int depth) {
    int m = 128;
    for (int d = 0; d < depth; ++d) m += 8 * ((m - 14 + 7) / 8);
    return m;
}
constexpr int kPwDepth = 13;
constexpr int kMaxEnvs = 128 << 12;   // 524 288 environments per rollout
static_assert(kMaxEnvs <= pw_max_n(kPwDepth), "np_pairwise_sum<kPwDepth> must cover every accepted E");

// RunningMeanStd.update_from_moments, one step (shared by the fused and the three-launch paths).
__device__ __forceinline__ void rms_step(double bm, double bv, double n, double& mean, double& var, double& count) {
    const double delta = __dsub_rn(bm, mean);
    const double tot = __dadd_rn(count, n);
    const double new_mean = __dadd_rn(mean, __ddiv_rn(__dmul_rn(delta, n), tot));
    const double m_a = __dmul_rn(var, count);
    const double m_b = __dmul_rn(bv, n);
    const double cross = __ddiv_rn(__dmul_rn(__dmul_rn(__dmul_rn(delta, delta), count), n), tot);
    const double m_2 = __dadd_rn(__dadd_rn(m_a, m_b), cross);
    mean = new_mean;
    var = __ddiv_rn(m_2, tot);
    count = __dadd_rn(n, count);
}

// Division by a divisor whose correctly rounded reciprocal r = RN(1/b) is already known (computed off the serial chain):
// one Newton refinement makes q1 a faithful quotient, and Markstein's correction step q = RN(q1 + (a - b q1) r) then
// yields the correctly rounded a / b (P. Markstein, IBM J. R&D 34(1), 1990, Thm 4.1; needs only that b's significand is
// not all ones -- the caller checks that and otherwise keeps __ddiv_rn).  5 dependent FMAs instead of the ~4x longer
// generic division sequence, with bit-identical results.
__device__ __forceinline__ double div_known_rcp(double a, double b, double r) {
    const double q0 = __dmul_rn(a, r);
    const double q1 = __fma_rn(__fma_rn(-b, q0, a), r, q0);
    return __fma_rn(__fma_rn(-b, q1, a), r, q1);
}
__device__ __forceinline__ bool significand_all_ones(double b) {
    return (__double_as_longlong(b) & 0x000fffffffffffffLL) == 0x000fffffffffffffLL;
}
// A: discounted cost return per environment.  state = {mean, var, count, cost_ret[E]} (float64).  Without training the
// return is not accumulated but is still zeroed at episode ends, as VecNormalizeWithCost.step_wait does (ret_t unused).
__global__ void cost_ret_kernel(const float* __restrict__ orig_costs, const float* __restrict__ dones,
                                const uint8_t* __restrict__ last_dones, int T, int E, double gamma, int training,
                                double* __restrict__ state, double* __restrict__ ret_t) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    double ret = state[3 + e];
    for (int t = 0; t < T; ++t) {
        if (training) {
            ret = __dadd_rn(__dmul_rn(ret, gamma), (double)orig_costs[(size_t)t * E + e]);
            ret_t[(size_t)t * E + e] = ret;
        }
        // `news` of step t is what the buffer stores as dones[t + 1] (on_policy_algorithm.py:406-415)
        const bool ended = (t + 1 < T) ? (dones[(size_t)(t + 1) * E + e] != 0.f) : (last_dones[e] != 0);
        if (ended) ret = 0.0;
    }
    state[3 + e] = ret;
}

// B: batch moments per step, then RunningMeanStd.update_from_moments T times.
__global__ void __launch_bounds__(1024) cost_rms_kernel(const double* __restrict__ ret_t, int T, int E,
                                                        double* __restrict__ state, double* __restrict__ bmean,
                                                        double* __restrict__ bvar, double* __restrict__ var_t) {
    const double n = (double)E;
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
        const double* row = ret_t + (size_t)t * E;
        const double m = __ddiv_rn(np_pairwise_sum<kPwDepth>(row, E, [](double x) { return x; }), n);
        const double v = __ddiv_rn(np_pairwise_sum<kPwDepth>(row, E, [m](double x) {
                                       const double d = __dsub_rn(x, m);
                                       return __dmul_rn(d, d);
                                   }), n);
        bmean[t] = m;
        bvar[t] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double mean = state[0], var = state[1], count = state[2];
        for (int t = 0; t < T; ++t) {
            rms_step(bmean[t], bvar[t], n, mean, var, count);
            var_t[t] = var;
        }
        state[0] = mean; state[1] = var; state[2] = count;
    }
}

// C: normalize_cost on every element with the statistics as they stood right after that step's update.
__global__ void cost_apply_kernel(const float* __restrict__ orig_costs, const double* __restrict__ var_t,
                                  const double* __restrict__ state, int training, long long total, int E, double epsilon,
                                  double clip, float* __restrict__ costs) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const double var = training ? var_t[i / E] : state[1];
        double c = __ddiv_rn((double)orig_costs[i], __dsqrt_rn(__dadd_rn(var, epsilon)));
        c = fmin(fmax(c, -clip), clip);
        costs[i] = (float)c;
    }
}

// Fused single-CTA path for small E.  Dynamic smem per tile of TT steps:
//   RET[TT*E] f64 (cost as double, then the discounted return) | BM (batch mean, then delta) MB CNT TOT RCP CROSS VT [TT] f64 |
//   C[TT*E] f32 | NEWS[TT*E] u8
// Only what is loop-carried stays on the serial chains: every conversion, the batch moments, tot = count + n, its
// reciprocal and the cross term of the Chan merge are computed in the parallel phases between them.
constexpr int K5_THREADS = 256;
constexpr int K5_STEP_BYTES = 7 * 8;     // per-step doubles above
__device__ __forceinline__ double k5_div(double a, double b, double r) {
    return r != 0.0 ? div_known_rcp(a, b, r) : __ddiv_rn(a, b);
}
__global__ void __launch_bounds__(K5_THREADS) cost_norm_fused_kernel(
        const float* __restrict__ orig_costs, const float* __restrict__ dones, const uint8_t* __restrict__ last_dones, int T,
        int E, int TT, double gamma, double epsilon, double clip, int norm_cost, int fastdiv, double* __restrict__ state,
        float* __restrict__ costs, double* __restrict__ var_out, long long* __restrict__ prof) {
    extern __shared__ __align__(16) unsigned char k5_smem[];
    double* RET = reinterpret_cast<double*>(k5_smem);
    double* BM = RET + (size_t)TT * E;
    double* MB = BM + TT;       // batch variance * n
    double* CNT = MB + TT;      // count before step t (its own rounding chain, independent of the data)
    double* TOT = CNT + TT;     // count_t + n
    double* RCP = TOT + TT;     // RN(1 / tot), or 0 where the Markstein shortcut does not apply
    double* CROSS = RCP + TT;   // delta^2 * count * n / tot
    double* VT = CROSS + TT;    // running variance after step t
    float* Cs = reinterpret_cast<float*>(VT + TT);
    unsigned char* NEWS = reinterpret_cast<unsigned char*>(Cs + (size_t)TT * E);
    __shared__ volatile int prog_slot;                               // steps of the tile whose delta has been published
    __shared__ volatile int prog2_slot;                              // steps whose cross term has been published
    volatile int* prog = &prog_slot;
    volatile int* prog2 = &prog2_slot;
    const int tid = threadIdx.x;
    const double n = (double)E;
    double ret = (tid < E) ? state[3 + tid] : 0.0;
    double mean = state[0];                                          // live in thread 0 only (mean chain)
    double var = state[1];                                           // live in thread 32 only (variance chain)
    double count = state[2];                                         // live in thread 64 (count chain)
    long long pc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, c0 = 0;
#define K5_MARK(i) if (prof && tid == 0) { const long long c1 = clock64(); pc[i] += c1 - c0; c0 = c1; }
    for (int t0 = 0; t0 < T; t0 += TT) {
        const int tt = min(TT, T - t0);
        if (prof && tid == 0) c0 = clock64();
        if (tid == 0) { *prog = 0; *prog2 = 0; }
        // ---- load: costs (kept as float for the final division, widened once for the return chain) and episode ends
        for (int i = tid; i < tt * E; i += K5_THREADS) {
            const int t = t0 + i / E, e = i % E;
            const float c = orig_costs[(size_t)t0 * E + i];
            Cs[i] = c;
            RET[i] = (double)c;
            NEWS[i] = (t + 1 < T) ? (dones[(size_t)(t + 1) * E + e] != 0.f) : (last_dones[e] != 0);
        }
        __syncthreads();
        K5_MARK(0)
        // ---- discounted return per environment (E chains) || sample count (one chain)
        if (tid < E) {
            int t = 0;
            for (; t + 4 <= tt; t += 4) {            // operands of four steps are fetched before the dependent chain runs
                double c[4];
                unsigned char nw[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) { c[u] = RET[(t + u) * E + tid]; nw[u] = NEWS[(t + u) * E + tid]; }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    ret = __dadd_rn(__dmul_rn(ret, gamma), c[u]);
                    RET[(t + u) * E + tid] = ret;
                    if (nw[u]) ret = 0.0;
                }
            }
            for (; t < tt; ++t) {
                ret = __dadd_rn(__dmul_rn(ret, gamma), RET[t * E + tid]);
                RET[t * E + tid] = ret;
                if (NEWS[t * E + tid]) ret = 0.0;
            }
        } else if (tid == 64) {
            for (int t = 0; t < tt; ++t) {
                CNT[t] = count;
                count = __dadd_rn(n, count);
            }
        }
        __syncthreads();
        K5_MARK(1)
        // ---- batch moments of every step (numpy's summation order), tot and its reciprocal
        for (int t = tid; t < tt; t += K5_THREADS) {
            const double* row = RET + (size_t)t * E;
            const double m = __ddiv_rn(np_pairwise_sum<0>(row, E, [](double x) { return x; }), n);
            BM[t] = m;
            const double bv = __ddiv_rn(np_pairwise_sum<0>(row, E, [m](double x) {
                                            const double d = __dsub_rn(x, m);
                                            return __dmul_rn(d, d);
                                        }), n);
            MB[t] = __dmul_rn(bv, n);
            const double tot = __dadd_rn(CNT[t], n);
            TOT[t] = tot;
            RCP[t] = (fastdiv && !significand_all_ones(tot)) ? __ddiv_rn(1.0, tot) : 0.0;
        }
        __syncthreads();
        K5_MARK(2)
        // ---- the Chan merge as a three-stage pipeline on three warps.  Thread 0: mean += (bm - mean) * n / tot, publishing
        // delta four steps at a time; thread 96 trails it with cross = delta^2 * count * n / tot (four independent divisions
        // per block); thread 32 trails that with var = ((var * count + m_b) + cross) / tot.  Steps whose tot has an all-ones significand (no
        // Markstein shortcut) take the generic division; the test is made once per block of four.
        long long tc0 = prof ? clock64() : 0;
        if (tid == 0) {
            int t = 0;
            for (; t + 4 <= tt; t += 4) {
                double bm[4], tot[4], r[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) { bm[u] = BM[t + u]; tot[u] = TOT[t + u]; r[u] = RCP[t + u]; }
                if (r[0] != 0.0 && r[1] != 0.0 && r[2] != 0.0 && r[3] != 0.0) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const double delta = __dsub_rn(bm[u], mean);
                        mean = __dadd_rn(mean, div_known_rcp(__dmul_rn(delta, n), tot[u], r[u]));
                        bm[u] = delta;
                    }
                } else {
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const double delta = __dsub_rn(bm[u], mean);
                        mean = __dadd_rn(mean, k5_div(__dmul_rn(delta, n), tot[u], r[u]));
                        bm[u] = delta;
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) BM[t + u] = bm[u];
                __threadfence_block();
                *prog = t + 4;
            }
            for (; t < tt; ++t) {
                const double delta = __dsub_rn(BM[t], mean);
                mean = __dadd_rn(mean, k5_div(__dmul_rn(delta, n), TOT[t], RCP[t]));
                BM[t] = delta;
                __threadfence_block();
                *prog = t + 1;
            }
        } else if (tid == 96) {
            // cross-term producer: trails the mean chain, four independent divisions per block
            int t = 0;
            for (; t + 4 <= tt; t += 4) {
                double cnt[4], tot[4], r[4], d[4], cr[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) { cnt[u] = CNT[t + u]; tot[u] = TOT[t + u]; r[u] = RCP[t + u]; }
                while (*prog < t + 4) {}
                __threadfence_block();
#pragma unroll
                for (int u = 0; u < 4; ++u) d[u] = BM[t + u];
                if (r[0] != 0.0 && r[1] != 0.0 && r[2] != 0.0 && r[3] != 0.0) {   // branch-free: the four divisions overlap
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        cr[u] = div_known_rcp(__dmul_rn(__dmul_rn(__dmul_rn(d[u], d[u]), cnt[u]), n), tot[u], r[u]);
                } else {
#pragma unroll
                    for (int u = 0; u < 4; ++u) cr[u] = k5_div(__dmul_rn(__dmul_rn(__dmul_rn(d[u], d[u]), cnt[u]), n), tot[u], r[u]);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) CROSS[t + u] = cr[u];
                __threadfence_block();
                *prog2 = t + 4;
            }
            for (; t < tt; ++t) {
                while (*prog < t + 1) {}
                __threadfence_block();
                const double dlt = BM[t];
                CROSS[t] = k5_div(__dmul_rn(__dmul_rn(__dmul_rn(dlt, dlt), CNT[t]), n), TOT[t], RCP[t]);
                __threadfence_block();
                *prog2 = t + 1;
            }
        } else if (tid == 32) {
            // variance chain: trails the cross-term producer
            int t = 0;
            for (; t + 4 <= tt; t += 4) {
                double cnt[4], mb[4], tot[4], r[4], cr[4], v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) { cnt[u] = CNT[t + u]; mb[u] = MB[t + u]; tot[u] = TOT[t + u]; r[u] = RCP[t + u]; }
                while (*prog2 < t + 4) {}
                __threadfence_block();
#pragma unroll
                for (int u = 0; u < 4; ++u) cr[u] = CROSS[t + u];
                if (r[0] != 0.0 && r[1] != 0.0 && r[2] != 0.0 && r[3] != 0.0) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        var = div_known_rcp(__dadd_rn(__dadd_rn(__dmul_rn(var, cnt[u]), mb[u]), cr[u]), tot[u], r[u]);
                        v[u] = var;
                    }
                } else {
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        var = k5_div(__dadd_rn(__dadd_rn(__dmul_rn(var, cnt[u]), mb[u]), cr[u]), tot[u], r[u]);
                        v[u] = var;
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) VT[t + u] = v[u];
            }
            for (; t < tt; ++t) {
                while (*prog2 < t + 1) {}
                __threadfence_block();
                var = k5_div(__dadd_rn(__dadd_rn(__dmul_rn(var, CNT[t]), MB[t]), CROSS[t]), TOT[t], RCP[t]);
                VT[t] = var;
            }
        }
        if (prof && (tid == 0 || tid == 96 || tid == 32)) atomicAdd((unsigned long long*)&prof[tid == 0 ? 4 : tid == 96 ? 5 : 7], (unsigned long long)(clock64() - tc0));
        __syncthreads();
        K5_MARK(3)
        // ---- the normalisation itself (a float64 division and square root per element) runs on the whole GPU afterwards
        // (cost_apply_kernel): in this single CTA it was 85 k of the kernel's 440 k cycles -- one SM's FP64 pipe -- and letting
        // half of the CTA trail the variance chain only slowed the chains down (they share that pipe: 239 -> 254 us).
        if (var_out != nullptr) {
            for (int i = tid; i < tt; i += K5_THREADS) var_out[t0 + i] = VT[i];
        } else {
            for (int i = tid; i < tt * E; i += K5_THREADS) {
                float c = Cs[i];
                if (norm_cost) {
                    const double x = __ddiv_rn((double)c, __dsqrt_rn(__dadd_rn(VT[i / E], epsilon)));
                    c = (float)fmin(fmax(x, -clip), clip);
                }
                costs[(size_t)t0 * E + i] = c;
            }
        }
        __syncthreads();
        K5_MARK(6)
    }
    if (prof && tid == 0)
        for (int i = 0; i < 8; ++i) if (i != 4 && i != 5 && i != 7) prof[i] = pc[i];
    if (tid < E) state[3 + tid] = ret;
    if (tid == 0) state[0] = mean;
    if (tid == 32) state[1] = var;
    if (tid == 64) state[2] = count;
}

}  // namespace icrl

extern "C" int icrl_cost_normalize(const float* orig_costs, const float* dones, const uint8_t* last_dones, int32_t T,
                                   int32_t E, double cost_gamma, double epsilon, double clip_cost, int32_t norm_cost,
                                   int32_t training, double* state, float* costs, void* stream) {
    using namespace icrl;
    ICRL_CHECK_ARG(orig_costs && dones && last_dones && state && costs, "icrl_cost_normalize: NULL pointer");
    ICRL_CHECK_ARG(T > 0 && E > 0, "icrl_cost_normalize: T and E must be positive (got %d, %d)", T, E);
    ICRL_CHECK_ARG(E <= kMaxEnvs, "icrl_cost_normalize: at most %d environments (got %d)", kMaxEnvs, E);
    cudaStream_t st = (cudaStream_t)stream;
    const long long total = (long long)T * E;
    double* scratch = nullptr;
    if (training && E <= 64) {
        // tile length: as many steps as fit ~96 KB of shared memory (13 B per element + 24 B per step), at most 1024
        int TT = (int)(96 * 1024 / (13 * (size_t)E + K5_STEP_BYTES));
        TT = TT > 1024 ? 1024 : TT;
        TT = TT > T ? T : TT;
        const size_t smem = (size_t)TT * E * 13 + (size_t)TT * K5_STEP_BYTES + 16;
        static const int fastdiv = getenv("ICRL_K5_GENERIC_DIV") ? 0 : 1;   // debugging aid: generic __ddiv_rn on the chain
        static bool attr_set = false;
        if (!attr_set) {
            ICRL_CUDA(cudaFuncSetAttribute(cost_norm_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
            attr_set = true;
        }
        long long* prof = nullptr;
        static const int timing = getenv("ICRL_K5_TIMING") ? 1 : 0;
        if (timing)
            if (int rc = device_scratch(SLOT_WORK3, 64, (void**)&prof)) return rc;
        if (prof) ICRL_CUDA(cudaMemsetAsync(prof, 0, 64, st));
        double* var_t = nullptr;                    // running variance after every step, for the grid-wide normalisation pass
        if (norm_cost)
            if (int rc = device_scratch(SLOT_K5, (size_t)T * sizeof(double), (void**)&var_t)) return rc;
        cost_norm_fused_kernel<<<1, K5_THREADS, smem, st>>>(orig_costs, dones, last_dones, T, E, TT, cost_gamma, epsilon,
                                                            clip_cost, norm_cost, fastdiv, state, costs, var_t, prof);
        ICRL_LAUNCH_CHECK();
        if (norm_cost) {
            const int blocks = (int)((total + 255) / 256 < (long long)sm_count() * 8 ? (total + 255) / 256 : (long long)sm_count() * 8);
            cost_apply_kernel<<<blocks, 256, 0, st>>>(orig_costs, var_t, state, 1, total, E, epsilon, clip_cost, costs);
            ICRL_LAUNCH_CHECK();
        }
        if (prof) {   // ICRL_K5_TIMING=1: per-phase cycles of thread 0 (load, return chain, moments, Chan chain, apply)
            long long h[8];
            ICRL_CUDA(cudaStreamSynchronize(st));
            ICRL_CUDA(cudaMemcpy(h, prof, sizeof(h), cudaMemcpyDeviceToHost));
            fprintf(stderr, "[k5] T=%d E=%d TT=%d cycles: load %lld ret %lld moments %lld chains %lld apply %lld | own loop time: mean %lld cross %lld var %lld\n",
                    T, E, TT, h[0], h[1], h[2], h[3], h[6], h[4], h[5], h[7]);
        }
        return 0;
    }
    if (training) {
        if (int rc = device_scratch(SLOT_WORK3, ((size_t)total + 3 * (size_t)T) * sizeof(double), (void**)&scratch)) return rc;
        double *ret_t = scratch, *bmean = scratch + total, *bvar = bmean + T, *var_t = bvar + T;
        cost_ret_kernel<<<(E + 63) / 64, 64, 0, st>>>(orig_costs, dones, last_dones, T, E, cost_gamma, 1, state, ret_t);
        ICRL_LAUNCH_CHECK();
        cost_rms_kernel<<<1, 1024, 0, st>>>(ret_t, T, E, state, bmean, bvar, var_t);
        ICRL_LAUNCH_CHECK();
        scratch = var_t;
    } else {
        cost_ret_kernel<<<(E + 63) / 64, 64, 0, st>>>(orig_costs, dones, last_dones, T, E, cost_gamma, 0, state, nullptr);
        ICRL_LAUNCH_CHECK();
    }
    if (norm_cost) {
        const int blocks = (int)((total + 255) / 256 < (long long)sm_count() * 8 ? (total + 255) / 256 : (long long)sm_count() * 8);
        cost_apply_kernel<<<blocks, 256, 0, st>>>(orig_costs, scratch, state, training, total, E, epsilon, clip_cost, costs);
        ICRL_LAUNCH_CHECK();
    } else if (costs != orig_costs) {
        ICRL_CUDA(cudaMemcpyAsync(costs, orig_costs, (size_t)total * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    return 0;
}
