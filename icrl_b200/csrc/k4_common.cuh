// Shared definitions of the K4 (PPO-Lagrangian) kernels.
#pragma once
#include <math.h>
#include <stdlib.h>

#include "common.cuh"

namespace icrl {

constexpr int H = 64;          // padded hidden width (both layers)
constexpr int RB = 64;         // rows per chunk
constexpr int NTH = 256;       // threads per CTA
constexpr int AMAX = 16;       // max action dims / discrete actions
constexpr int WA_LD = 68;      // leading dim of the action-head weight in smem
constexpr int LDH = 68;        // row stride of activation tiles and of W2 in smem: == 4 (mod 32) makes every mma.sync
                               // fragment read (row g, col t) hit 32 distinct banks
constexpr float LOG_SQRT_2PI = 0.91893853320467274178f;
constexpr float HALF_LOG_2PI_PLUS_HALF = 1.4189385332046727418f;

// K extent of the obs GEMMs (multiple of the mma K = 8) and the row stride of obs tiles / W1 / the obs stream
__host__ __device__ inline int ppo_kp(int D) { return (D + 7) / 8 * 8; }
__host__ __device__ inline int ppo_ldx(int D) {
    const int kp = (D + 15) / 16 * 16;   // the dW1 n-tiles come in pairs (one per warp group): rows are padded to 16 columns
    int ld = kp / 32 * 32 + 4;
    if (ld < kp) ld += 32;
    return ld;                 // >= round16(D), == 4 (mod 32), multiple of 4 floats (16-byte rows for the TMA bulk copies)
}

struct PpoArgs {
    int D, DP, KP, A, is_discrete;
    int h0[3], h1[3];             // hidden widths of the pi, vf and cvf trunks (every tile is padded to H = 64 regardless)
    int T, E, N, B, n_epochs, steps_per_epoch, max_steps;
    int has_target_kl, has_clip_vf_r, has_clip_vf_c;
    float clip_range, clip_vf_r, clip_vf_c, ent_coef, vf_coef_r, vf_coef_c, max_grad_norm, nu;
    double target_kl, lr, beta1, beta2, adam_eps;
    long long step_before;
    // flat parameter offsets (reference parameters() order)
    int off_logstd, off_w1[3], off_b1[3], off_w2[3], off_b2[3], off_hw[3], off_hb[3];
    const float *obs, *act, *old_logp, *old_vr, *adv_r, *ret_r, *old_vc, *adv_c, *ret_c;
    const int* perm;
    const float *xs, *as, *ss; // minibatch-ordered streams built by the prologue: obs [P][DP], actions [P][AP], scalars [P][8]
    int AP;                    // padded action width of the stream (multiple of 4)
    const float* advstats;     // [steps][8]: mean(adv_r), std(adv_r) (unbiased), mean(adv_c), 1/sqrt(1-b2^t), -lr/(1-b1^t)
    const float* nu_dev;
    float *params, *adam_m, *adam_v, *stats;
    int* result;
    unsigned long long* timing;   // optional [3 roles][16 phases] cycle accumulators (profiling aid)
    // data-parallel mode (world > 1): peer receive buffers / flags (CUDA IPC mapped), see include/icrl_b200.h
    int rank, world;
    float* recv[ICRL_PPO_MAX_RANKS];
    unsigned int* flags[ICRL_PPO_MAX_RANKS];
    unsigned int flag_base;
    int dist_mode;                // 0 auto (tagged broadcast + sum for 2 / 4 ranks, RS/AG for 8, {value, seq} words otherwise),
                                  // 1 {value, seq} words, 2 RS/AG, 3 broadcast + sum   (ICRL_PPO_DIST_MODE)
    const double* advsums;        // all-reduced per-step sums (sum adv_r, sum adv_r^2, sum adv_c, count) or NULL
    // large-batch ("wide") mode: `ncl` 6-CTA clusters share every minibatch (one launch per epoch), see k4_ppo_lag.cu
    int ncl, epoch_base, n_epochs_total;
    float* wide_part;             // [3 trunks][ncl][F][256 threads]: every cluster's pair-summed gradient fragments
    float* wide_red;              // [3 trunks][F][256 threads]: the cluster-order sums
    unsigned int* wide_sync;      // [3 trunks] arrival counters of the grid-wide barriers (zeroed before every launch)
};
constexpr int WIDE_SMAX = 6;      // floats a (cluster, half) reducer sums per step: F <= 2 * ncl * WIDE_SMAX
constexpr int WIDE_MAXCTA = 192;  // CTAs of a wide launch (<= 32 clusters) addressable in the data-parallel receive buffer
constexpr int WIDE_MIN_BATCH = 2048;   // batch_size from which the many-cluster kernel is used
constexpr int DIST_SLOTS = 72;    // floats per thread in a receive-buffer slab
constexpr int RSAG_MAXW = 20;     // 16-byte words per (rank, role, thread) slab of the reduce-scatter / all-gather exchange:
                                  // layout [region 3][parity 2][src 8][role 3][RSAG_MAXW][256 threads] uint4 = 11.8 MB (regions: reduce-scatter, all-gather,
                                  // 2-rank broadcast),
                                  // overlaid on the same receive buffer (sequence numbers keep the two layouts apart)

inline int ppo_fill_offsets(PpoArgs& a) {
    int o = 0;
    a.off_logstd = a.is_discrete ? -1 : 0;
    if (!a.is_discrete) o += a.A;
    for (int t = 0; t < 3; ++t) {
        const int h0 = a.h0[t], h1 = a.h1[t];
        a.off_w1[t] = o; o += h0 * a.D;
        a.off_b1[t] = o; o += h0;
        a.off_w2[t] = o; o += h1 * h0;
        a.off_b2[t] = o; o += h1;
    }
    const int outs[3] = {a.A, 1, 1};
    for (int t = 0; t < 3; ++t) {
        a.off_hw[t] = o; o += outs[t] * a.h1[t];
        a.off_hb[t] = o; o += outs[t];
    }
    return o;
}

inline int ppo_make_args(const icrl_ppo_cfg* c, PpoArgs& a) {
    ICRL_CHECK_ARG(c != nullptr, "ppo cfg is NULL");
    ICRL_CHECK_ARG(c->obs_dim >= 1, "obs_dim must be >= 1");
    ICRL_CHECK_ARG(c->act_dim >= 1 && c->act_dim <= AMAX, "act_dim %d out of range (1..%d)", c->act_dim, AMAX);
    bool per_trunk = false;
    for (int t = 0; t < 3; ++t) per_trunk |= c->trunk_hidden[t][0] != 0 || c->trunk_hidden[t][1] != 0;
    if (per_trunk) {
        static const char* const names[3] = {"pi", "vf", "cvf"};
        for (int t = 0; t < 3; ++t)
            ICRL_CHECK_ARG(c->trunk_hidden[t][0] >= 1 && c->trunk_hidden[t][0] <= H && c->trunk_hidden[t][1] >= 1 &&
                               c->trunk_hidden[t][1] <= H,
                           "trunk_hidden[%d] (%s) = (%d, %d): both widths must be in 1..%d (two hidden layers per trunk)", t,
                           names[t], c->trunk_hidden[t][0], c->trunk_hidden[t][1], H);
    } else {
        ICRL_CHECK_ARG(c->hidden[0] >= 1 && c->hidden[0] <= H && c->hidden[1] >= 1 && c->hidden[1] <= H,
                       "policy hidden sizes (%d, %d) must be in 1..%d (two hidden layers per trunk)", c->hidden[0],
                       c->hidden[1], H);
    }
    a.D = c->obs_dim; a.DP = ppo_ldx(c->obs_dim); a.KP = ppo_kp(c->obs_dim); a.A = c->act_dim; a.is_discrete = c->is_discrete;
    for (int t = 0; t < 3; ++t) {
        a.h0[t] = per_trunk ? c->trunk_hidden[t][0] : c->hidden[0];
        a.h1[t] = per_trunk ? c->trunk_hidden[t][1] : c->hidden[1];
    }
    a.T = c->T; a.E = c->E; a.N = c->T * c->E;
    a.B = c->batch_size > 0 ? c->batch_size : a.N;
    if (a.B > a.N && a.N > 0) a.B = a.N;
    a.n_epochs = c->n_epochs;
    a.steps_per_epoch = a.N > 0 ? (a.N + a.B - 1) / a.B : 0;
    a.max_steps = c->max_steps;
    a.has_target_kl = c->has_target_kl; a.has_clip_vf_r = c->has_clip_vf_reward; a.has_clip_vf_c = c->has_clip_vf_cost;
    a.clip_range = c->clip_range; a.clip_vf_r = c->clip_range_reward_vf; a.clip_vf_c = c->clip_range_cost_vf;
    a.ent_coef = c->ent_coef; a.vf_coef_r = c->reward_vf_coef; a.vf_coef_c = c->cost_vf_coef;
    a.max_grad_norm = c->max_grad_norm; a.nu = c->nu; a.target_kl = c->target_kl;
    a.lr = c->lr; a.beta1 = c->adam_beta1; a.beta2 = c->adam_beta2; a.adam_eps = c->adam_eps;
    ppo_fill_offsets(a);
    return 0;
}

}  // namespace icrl
