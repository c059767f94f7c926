// K4 -- the whole PPOLagrangian.train() epoch/minibatch loop as ONE persistent thread-block-cluster launch.
// Replaces stable_baselines3/ppo_lag/ppo_lag.py:198-297 (+ policies.py:752-767, distributions.py, clip_grad_norm_,
// Adam): per minibatch gather -> 3 tanh MLP forward -> losses -> backward -> global-norm clip -> Adam, for every
// minibatch of every epoch, with the per-epoch target_kl early stop decided on the device.
//
// Why this shape.  The reference runs 1 600 *dependent* optimiser steps per rollout on 64-128 rows each: the path is
// latency-bound, not HBM-bound (65 KB of algorithmic traffic per step).  So:
//   * one launch; no host round trip between steps (the host only supplies numpy's permutations up front);
//   * the minibatch schedule is data-independent, so two massively parallel prologue kernels take everything that does
//     not depend on the parameters out of the step chain: the random-access gather (minibatch-ordered streams in HBM),
//     the per-minibatch advantage statistics and the Adam bias corrections;
//   * the three trunks (pi / vf / cvf) are independent networks (torch_layers.py:129-254), so each gets its own CTA PAIR of
//     a 6-CTA cluster (each CTA takes 32 rows of every 64-row chunk) -- model parallel with NO activation exchange.  A pair
//     exchanges its gradient halves through distributed shared memory: st.async stores that complete transaction bytes on
//     the partner's mbarrier, no cluster barrier.  The only coupling between trunks is clip_grad_norm_'s global norm: one
//     8-byte st.async per CTA per step to every CTA's norm mbarrier;
//   * the head pieces are MMA tiles too: the action head is fused into the layer-2 epilogue (a C fragment is an A fragment
//     under a permutation of K), dHW and dH2 are 3xTF32 tiles;
//   * each chunk arrives by TMA bulk copies (cp.async.bulk + mbarrier) issued one chunk ahead by a single thread;
//   * weights live in shared memory for the whole launch; Adam moments and the gradient live in REGISTERS: every thread
//     owns fixed fragments of W1/W2 plus a few scalars for all 1 600 steps, so gradients are never materialised;
//   * the five GEMMs per chunk (X W1^T, H1 W2^T, dH2 W2, dH2^T H1, dH1^T X) run on the tensor cores as mma.sync
//     m16n8k8 TF32 with the 3xTF32 split (x = hi + lo; lo*hi + hi*lo + hi*hi), which keeps fp32-class accuracy
//     (~2^-21) as the parity tolerances require.  Measured on B200: FFMA register tiles take 4.1k cycles per 64^3 GEMM
//     (one 3-register FFMA per 2 cycles per SMSP), mma.sync TF32 sustains 512 FMA/cycle/SM -- see DESIGN.md.
//     tcgen05 is not used here on purpose: M=64 tiles on a dependent chain of five tiny GEMMs would pay a TMEM
//     allocate / commit / mbarrier / tcgen05.ld round trip per layer, and the epilogues (tanh, derivative masks, Adam)
//     want the accumulators in registers.
#include <type_traits>

#include "k4_common.cuh"

namespace icrl {

// ---------------------------------------------------------------- cluster primitives (raw PTX)
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// mbar_wait_bounded with cluster-scope acquire: the phase is completed by remote arrivals of peer CTAs
__device__ __forceinline__ bool mbar_wait_bounded_cluster(uint64_t* bar, uint32_t parity, long long max_cycles) {
    const long long t0 = clock64();
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (done) return true;
        if (clock64() - t0 > max_cycles) return false;
    }
}
__device__ __forceinline__ void st_remote_f32(float* local_ptr, uint32_t rank, float v) {
    uint32_t a = smem_u32(local_ptr), ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(a), "r"(rank));
    asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(ra), "f"(v) : "memory");
}

// ---------------------------------------------------------------- geometry of the train kernel
constexpr int NHALF = 2;       // CTAs per trunk: each takes RBH rows of every 64-row chunk (a CTA pair)
constexpr int RBH = RB / NHALF;
constexpr int NCTA = 3 * NHALF; // cluster size
constexpr int NTT = 256;       // threads of the train kernel: 8 warps (16 warps measured slower: 31.4k vs 27.5k cycles/step on HC)
constexpr int NWT = NTT / 32;
constexpr int NTW2 = 4;        // n-tiles of a 64 x 64 output per warp (warp tile 16 x 32)

// ---------------------------------------------------------------- shared memory carve-up (float offsets)
struct PpoSmem {
    int w1, w2, b1, b2, hw, hb, logstd, sig, x, h1, h2, dh, rowf, dmean, act, mu, part, bar, scratch, tacc, xch, pay, shr, shbar,
        total_bytes;
};
// shared: the launch trains shared trunk layers and needs the activation-gradient exchange's receive tiles and barriers
__host__ __device__ inline PpoSmem ppo_smem_layout(int LDX, int NP, bool shared = false) {
    PpoSmem s;
    int o = 0;
    s.w1 = o; o += H * LDX;          // W1[j][k], row stride LDX
    s.w2 = o; o += H * LDH;          // W2[j][k], row stride LDH
    s.b1 = o; o += H;
    s.b2 = o; o += H;
    s.hw = o; o += AMAX * WA_LD;
    s.hb = o; o += AMAX;
    s.logstd = o; o += AMAX;
    s.sig = o; o += 2 * AMAX;        // per action dim: 1/sigma^2, log(sigma) -- refreshed by the thread that updates log_std
    s.x = o; o += 2 * RBH * LDX;      // double buffered obs chunks (TMA destinations)
    s.h1 = o; o += RBH * LDH;
    s.h2 = o; o += RBH * LDH;
    s.dh = o; o += RBH * LDH;
    s.rowf = o; o += 2 * RBH * 8;    // per-row scalars of the stream: old_logp, adv_r, adv_c, ret_r, old_vr, ret_c, old_vc, (g)
    s.dmean = o; o += RBH * AMAX;
    s.act = o; o += 2 * RBH * AMAX;
    s.mu = o; o += RBH * AMAX;       // action-head outputs (means / logits)
    s.part = o; o += NWT * RBH * AMAX; // per-warp K-slice partials of the action head; later reused as the [16][LDH] dHW staging tile
    s.bar = o; o += 8;               // four 8-byte mbarriers: one per chunk buffer (TMA), pair exchange, norm exchange
    s.scratch = o; o += 128;
    s.tacc = o; o += 40;             // per-phase cycle counters of thread 0 (ICRL_PPO_TIMING): 20 x 8 bytes
    s.xch = o; o += 2 * 8 * 2;       // [parity][cluster rank][{sumsq, stop}]
    s.pay = o; o += NP * NTT;        // the partner CTA's gradient fragments land here (DSMEM stores)
    s.shr = o; o += shared ? 2 * RBH * H : 0;   // the two other trunks' [RBH][H] activation-gradient tiles (DSMEM stores)
    s.shbar = o; o += shared ? 4 : 0;           // two 8-byte mbarriers: tiles received, own tiles consumed by both peers
    s.total_bytes = o * 4;
    return s;
}

// one Adam update in torch's single-tensor form (torch/optim/adam.py); returns the new parameter
struct AdamConsts {
    float one_minus_b1, b2, one_minus_b2, inv_bc2_sqrt, eps, neg_step_size;
};
__device__ __forceinline__ float adam_update(float p, float g, float& m, float& v, const AdamConsts& c) {
    m = fmaf(c.one_minus_b1, g - m, m);                        // exp_avg.lerp_(grad, 1 - beta1)
    v = fmaf(c.one_minus_b2 * g, g, v * c.b2);                 // exp_avg_sq.mul_(beta2).addcmul_(g, g, 1 - beta2)
    // (sqrt(v) / sqrt(bc2)).add_(eps); param.addcdiv_(m, denom, value=-step_size).  The two divisions are done as a
    // multiply by the precomputed reciprocal, an approximate square root and a 2-ulp fast division: <= 5e-7 relative on
    // an lr-sized update.
    float sq;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq) : "f"(v));       // one MUFU op, <= 2 ulp (sqrtf's IEEE path costs ~8 instructions)
    const float denom = fmaf(sq, c.inv_bc2_sqrt, c.eps);
    return fmaf(c.neg_step_size, __fdividef(m, denom), p);
}

// ---------------------------------------------------------------- prologue kernels (massively parallel, HBM-bound)
// The minibatch schedule is known before the first optimiser step (numpy's permutations come from the host), so the
// random-access gather is taken OUT of the dependent step chain: one pass builds minibatch-ordered streams
//     xs[p][DP] obs (zero padded), as[p][AP] actions, ss[p][8] = {old_logp, adv_r, adv_c, ret_r, old_vr, ret_c, old_vc, -}
// for p = epoch*N + position, translating numpy's env-major index (row = e*T + t, buffers.py:52-65) to the buffer's
// time-major storage on the fly.  The persistent kernel then fetches each 64-row chunk with TMA bulk copies.
__global__ void __launch_bounds__(256) ppo_gather_kernel(const __grid_constant__ PpoArgs a, float* __restrict__ xs,
                                                         float* __restrict__ as, float* __restrict__ ss,
                                                         long long n_rows, long long n_alloc) {
    const int lane = threadIdx.x & 31;
    const int aw = a.is_discrete ? 1 : a.A;
    for (long long p = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); p < n_alloc; p += (long long)gridDim.x * 8) {
        int o = -1;
        if (p < n_rows) {
            const int row = a.perm[p], t = row % a.T, e = row / a.T;
            o = t * a.E + e;
        }
        for (int k = lane; k < a.DP; k += 32) xs[p * a.DP + k] = (o >= 0 && k < a.D) ? a.obs[(size_t)o * a.D + k] : 0.f;
        if (lane < a.AP) as[p * a.AP + lane] = (o >= 0 && lane < aw) ? a.act[(size_t)o * aw + lane] : 0.f;
        if (lane < 8) {
            float v = 0.f;
            if (o >= 0) {
                switch (lane) {
                    case 0: v = a.old_logp[o]; break;
                    case 1: v = a.adv_r[o]; break;
                    case 2: v = a.adv_c[o]; break;
                    case 3: v = a.ret_r[o]; break;
                    case 4: v = a.old_vr[o]; break;
                    case 5: v = a.ret_c[o]; break;
                    case 6: v = a.old_vc[o]; break;
                }
            }
            ss[p * 8 + lane] = v;
        }
    }
}

// One CTA per optimiser step: the minibatch statistics of ppo_lag.py:218-222 (mean and unbiased std of the reward
// advantages, mean of the cost advantages; float64 accumulation like ATen's CPU reductions) and that step's Adam bias
// corrections.  They depend only on data and the step number, never on parameters.
__global__ void __launch_bounds__(128) ppo_stats_kernel(const float* __restrict__ ss, float* __restrict__ advstats, int N,
                                                        int B, int spe, double beta1, double beta2, double lr,
                                                        long long step_before, const double* __restrict__ advsums) {
    __shared__ double red[2][4];
    const int step = blockIdx.x, epoch = step / spe, mb = step - epoch * spe;
    if (advsums != nullptr) {
        // data-parallel: statistics of the GLOBAL minibatch from the all-reduced sums (float64, so the one-pass
        // variance formula is safe)
        if (threadIdx.x == 0) {
            const double sx = advsums[step * 4 + 0], sxx = advsums[step * 4 + 1], sc = advsums[step * 4 + 2],
                         n = advsums[step * 4 + 3];
            const double mean = sx / n;
            advstats[step * 8 + 0] = (float)mean;
            advstats[step * 8 + 1] = (float)sqrt(fmax(sxx - sx * mean, 0.0) / (n - 1.0));
            advstats[step * 8 + 2] = (float)(sc / n);
            const double t = (double)(step_before + step + 1);
            advstats[step * 8 + 3] = (float)(1.0 / sqrt(1.0 - pow(beta2, t)));
            advstats[step * 8 + 4] = (float)(-(lr / (1.0 - pow(beta1, t))));
        }
        return;
    }
    const int Bn = min(B, N - mb * B);
    const size_t base = (size_t)epoch * N + (size_t)mb * B;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double sr = 0.0, sc = 0.0;
    for (int i = tid; i < Bn; i += blockDim.x) {
        sr += (double)ss[(base + i) * 8 + 1];
        sc += (double)ss[(base + i) * 8 + 2];
    }
    sr = warp_sum(sr); sc = warp_sum(sc);
    if (lane == 0) { red[0][warp] = sr; red[1][warp] = sc; }
    __syncthreads();
    const double mr = (red[0][0] + red[0][1] + red[0][2] + red[0][3]) / Bn;
    const double mc = (red[1][0] + red[1][1] + red[1][2] + red[1][3]) / Bn;
    __syncthreads();
    double ssq = 0.0;
    for (int i = tid; i < Bn; i += blockDim.x) {
        const double dv = (double)ss[(base + i) * 8 + 1] - mr;
        ssq += dv * dv;
    }
    ssq = warp_sum(ssq);
    if (lane == 0) red[0][warp] = ssq;
    __syncthreads();
    if (tid == 0) {
        const double tot = red[0][0] + red[0][1] + red[0][2] + red[0][3];
        advstats[step * 8 + 0] = (float)mr;
        advstats[step * 8 + 1] = (float)sqrt(tot / (double)(Bn - 1));
        advstats[step * 8 + 2] = (float)mc;
        // Adam bias corrections of optimiser step t (torch/optim/adam.py: 1 - beta ** step, python float64 pow)
        const double t = (double)(step_before + step + 1);
        advstats[step * 8 + 3] = (float)(1.0 / sqrt(1.0 - pow(beta2, t)));
        advstats[step * 8 + 4] = (float)(-(lr / (1.0 - pow(beta1, t))));
    }
}

// Local partial sums of the per-step advantage statistics (data-parallel mode): sum adv_r, sum adv_r^2, sum adv_c, count.
__global__ void __launch_bounds__(128) ppo_local_advsums_kernel(const int* __restrict__ perm, const float* __restrict__ adv_r,
                                                                const float* __restrict__ adv_c, int T, int E, int N, int B,
                                                                int spe, double* __restrict__ out) {
    __shared__ double red[3][4];
    const int step = blockIdx.x, epoch = step / spe, mb = step - epoch * spe;
    const int Bn = min(B, N - mb * B);
    const size_t base = (size_t)epoch * N + (size_t)mb * B;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double sx = 0.0, sxx = 0.0, sc = 0.0;
    for (int i = tid; i < Bn; i += blockDim.x) {
        const int row = perm[base + i], t = row % T, e = row / T, o = t * E + e;
        const double x = (double)adv_r[o];
        sx += x; sxx += x * x; sc += (double)adv_c[o];
    }
    sx = warp_sum(sx); sxx = warp_sum(sxx); sc = warp_sum(sc);
    if (lane == 0) { red[0][warp] = sx; red[1][warp] = sxx; red[2][warp] = sc; }
    __syncthreads();
    if (tid == 0) {
        out[step * 4 + 0] = red[0][0] + red[0][1] + red[0][2] + red[0][3];
        out[step * 4 + 1] = red[1][0] + red[1][1] + red[1][2] + red[1][3];
        out[step * 4 + 2] = red[2][0] + red[2][1] + red[2][2] + red[2][3];
        out[step * 4 + 3] = (double)Bn;
    }
}

__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

template <int NT1>
constexpr int ppo_frag_floats() { return NTW2 * 4 + NT1 * 4 + 4 + 1 + 5; }     // F: floats a thread owns in the exchanges
template <int NT1>
constexpr int ppo_pay_floats() { return (ppo_frag_floats<NT1>() + 3) / 4 * 4; }   // floats per thread of the pair-exchange buffer

template <bool IN_REGS>
struct TimingCounters;
template <>
struct TimingCounters<true> {
    unsigned long long v[20];
    __device__ __forceinline__ void init(void*, bool) {
#pragma unroll
        for (int i = 0; i < 20; ++i) v[i] = 0;
    }
    __device__ __forceinline__ unsigned long long& operator[](int i) { return v[i]; }
};
template <>
struct TimingCounters<false> {
    unsigned long long* v;
    __device__ __forceinline__ void init(void* smem, bool timed) {
        v = reinterpret_cast<unsigned long long*>(smem);
        if (timed)
            for (int i = 0; i < 20; ++i) v[i] = 0;
    }
    __device__ __forceinline__ unsigned long long& operator[](int i) { return v[i]; }
};

// ---------------------------------------------------------------- the persistent train kernel
// NT1 = n-tiles of dW1 (64 x KP) each warp owns (warp w: m-tile w & 3, n-tiles (w >> 2) + 2 i).
// WIDE (large batches): the launch holds a.ncl such clusters and covers ONE epoch.  Every cluster keeps a full replica of the
// weights / Adam moments and takes a contiguous slice of every minibatch; per optimiser step the clusters' pair-summed
// gradients meet in global memory (L2): write -> grid barrier -> each (cluster, half) sums its few floats over all clusters in
// cluster order (and, data parallel, exchanges that slice with the peer GPUs' same reducer over NVLink) -> grid barrier ->
// everybody reads the totals.  All replicas then apply the identical clip + Adam update, so they never diverge.
// SHARED (a.n_shared = 1 or 2 leading layers shared by the three trunks, MlpExtractor.shared_net; single GPU only): every
// trunk keeps a replica of the shared layers and recomputes them on its rows, which are the same rows as the other trunks'
// CTAs of the same half.  At the top of the shared part (dH1 with one shared layer, dH2 with two) the three CTAs of a half
// swap their activation-gradient tiles through DSMEM and each adds the three in the fixed order (pi + vf) + cvf, so every
// layer below back-propagates the same bits in all three trunks: the replicas get identical gradients, moments and updates
// without any weight-gradient exchange.  Only the pi CTAs count the shared gradients in the norm and write them back.
template <int NT1, bool DIST, bool WIDE, bool TIMED, bool SHARED = false>
#ifdef ICRL_K4_MAXREG       // A/B builds (tools/build_variants.sh): an explicit register cap instead of the launch bounds
#define ICRL_K4_BOUNDS __maxnreg__(ICRL_K4_MAXREG)
#else
#define ICRL_K4_BOUNDS __launch_bounds__(NTT, 1)
#endif
__global__ void ICRL_K4_BOUNDS ppo_train_kernel(const __grid_constant__ PpoArgs a) {
    extern __shared__ __align__(16) float sm[];
    if (WIDE && a.result[3] != 0) return;     // an earlier epoch's launch hit the target_kl stop: nothing left to do
    const float nu = a.nu_dev ? *a.nu_dev : a.nu;
    const int cluster_id = WIDE ? (int)(blockIdx.x / NCTA) : 0;
    const int ncl = WIDE ? a.ncl : 1;
    // rows of a minibatch this cluster takes: [cluster_id * Bc, (cluster_id + 1) * Bc) clipped to the minibatch
    const int Bc = WIDE ? ((a.B + ncl - 1) / ncl + RB - 1) / RB * RB : 0;
    auto range_lo = [&](int Bn) { return WIDE ? min(cluster_id * Bc, Bn) : 0; };
    auto range_len = [&](int Bn) { return WIDE ? max(min((cluster_id + 1) * Bc, Bn) - cluster_id * Bc, 0) : Bn; };
    const int LDX = a.DP, KP = a.KP, D = a.D;
    // payload of the pair exchange: gradient fragments + the five loss partial sums (thread 0)
    constexpr int NP = ppo_pay_floats<NT1>();
    constexpr int PAY_V4 = NTW2 + NT1 + 3;      // float4 groups every thread sends to its partner per step
    static_assert(PAY_V4 * 4 <= NP, "PAY too small");
    // bytes a CTA receives per step: every thread's groups, except the last one ({kl, entropy} sums), which only the threads
    // that own loss partials (hq == 0: every 8th) send
    constexpr int PAY_BYTES = (PAY_V4 - 1) * NTT * 16 + (NTT / 8) * 16;
    const PpoSmem L = ppo_smem_layout(LDX, NP, SHARED);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int crank = (int)cluster_ctarank();       // cluster rank: trunk = crank / 2 (0 pi, 1 vf, 2 cvf), half = crank % 2
    const int ncta = (int)cluster_nctarank();
    const int role = crank >> 1, half = crank & 1;
    const bool working = crank < NCTA;
    const int trunk = working ? role : 0;
    const int AOUT = (role == 0) ? a.A : 1;
    const bool has_logstd = (role == 0) && !a.is_discrete;
    // this CTA counts (norm) and writes back layer 1 / layer 2 of its trunk: a shared layer belongs to the pi CTAs
    const bool own_l1 = !SHARED || role == 0;
    const bool own_l2 = !SHARED || role == 0 || a.n_shared < 2;

    float* W1 = sm + L.w1; float* W2 = sm + L.w2;
    float* B1 = sm + L.b1; float* B2 = sm + L.b2; float* HW = sm + L.hw; float* HB = sm + L.hb;
    float* LOGSTD = sm + L.logstd; float* SIG = sm + L.sig;
    float* X = sm + L.x; float* H1 = sm + L.h1; float* H2 = sm + L.h2; float* DH = sm + L.dh;
    float* ROWF = sm + L.rowf; float* DMEAN = sm + L.dmean; float* ACT = sm + L.act; float* MU = sm + L.mu;
    float* PART = sm + L.part;
    uint64_t* BAR = reinterpret_cast<uint64_t*>(sm + L.bar);
    float* scratch = sm + L.scratch;
    float* XCH = sm + L.xch;
    float* PAY = sm + L.pay;

    // ---- warp tiling of every 64 x 64 (or 64 x KP) GEMM output, and the parameter ownership that follows from it
    const int g = lane >> 2, t = lane & 3;          // mma fragment coordinates
    const int mt = warp & 3, ng = warp >> 2;        // warp's m-tile (16 rows) and n-group (32 columns of a 64-wide output)
    // W2[j][k] owned by this thread: j = 16 mt + g (+8), k = 32 ng + 8 nt + 2 t (+1), nt < 4     -> [nt][c] as the C fragment
    // W1[j][k] owned by this thread: j as above,        k = 8 (ng + 2 i) + 2 t (+1),  i < NT1   (valid while k < KP)
    const int oj = 16 * mt + g;
    auto w2_k = [&](int nt) { return 32 * ng + 8 * nt + 2 * t; };
    auto w1_k = [&](int i) { return 8 * (ng + 2 * i) + 2 * t; };
    const int hd = tid >> 4, hk4 = tid & 15;        // head weight: row hd, cols 4*hk4..
    int s_kind = -1, s_idx = 0;                     // scalar slot: b1 | b2 | head bias | log_std
    if (tid < 64) { s_kind = 0; s_idx = tid; }
    else if (tid < 128) { s_kind = 1; s_idx = tid - 64; }
    else if (tid < 128 + AOUT) { s_kind = 2; s_idx = tid - 128; }
    else if (tid >= 160 && tid < 160 + a.A && has_logstd) { s_kind = 3; s_idx = tid - 160; }

    // flat index of an owned parameter, -1 for the padding of this CTA's trunk
    auto flat_w2 = [&](int j, int k) {
        const int h0 = a.h0[trunk];
        return (j < a.h1[trunk] && k < h0) ? a.off_w2[trunk] + j * h0 + k : -1;
    };
    auto flat_w1 = [&](int j, int k) { return (j < a.h0[trunk] && k < D) ? a.off_w1[trunk] + j * D + k : -1; };
    auto flat_hw = [&](int d, int k) {
        const int h1 = a.h1[trunk];
        return (d < AOUT && k < h1) ? a.off_hw[trunk] + d * h1 + k : -1;
    };
    auto flat_scalar = [&]() {
        switch (s_kind) {
            case 0: return s_idx < a.h0[trunk] ? a.off_b1[trunk] + s_idx : -1;
            case 1: return s_idx < a.h1[trunk] ? a.off_b2[trunk] + s_idx : -1;
            case 2: return a.off_hb[trunk] + s_idx;
            case 3: return a.off_logstd + s_idx;
        }
        return -1;
    };
    // element c of an owned fragment -> (row, column offset)
    auto frag_j = [&](int c) { return oj + ((c & 2) ? 8 : 0); };
    auto frag_dk = [&](int c) { return c & 1; };

    // ---- parameters -> shared memory (zero padded), Adam moments -> registers
    float m_w2[NTW2][4], v_w2[NTW2][4], m_w1[NT1][4], v_w1[NT1][4], m_hw[4], v_hw[4], m_s = 0.f, v_s = 0.f;
    for (int i = tid; i < H * LDX; i += NTT) {
        const int j = i / LDX, k = i - j * LDX;
        const int f = working ? flat_w1(j, k) : -1;
        W1[i] = f >= 0 ? a.params[f] : 0.f;
    }
    for (int i = tid; i < H * LDH; i += NTT) {
        const int j = i / LDH, k = i - j * LDH;
        const int f = (working && k < H) ? flat_w2(j, k) : -1;
        W2[i] = f >= 0 ? a.params[f] : 0.f;
    }
    for (int i = tid; i < AMAX * WA_LD; i += NTT) {
        const int d = i / WA_LD, k = i - d * WA_LD;
        const int f = working ? flat_hw(d, k) : -1;
        HW[i] = f >= 0 ? a.params[f] : 0.f;
    }
    if (tid < H) { B1[tid] = 0.f; B2[tid] = 0.f; }
    if (tid < AMAX) { HB[tid] = 0.f; LOGSTD[tid] = 0.f; }
    if (tid < 32) XCH[tid] = 0.f;
    for (int i = tid; i < RBH * AMAX; i += NTT) DMEAN[i] = 0.f;   // unused head columns stay zero (they feed the MMA tiles)
    __syncthreads();
#pragma unroll
    for (int nt = 0; nt < NTW2; ++nt)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int f = working ? flat_w2(frag_j(c), w2_k(nt) + frag_dk(c)) : -1;
            m_w2[nt][c] = f >= 0 ? a.adam_m[f] : 0.f;
            v_w2[nt][c] = f >= 0 ? a.adam_v[f] : 0.f;
        }
#pragma unroll
    for (int i = 0; i < NT1; ++i)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int f = working ? flat_w1(frag_j(c), w1_k(i) + frag_dk(c)) : -1;
            m_w1[i][c] = f >= 0 ? a.adam_m[f] : 0.f;
            v_w1[i][c] = f >= 0 ? a.adam_v[f] : 0.f;
        }
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
        const int f = working ? flat_hw(hd, 4 * hk4 + kk) : -1;
        m_hw[kk] = f >= 0 ? a.adam_m[f] : 0.f;
        v_hw[kk] = f >= 0 ? a.adam_v[f] : 0.f;
    }
    if (working) {
        const int f = flat_scalar();
        if (f >= 0) {
            m_s = a.adam_m[f]; v_s = a.adam_v[f];
            const float p = a.params[f];
            if (s_kind == 0) B1[s_idx] = p; else if (s_kind == 1) B2[s_idx] = p;
            else if (s_kind == 2) HB[s_idx] = p; else LOGSTD[s_idx] = p;
        }
    }
    __syncthreads();
    if (tid < AMAX) {
        const float sigma = expf(LOGSTD[tid]);
        SIG[tid] = 1.f / (sigma * sigma);
        SIG[AMAX + tid] = logf(sigma);
    }
    if (tid == 0) {
        mbar_init(&BAR[0], 1);
        mbar_init(&BAR[1], 1);
        mbar_init(&BAR[2], 1);     // pair exchange: armed by thread 0 every step, completed by the partner's st.async bytes
        mbar_init(&BAR[3], 1);     // norm exchange: completed by one 8-byte st.async from each CTA of the cluster
        if constexpr (SHARED) {
            uint64_t* SB = reinterpret_cast<uint64_t*>(sm + L.shbar);
            mbar_init(&SB[0], 1);  // tiles received: armed by thread 0 every chunk, completed by the two peers' st.async bytes
            mbar_init(&SB[1], 2);  // own tile consumed: one remote arrival from each of the two peers per chunk
        }
        fence_mbar_init();
    }
    __syncthreads();
    cluster_sync_all();   // every CTA has zeroed its exchange slots before any peer writes into them

    const int hr = tid >> 3, hq = tid & 7;      // head mapping: row hr (RBH rows), eighth hq
    const int mtf = warp & 1, ngf = warp >> 1;  // forward / dH1 tiling of a 32 x 64 output: m-tile, 16-column group
    const int ojf = 16 * mtf + g;
    auto fw_k = [&](int nt) { return 16 * ngf + 8 * nt + 2 * t; };
    const int AP = a.AP;

    // ---- chunk pipeline: chunk q+1 of the minibatch-ordered streams is fetched by TMA bulk copies (one elected thread,
    // completion on an mbarrier) while chunk q is being computed.  No global latency is exposed to the step chain.
    struct Cursor { int epoch, mb, c0; };
    auto cur_valid = [&](const Cursor& c) { return c.epoch < a.n_epochs; };
    auto cur_bn = [&](const Cursor& c) { return min(a.B, a.N - c.mb * a.B); };
    auto cur_len = [&](const Cursor& c) { return range_len(cur_bn(c)); };
    auto cur_skip_empty = [&](Cursor c) {      // (wide mode) minibatches in which this cluster has no rows
        while (cur_valid(c) && cur_len(c) == 0) { if (++c.mb >= a.steps_per_epoch) { c.mb = 0; ++c.epoch; } }
        return c;
    };
    auto cur_next = [&](Cursor c) {
        c.c0 += RB;
        if (c.c0 >= cur_len(c)) { c.c0 = 0; if (++c.mb >= a.steps_per_epoch) { c.mb = 0; ++c.epoch; } c = cur_skip_empty(c); }
        return c;
    };
    auto fetch_chunk = [&](const Cursor& c, int buf) {   // called by thread 0 only
        const size_t p = (size_t)c.epoch * a.N + (size_t)c.mb * a.B + range_lo(cur_bn(c)) + c.c0 + RBH * half;   // streams carry RB rows of tail padding
        const uint32_t xb = RBH * LDX * 4, sb = RBH * 8 * 4, ab = (role == 0) ? RBH * AP * 4 : 0;
        fence_proxy_async();   // the row buffer takes one generic-proxy write per row (dL/dlogp): order it before the async-proxy writes
        mbar_expect_tx(&BAR[buf], xb + sb + ab);
        bulk_g2s(X + buf * RBH * LDX, a.xs + p * LDX, xb, &BAR[buf]);
        bulk_g2s(ROWF + buf * RBH * 8, a.ss + p * 8, sb, &BAR[buf]);
        if (role == 0) bulk_g2s(ACT + buf * RBH * AMAX, a.as + p * AP, ab, &BAR[buf]);
    };

    // ---- shared trunk layers: swap this chunk's activation-gradient tile T ([RBH][LDH]) with the CTAs of the same half of the
    // other two trunks (the same rows) and replace it by the sum of the three in trunk order, identical bits in every trunk.
    // One receive tile per peer: two per peer do not fit beside the NT1 = 8 layout (200.3 + 32 KB > 227 KB).  So a CTA sends
    // its tile of chunk qx only after both peers have consumed the one of chunk qx - 1: each CTA arrives on both peers'
    // "consumed" mbarrier after its sum and waits on its own before it sends.
    auto share_tile = [&](float* T, int qx) {
        if constexpr (SHARED) {
            uint64_t* SB = reinterpret_cast<uint64_t*>(sm + L.shbar);
            float* RX = sm + L.shr;
            if (qx > 0 && *(volatile float*)&XCH[31] == 0.f &&
                !mbar_wait_bounded_cluster(&SB[1], (uint32_t)((qx - 1) & 1), 2000000000LL))
                XCH[31] = 1.f;
            float4 mine[2];                                   // float4 groups i = tid, tid + 256 of the 32 x 64 tile
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int i = tid + u * NTT;
                mine[u] = *reinterpret_cast<const float4*>(T + (i >> 4) * LDH + 4 * (i & 15));
            }
#pragma unroll
            for (int pp = 1; pp < 3; ++pp) {
                const int prole = (role + pp) % 3;
                const uint32_t prank = (uint32_t)(2 * prole + half);
                const int slot = role - (role > prole ? 1 : 0);   // a receiver's two slots hold the other trunks in trunk order
                uint32_t rx, rb;
                asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rx) : "r"(smem_u32(RX + slot * RBH * H)), "r"(prank));
                asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rb) : "r"(smem_u32(&SB[0])), "r"(prank));
#pragma unroll
                for (int u = 0; u < 2; ++u)
                    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(
                                     rx + (uint32_t)((tid + u * NTT) * 16)),
                                 "f"(mine[u].x), "f"(mine[u].y), "f"(mine[u].z), "f"(mine[u].w), "r"(rb) : "memory");
            }
            if (*(volatile float*)&XCH[31] == 0.f && !mbar_wait_bounded(&SB[0], (uint32_t)(qx & 1), 2000000000LL)) XCH[31] = 1.f;
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int i = tid + u * NTT;
                const float4 x = *reinterpret_cast<const float4*>(RX + 4 * i);
                const float4 y = *reinterpret_cast<const float4*>(RX + RBH * H + 4 * i);
                const float4 t0 = role == 0 ? mine[u] : x;
                const float4 t1 = role == 0 ? x : role == 1 ? mine[u] : y;
                const float4 t2 = role == 2 ? mine[u] : y;
                *reinterpret_cast<float4*>(T + (i >> 4) * LDH + 4 * (i & 15)) =
                    make_float4((t0.x + t1.x) + t2.x, (t0.y + t1.y) + t2.y, (t0.z + t1.z) + t2.z, (t0.w + t1.w) + t2.w);
            }
            __syncthreads();          // the sum is complete in T, and no thread of this CTA reads its slots any more
            if (tid < 2) {            // thread p tells peer p that its tile of this chunk has been consumed
                uint32_t rb;
                asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rb)
                             : "r"(smem_u32(&SB[1])), "r"((uint32_t)(2 * ((role + 1 + tid) % 3) + half)));
                asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(rb) : "memory");
            }
        }
    };

    Cursor cur = cur_skip_empty(Cursor{0, 0, 0});
    int q = 0;                                   // running chunk counter (buffer parity / mbarrier phase)
    if (working && tid == 0 && cur_valid(cur)) fetch_chunk(cur, 0);

    int step = 0, early_stop_epoch = a.n_epochs;
    bool kl_stopped = false;
    double epoch_kl_sum = 0.0;
    bool stop_all = false;
    // TIMED = false (every launch unless ICRL_PPO_TIMING is set): the per-phase counters and their marks are compiled out --
    // measured 1.3 % (HalfCheetah) to 4.7 % (AntWall) per optimiser step against a run-time `if (timed)` around every mark
    const bool timed = TIMED && (a.timing != nullptr) && tid == 0 && working && cluster_id == 0;
    long long tmark = clock64();
    // per-phase cycle counters of thread 0 (ICRL_PPO_TIMING).  Measured (profiles/k4_variants_r02.txt): the wide dW1 tiles
    // (NT1 >= 4, AntWall) have no registers to spare -- keeping the 20 counters in shared memory takes 21.5 -> 19.5 us per
    // optimiser step there -- while the HalfCheetah instantiation is 2 % faster with them in registers.
    TimingCounters<(NT1 <= 2)> tacc;
    if (TIMED) tacc.init(sm + L.tacc, timed);
#define ICRL_MARK(i)                                   \
    if (TIMED && timed) {                              \
        const long long now__ = clock64();             \
        tacc[i] += (unsigned long long)(now__ - tmark); \
        tmark = now__;                                 \
    }

    for (int epoch = 0; epoch < a.n_epochs && !stop_all; ++epoch) {
        epoch_kl_sum = 0.0;
        int epoch_steps = 0;
        for (int mb = 0; mb < a.steps_per_epoch && !stop_all; ++mb, ++step) {
            const int parity = step & 1;
            const int Bn = min(a.B, a.N - mb * a.B);
            const float invB = 1.0f / (float)(Bn * a.world);   // data-parallel: every rank holds Bn rows of the global minibatch

            // gradient accumulators (registers, mma C-fragment layout)
            float g_w2[NTW2][4], g_w1[NT1][4], g_hw[4], g_s = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i) g_hw[i] = 0.f;
#pragma unroll
            for (int i = 0; i < NTW2; ++i)
#pragma unroll
                for (int c = 0; c < 4; ++c) g_w2[i][c] = 0.f;
#pragma unroll
            for (int i = 0; i < NT1; ++i)
#pragma unroll
                for (int c = 0; c < 4; ++c) g_w1[i][c] = 0.f;
            // loss partial sums (thread-local, one merged block reduction at the end of the step)
            float s_a = 0.f, s_b = 0.f, s_c = 0.f, s_d = 0.f, s_e = 0.f;
            // minibatch statistics of the advantages (ppo_lag.py:218-222) and Adam constants from the prologue's table
            const float adv_mean_r = a.advstats[step * 8 + 0], adv_std_r = a.advstats[step * 8 + 1],
                        adv_mean_c = a.advstats[step * 8 + 2];
            const float adam_inv_bc2_sqrt = a.advstats[step * 8 + 3], adam_neg_step = a.advstats[step * 8 + 4];

            // DSMEM address of this thread's slot in the PARTNER CTA's PAY buffer; gradient groups are pushed as soon as
            // they are final (asynchronous stores that overlap the rest of the backward pass)
            uint32_t pay_remote = 0;
            if (working) {
                const uint32_t local = smem_u32(PAY + 4 * tid);
                asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(pay_remote) : "r"(local), "r"((uint32_t)(crank ^ 1)));
            }
            // st.async: the store completes 16 transaction bytes on the PARTNER's pair-exchange mbarrier when it lands, so the
            // receiver waits on its own mbarrier instead of a cluster barrier
            uint32_t pbar_remote = 0;
            if (working) {
                asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(pbar_remote) : "r"(smem_u32(&BAR[2])), "r"((uint32_t)(crank ^ 1)));
            }
            auto st4 = [&](int v4, float x, float y, float z, float w) {
                asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(
                                 pay_remote + (uint32_t)(v4 * NTT * 16)),
                             "f"(x), "f"(y), "f"(z), "f"(w), "r"(pbar_remote) : "memory");
            };
            const int len = range_len(Bn);           // rows of this minibatch that THIS cluster processes
            if (working) {
                for (int c0 = 0; c0 < len; c0 += RB, ++q) {
                    const bool last_chunk = (c0 + RB >= len);
                    const int rows = min(max(min(RB, len - c0) - RBH * half, 0), RBH);   // valid rows of THIS CTA's half
                    const int buf = q & 1;
                    const float* Xc = X + buf * RBH * LDX;
                    float* Rc = ROWF + buf * RBH * 8;
                    const float* Ac = ACT + buf * RBH * AMAX;   // rows at stride AP (as the stream stores them)
                    mbar_wait(&BAR[buf], (uint32_t)((q >> 1) & 1));
                    __syncthreads();          // chunk q landed, and everybody is done with chunk q-1's buffers
                    if (c0 == 0 && tid == 0) {
                        // arm this step's exchange barriers.  After the __syncthreads above no thread of this CTA is still
                        // waiting on the previous phase, and bytes that arrive before the arming are accounted for (the
                        // phase cannot complete without this arrival).
                        mbar_expect_tx(&BAR[2], (uint32_t)PAY_BYTES);
                        mbar_expect_tx(&BAR[3], (uint32_t)(NCTA * 8));
                    }
                    if constexpr (SHARED) {   // this chunk's shared-layer tiles from the two peers (see share_tile)
                        if (tid == 0) mbar_expect_tx(reinterpret_cast<uint64_t*>(sm + L.shbar), (uint32_t)(2 * RBH * H * 4));
                    }
                    ICRL_MARK(0)
                    {
                        const Cursor nxt = cur_next(cur);
                        if (tid == 0 && cur_valid(nxt)) fetch_chunk(nxt, buf ^ 1);
                        cur = nxt;
                    }
                    ICRL_MARK(1)

                    // ---- forward layer 1: H1 = tanh(X W1^T + b1)          [warp tile: rows 16mt.., cols 32ng..]
                    {
                        float acc[2][4];
#pragma unroll
                        for (int nt = 0; nt < 2; ++nt) {
                            const float2 b = *reinterpret_cast<const float2*>(B1 + fw_k(nt));
                            acc[nt][0] = b.x; acc[nt][1] = b.y; acc[nt][2] = b.x; acc[nt][3] = b.y;
                        }
                        // compile-time trip count for the two K values that map to this NT1 exactly (all named workloads): fully
                        // unrolled, so the fragment loads of later k-steps are issued ahead of the MMAs
                        if (KP == 16 * NT1)
                            warp_gemm_3xtf32<2, 16 * NT1>(acc, Xc + 16 * mtf * LDX, LDX, 1, W1, 1, LDX, 16 * NT1, 16 * ngf, 8, H, g, t);
                        else if (KP == 16 * NT1 - 8)
                            warp_gemm_3xtf32<2, 16 * NT1 - 8>(acc, Xc + 16 * mtf * LDX, LDX, 1, W1, 1, LDX, 16 * NT1 - 8, 16 * ngf, 8, H, g, t);
                        else
                            warp_gemm_3xtf32<2>(acc, Xc + 16 * mtf * LDX, LDX, 1, W1, 1, LDX, KP, 16 * ngf, 8, H, g, t);
#pragma unroll
                        for (int nt = 0; nt < 2; ++nt) {
                            *reinterpret_cast<float2*>(H1 + ojf * LDH + fw_k(nt)) = make_float2(tanhf(acc[nt][0]), tanhf(acc[nt][1]));
                            *reinterpret_cast<float2*>(H1 + (ojf + 8) * LDH + fw_k(nt)) = make_float2(tanhf(acc[nt][2]), tanhf(acc[nt][3]));
                        }
                    }
                    __syncthreads();
                    ICRL_MARK(2)
                    // ---- forward layer 2: H2 = tanh(H1 W2^T + b2)
                    {
                        float acc[2][4];
#pragma unroll
                        for (int nt = 0; nt < 2; ++nt) {
                            const float2 b = *reinterpret_cast<const float2*>(B2 + fw_k(nt));
                            acc[nt][0] = b.x; acc[nt][1] = b.y; acc[nt][2] = b.x; acc[nt][3] = b.y;
                        }
                        warp_gemm_3xtf32<2, H>(acc, H1 + 16 * mtf * LDH, LDH, 1, W2, 1, LDH, H, 16 * ngf, 8, H, g, t);
#pragma unroll
                        for (int nt = 0; nt < 2; ++nt) {
#pragma unroll
                            for (int c = 0; c < 4; ++c) acc[nt][c] = tanhf(acc[nt][c]);
                            *reinterpret_cast<float2*>(H2 + ojf * LDH + fw_k(nt)) = make_float2(acc[nt][0], acc[nt][1]);
                            *reinterpret_cast<float2*>(H2 + (ojf + 8) * LDH + fw_k(nt)) = make_float2(acc[nt][2], acc[nt][3]);
                        }
                        if (role == 0) {
                            // action head, fused into this epilogue: the warp's 16 x 16 tile of H2 is still in registers in the
                            // MMA C layout; with the K index permuted (k' = 2t -> slot t, 2t + 1 -> slot t + 4, the same
                            // permutation applied to the HW operand) it IS an A fragment, so the warp multiplies its tile by
                            // its 16-column slice of HW^T right away.  The four partial [16 x A] tiles of a row block meet
                            // in PART after the barrier.
                            const int nmaxA = (a.A + 7) & ~7;
                            float pacc[2][4];
#pragma unroll
                            for (int no = 0; no < 2; ++no)
#pragma unroll
                                for (int c = 0; c < 4; ++c) pacc[no][c] = 0.f;
#pragma unroll
                            for (int nt = 0; nt < 2; ++nt) {
                                uint32_t ahi[4], alo[4];
                                split_tf32(acc[nt][0], ahi[0], alo[0]);
                                split_tf32(acc[nt][2], ahi[1], alo[1]);
                                split_tf32(acc[nt][1], ahi[2], alo[2]);
                                split_tf32(acc[nt][3], ahi[3], alo[3]);
#pragma unroll
                                for (int no = 0; no < 2; ++no) {
                                    if (8 * no < nmaxA) {
                                        const float2 b = *reinterpret_cast<const float2*>(HW + (8 * no + g) * WA_LD + fw_k(nt));
                                        uint32_t bhi[2], blo[2];
                                        split_tf32(b.x, bhi[0], blo[0]);
                                        split_tf32(b.y, bhi[1], blo[1]);
                                        mma_tf32(pacc[no], alo, bhi);
                                        mma_tf32(pacc[no], ahi, blo);
                                        mma_tf32(pacc[no], ahi, bhi);
                                    }
                                }
                            }
#pragma unroll
                            for (int no = 0; no < 2; ++no) {
                                if (8 * no < nmaxA) {
                                    float* pp = PART + (ngf * RBH + ojf) * AMAX + 8 * no + 2 * t;
                                    *reinterpret_cast<float2*>(pp) = make_float2(pacc[no][0], pacc[no][1]);
                                    *reinterpret_cast<float2*>(pp + 8 * AMAX) = make_float2(pacc[no][2], pacc[no][3]);
                                }
                            }
                        }
                    }
                    __syncthreads();
                    ICRL_MARK(3)

                    // ---- heads + losses + d(loss)/d(head output).  8 threads per row (hr < RBH, hq < 8).
                    if (role == 0) {
                        // outputs d = hq, hq + 8 of row hr
                        float out[2];
#pragma unroll
                        for (int u = 0; u < 2; ++u) {
                            const int d = hq + 8 * u;
                            float acc = 0.f;
                            if (d < a.A) {
                                acc = HB[d];
#pragma unroll
                                for (int q4 = 0; q4 < 4; ++q4) acc += PART[(q4 * RBH + hr) * AMAX + d];   // the four column groups
                            }
                            out[u] = acc;
                            MU[hr * AMAX + d] = acc;
                        }
                        ICRL_MARK(11)
                        const bool valid = hr < rows;
                        float logp = 0.f, ent = 0.f;
                        float dcoef[2] = {0.f, 0.f};   // d logp / d out[u]
                        float dent[2] = {0.f, 0.f};    // d entropy / d out[u] (discrete only)
                        auto sum8 = [](float v) {
                            v += __shfl_xor_sync(0xffffffffu, v, 1);
                            v += __shfl_xor_sync(0xffffffffu, v, 2);
                            v += __shfl_xor_sync(0xffffffffu, v, 4);
                            return v;
                        };
                        if (!a.is_discrete) {
                            float lp = 0.f, en = 0.f;
#pragma unroll
                            for (int u = 0; u < 2; ++u) {
                                const int d = hq + 8 * u;
                                if (d < a.A) {
                                    const float inv_var = SIG[d], log_scale = SIG[AMAX + d];
                                    const float diff = Ac[hr * AP + d] - out[u];
                                    lp += -(diff * diff) * (0.5f * inv_var) - log_scale - LOG_SQRT_2PI;
                                    en += HALF_LOG_2PI_PLUS_HALF + log_scale;
                                    dcoef[u] = diff * inv_var;
                                }
                            }
                            logp = sum8(lp); ent = sum8(en);
                        } else {
                            float mx = -INFINITY;
#pragma unroll
                            for (int u = 0; u < 2; ++u) if (hq + 8 * u < a.A) mx = fmaxf(mx, out[u]);
                            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
                            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
                            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 4));
                            float se = 0.f;
#pragma unroll
                            for (int u = 0; u < 2; ++u) if (hq + 8 * u < a.A) se += expf(out[u] - mx);
                            se = sum8(se);
                            const float lse = mx + logf(se);
                            const int ai = (int)Ac[hr * AP + 0];
                            float lp = 0.f, en = 0.f, pr[2], lg[2];
#pragma unroll
                            for (int u = 0; u < 2; ++u) {
                                const int d = hq + 8 * u;
                                pr[u] = 0.f; lg[u] = 0.f;
                                if (d < a.A) {
                                    lg[u] = out[u] - lse;
                                    pr[u] = expf(lg[u]);
                                    en -= lg[u] * pr[u];
                                    if (d == ai) lp = lg[u];
                                }
                            }
                            logp = sum8(lp); ent = sum8(en);
#pragma unroll
                            for (int u = 0; u < 2; ++u) {
                                const int d = hq + 8 * u;
                                if (d < a.A) {
                                    dcoef[u] = (d == ai ? 1.f : 0.f) - pr[u];
                                    dent[u] = -pr[u] * (lg[u] + ent);
                                }
                            }
                        }
                        // surrogate (ppo_lag.py:218-236); advantages normalised here with the minibatch statistics
                        const float old_lp = Rc[hr * 8 + 0];
                        const float A_r = (Rc[hr * 8 + 1] - adv_mean_r) / (adv_std_r + 1e-8f);
                        const float A_c = Rc[hr * 8 + 2] - adv_mean_c;
                        const float ratio = expf(logp - old_lp);
                        const float lo = 1.f - a.clip_range, hi = 1.f + a.clip_range;
                        const float clipped = fminf(fmaxf(ratio, lo), hi);
                        const float pl1 = A_r * ratio, pl2 = A_r * clipped;
                        const bool inrange = (ratio >= lo) && (ratio <= hi);
                        float wgt;   // d min(pl1, pl2) / d ratio divided by A_r (torch.min splits ties evenly)
                        if (pl1 < pl2) wgt = 1.f;
                        else if (pl1 > pl2) wgt = inrange ? 1.f : 0.f;
                        else wgt = 0.5f + (inrange ? 0.5f : 0.f);
                        const float inv1pnu = 1.f / (1.f + nu);
                        float gl = 0.f;
                        if (valid) {
                            gl = ratio * (-A_r * wgt + nu * A_c) * invB * inv1pnu;       // dL/dlogp
                            if (hq == 0) {
                                s_a += fminf(pl1, pl2);                                   // sum min(pl1, pl2)
                                s_b += A_c * ratio;                                       // sum cost_adv * ratio
                                s_c += (fabsf(ratio - 1.f) > a.clip_range) ? 1.f : 0.f;   // clip count
                                s_d += old_lp - logp;                                     // approx kl numerator
                                s_e += ent;                                               // entropy sum
                            }
                        }
                        const float ge = valid ? -a.ent_coef * invB : 0.f;               // d(ent_coef*entropy_loss)/d ent
#pragma unroll
                        for (int u = 0; u < 2; ++u) {
                            const int d = hq + 8 * u;
                            DMEAN[hr * AMAX + d] = (d < a.A) ? (gl * dcoef[u] + ge * dent[u]) : 0.f;
                        }
                        if (hq == 0) Rc[hr * 8 + 7] = gl;
                    } else {
                        // value head: partial dot over k in [8hq, 8hq+8)
                        float acc = 0.f;
                        const float4* hrow = reinterpret_cast<const float4*>(H2 + hr * LDH + 8 * hq);
                        const float4* wrow = reinterpret_cast<const float4*>(HW + 8 * hq);
#pragma unroll
                        for (int k = 0; k < 2; ++k) {
                            const float4 h = hrow[k], w = wrow[k];
                            acc = fmaf(h.x, w.x, acc); acc = fmaf(h.y, w.y, acc);
                            acc = fmaf(h.z, w.z, acc); acc = fmaf(h.w, w.w, acc);
                        }
                        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
                        acc += __shfl_xor_sync(0xffffffffu, acc, 2);
                        acc += __shfl_xor_sync(0xffffffffu, acc, 4);
                        const float V = acc + HB[0];
                        const float target = Rc[hr * 8 + (role == 1 ? 3 : 5)], oldv = Rc[hr * 8 + (role == 1 ? 4 : 6)];
                        const bool clipvf = (role == 1) ? a.has_clip_vf_r : a.has_clip_vf_c;
                        const float cr = (role == 1) ? a.clip_vf_r : a.clip_vf_c;
                        float Vp = V, pass = 1.f;
                        if (clipvf) {
                            const float dv = V - oldv;
                            Vp = oldv + fminf(fmaxf(dv, -cr), cr);
                            pass = (dv >= -cr && dv <= cr) ? 1.f : 0.f;
                        }
                        const float coef = (role == 1) ? a.vf_coef_r : a.vf_coef_c;
                        const float err = Vp - target;
                        float dV = 0.f;
                        if (hr < rows) {
                            dV = coef * 2.f * err * invB * pass;
                            if (hq == 0) s_a += err * err;
                        }
                        if (hq == 0) { DMEAN[hr * AMAX + 0] = dV; }
                    }
                    ICRL_MARK(12)
                    __syncthreads();
                    ICRL_MARK(4)

                    // ---- head weight gradient G[d][k] = sum_r dmean[r][d] H2[r][k] on tensor cores (rows beyond `rows` carry zero
                    // dmean): warp w owns columns [8w, 8w + 8); the tile is staged in shared memory and added by the owner
                    // threads after the next barrier
                    {
                        float acc[1][4] = {{0.f, 0.f, 0.f, 0.f}};
                        warp_gemm_3xtf32<1, RBH>(acc, DMEAN, 1, AMAX, H2 + 8 * warp, LDH, 1, RBH, 0, 8, 8, g, t);   // (DMEAN's stride 16 would turn KPERM into 4-way conflicts)
                        float* sp = PART + g * LDH + 8 * warp + 2 * t;
                        *reinterpret_cast<float2*>(sp) = make_float2(acc[0][0], acc[0][1]);
                        *reinterpret_cast<float2*>(sp + 8 * LDH) = make_float2(acc[0][2], acc[0][3]);
                    }
                    ICRL_MARK(13)
                    if (s_kind == 2) {
                        float acc = 0.f;
#pragma unroll 8
                        for (int r = 0; r < RBH; ++r) acc += DMEAN[r * AMAX + s_idx];
                        g_s += acc;
                    } else if (s_kind == 3) {
                        // d logp / d log_std_d = diff^2/var - 1 ; entropy: d(-mean H)/d log_std = -1
                        const float inv_var = SIG[s_idx];
                        float acc = 0.f;
#pragma unroll 8
                        for (int r = 0; r < RBH; ++r) {
                            const float diff = Ac[r * AP + s_idx] - MU[r * AMAX + s_idx];
                            acc = fmaf(Rc[r * 8 + 7], diff * diff * inv_var - 1.f, acc);
                        }
                        g_s += acc - a.ent_coef * (float)rows * invB;
                    }
                    ICRL_MARK(14)
                    // ---- dH2pre[r][k] = (sum_d dmean[r][d] * HW[d][k]) * (1 - H2^2) on tensor cores   (K = padded head width)
                    {
                        float acc[2][4];
#pragma unroll
                        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                            for (int c = 0; c < 4; ++c) acc[nt][c] = 0.f;
                        if (AOUT > 8)
                            warp_gemm_3xtf32<2, 16>(acc, DMEAN + 16 * mtf * AMAX, AMAX, 1, HW, WA_LD, 1, 16, 16 * ngf, 8, H, g, t);
                        else
                            warp_gemm_3xtf32<2, 8>(acc, DMEAN + 16 * mtf * AMAX, AMAX, 1, HW, WA_LD, 1, 8, 16 * ngf, 8, H, g, t);
#pragma unroll
                        for (int nt = 0; nt < 2; ++nt) {
                            const float2 ha = *reinterpret_cast<const float2*>(H2 + ojf * LDH + fw_k(nt));
                            const float2 hb = *reinterpret_cast<const float2*>(H2 + (ojf + 8) * LDH + fw_k(nt));
                            *reinterpret_cast<float2*>(DH + ojf * LDH + fw_k(nt)) =
                                make_float2(acc[nt][0] * (1.f - ha.x * ha.x), acc[nt][1] * (1.f - ha.y * ha.y));
                            *reinterpret_cast<float2*>(DH + (ojf + 8) * LDH + fw_k(nt)) =
                                make_float2(acc[nt][2] * (1.f - hb.x * hb.x), acc[nt][3] * (1.f - hb.y * hb.y));
                        }
                    }
                    ICRL_MARK(15)
                    __syncthreads();
                    ICRL_MARK(5)
                    if (SHARED && a.n_shared == 2) share_tile(DH, q);     // dH2pre of the three heads -> their sum
                    if (hd < AOUT) {
                        const float4 v = *reinterpret_cast<const float4*>(PART + hd * LDH + 4 * hk4);
                        g_hw[0] += v.x; g_hw[1] += v.y; g_hw[2] += v.z; g_hw[3] += v.w;
                    }

                    // ---- dW2[j][k] += sum_r dH2pre[r][j] H1[r][k]   (A = dH2pre^T read in place, B = H1)
                    warp_gemm_3xtf32<NTW2, RBH, false, true>(g_w2, DH + 16 * mt, 1, LDH, H1, LDH, 1, RBH, 32 * ng, 8, H, g, t);
                    if (last_chunk) {
#pragma unroll
                        for (int i = 0; i < NTW2; ++i) st4(i, g_w2[i][0], g_w2[i][1], g_w2[i][2], g_w2[i][3]);
                        st4(NTW2 + NT1, g_hw[0], g_hw[1], g_hw[2], g_hw[3]);
                    }
                    if (s_kind == 1) {                                   // db2
                        float acc = 0.f;
#pragma unroll 8
                        for (int r = 0; r < RBH; ++r) acc += DH[r * LDH + s_idx];
                        g_s += acc;
                    }
                    // ---- dH1pre = (dH2pre W2) * (1 - H1^2) -> written over H2      (B[k = j][n = k] = W2[j][k] read in place)
                    {
                        float acc[2][4];
#pragma unroll
                        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                            for (int c = 0; c < 4; ++c) acc[nt][c] = 0.f;
                        warp_gemm_3xtf32<2, H>(acc, DH + 16 * mtf * LDH, LDH, 1, W2, LDH, 1, H, 16 * ngf, 8, H, g, t);
#pragma unroll
                        for (int nt = 0; nt < 2; ++nt) {
                            const float2 ha = *reinterpret_cast<const float2*>(H1 + ojf * LDH + fw_k(nt));
                            const float2 hb = *reinterpret_cast<const float2*>(H1 + (ojf + 8) * LDH + fw_k(nt));
                            *reinterpret_cast<float2*>(H2 + ojf * LDH + fw_k(nt)) =
                                make_float2(acc[nt][0] * (1.f - ha.x * ha.x), acc[nt][1] * (1.f - ha.y * ha.y));
                            *reinterpret_cast<float2*>(H2 + (ojf + 8) * LDH + fw_k(nt)) =
                                make_float2(acc[nt][2] * (1.f - hb.x * hb.x), acc[nt][3] * (1.f - hb.y * hb.y));
                        }
                    }
                    __syncthreads();
                    ICRL_MARK(6)
                    if (SHARED && a.n_shared == 1) share_tile(H2, q);     // dH1pre of the three trunks -> their sum
                    // ---- dW1[j][k] += sum_r dH1pre[r][j] X[r][k] ; db1
                    // every warp group has NT1 n-tiles inside the (zero padded) row when round16(D) == 16 NT1 -- true for all the
                    // named workloads; otherwise the last tile of the second group is skipped by the guarded variant
                    if (((KP + 15) & ~15) == 16 * NT1)
                        warp_gemm_3xtf32<NT1, RBH, false, true>(g_w1, H2 + 16 * mt, 1, LDH, Xc, LDX, 1, RBH, 8 * ng, 16, KP, g, t);
                    else
                        warp_gemm_3xtf32<NT1, RBH, true, true>(g_w1, H2 + 16 * mt, 1, LDH, Xc, LDX, 1, RBH, 8 * ng, 16, KP, g, t);
                    if (s_kind == 0) {
                        float acc = 0.f;
#pragma unroll 8
                        for (int r = 0; r < RBH; ++r) acc += H2[r * LDH + s_idx];
                        g_s += acc;
                    }
                    ICRL_MARK(7)
                }  // chunks
                if (WIDE && len == 0) {
                    // no rows of this minibatch fall to this cluster: it still takes part in every exchange (with zeros)
                    __syncthreads();
                    if (tid == 0) {
                        mbar_expect_tx(&BAR[2], (uint32_t)PAY_BYTES);
                        mbar_expect_tx(&BAR[3], (uint32_t)(NCTA * 8));
                    }
#pragma unroll
                    for (int i = 0; i < NTW2; ++i) st4(i, 0.f, 0.f, 0.f, 0.f);
                    st4(NTW2 + NT1, 0.f, 0.f, 0.f, 0.f);
                }
            }      // working

            // ---- (1) block-reduce the five loss partial sums of this CTA's rows (measured: a variant where only warp 0 totals
            // the per-warp sums -- one barrier, 8 x fewer shared-memory reads -- is no faster: profiles/k4_variants_r02.txt)
            auto block_reduce = [&](float (&r)[6]) {
#pragma unroll
                for (int i = 0; i < 6; ++i) r[i] = warp_sum(r[i]);
                __syncthreads();
                if (lane == 0) {
#pragma unroll
                    for (int i = 0; i < 6; ++i) scratch[warp * 8 + i] = r[i];
                }
                __syncthreads();
#pragma unroll
                for (int i = 0; i < 6; ++i) {
                    float tsum = 0.f;
#pragma unroll
                    for (int wv = 0; wv < NWT; ++wv) tsum += scratch[wv * 8 + i];
                    r[i] = tsum;
                }
            };
            auto local_sumsq = [&]() {
                float q2 = 0.f;
                if (working) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) q2 = fmaf(g_hw[i], g_hw[i], q2);
                    if constexpr (SHARED) {      // a shared layer's gradient counts once: in the pi CTAs' sums
                        if (own_l2) {
#pragma unroll
                            for (int i = 0; i < NTW2; ++i)
#pragma unroll
                                for (int c = 0; c < 4; ++c) q2 = fmaf(g_w2[i][c], g_w2[i][c], q2);
                        }
                        if (own_l1) {
#pragma unroll
                            for (int i = 0; i < NT1; ++i)
#pragma unroll
                                for (int c = 0; c < 4; ++c) q2 = fmaf(g_w1[i][c], g_w1[i][c], q2);
                        }
                        if ((s_kind != 0 || own_l1) && (s_kind != 1 || own_l2)) q2 = fmaf(g_s, g_s, q2);
                    } else {
#pragma unroll
                        for (int i = 0; i < NTW2; ++i)
#pragma unroll
                            for (int c = 0; c < 4; ++c) q2 = fmaf(g_w2[i][c], g_w2[i][c], q2);
#pragma unroll
                        for (int i = 0; i < NT1; ++i)
#pragma unroll
                            for (int c = 0; c < 4; ++c) q2 = fmaf(g_w1[i][c], g_w1[i][c], q2);
                        q2 = fmaf(g_s, g_s, q2);
                    }
                }
                return q2;
            };
            // loss partial sums: every thread carries its own partials through the exchanges (slot-wise sums); the single block
            // reduction after the exchanges totals them together with the gradient norm
            float red[6];

            // ---- (2) CTA-pair exchange through distributed shared memory: every thread stores its gradient fragments and its
            // loss partial sums into the partner's PAY buffer as float4 groups straight from registers (st.async, completing
            // bytes on the partner's mbarrier; the W2 / head groups already left during the backward pass), waits for its own
            // mbarrier and adds.  a + b == b + a in floating point, so both CTAs of a pair end up with bit-identical sums and
            // keep their weight copies identical.   Groups: g_w2[0..NTW2), g_w1[0..NT1), g_hw, {g_s, s0, s1, s2}, {s3, s4, -, -}
            float tot[5];                                                 // loss sums: this warp -> pair -> all ranks
#pragma unroll
            for (int i = 0; i < 5; ++i) tot[i] = (i == 0) ? s_a : (i == 1) ? s_b : (i == 2) ? s_c : (i == 3) ? s_d : s_e;
            if (working) {
                const bool t0 = true;   // every thread sends its slot (non-zero for lane 0 of each warp)
#pragma unroll
                for (int i = 0; i < NT1; ++i) st4(NTW2 + i, g_w1[i][0], g_w1[i][1], g_w1[i][2], g_w1[i][3]);
                st4(NTW2 + NT1 + 1, g_s, t0 ? tot[0] : 0.f, t0 ? tot[1] : 0.f, t0 ? tot[2] : 0.f);
                if ((tid & 7) == 0) st4(NTW2 + NT1 + 2, tot[3], tot[4], 0.f, 0.f);
            }
            // all of the partner's words of this step have landed (bounded: a vanished partner ends the launch with an error)
            if (*(volatile float*)&XCH[31] == 0.f && !mbar_wait_bounded(&BAR[2], (uint32_t)(step & 1), 2000000000LL)) XCH[31] = 1.f;
            if (working) {
                auto ld4 = [&](int v4) { return *reinterpret_cast<const float4*>(PAY + (v4 * NTT + tid) * 4); };
                int v4 = 0;
#pragma unroll
                for (int i = 0; i < NTW2; ++i) {
                    const float4 x = ld4(v4++);
                    g_w2[i][0] += x.x; g_w2[i][1] += x.y; g_w2[i][2] += x.z; g_w2[i][3] += x.w;
                }
#pragma unroll
                for (int i = 0; i < NT1; ++i) {
                    const float4 x = ld4(v4++);
                    g_w1[i][0] += x.x; g_w1[i][1] += x.y; g_w1[i][2] += x.z; g_w1[i][3] += x.w;
                }
                {
                    const float4 x = ld4(v4++);
                    g_hw[0] += x.x; g_hw[1] += x.y; g_hw[2] += x.z; g_hw[3] += x.w;
                }
                {
                    const float4 x = ld4(v4++);
                    g_s += x.x; tot[0] += x.y; tot[1] += x.z; tot[2] += x.w;
                    if ((tid & 7) == 0) {
                        const float4 y = ld4(v4);
                        tot[3] += y.x; tot[4] += y.y;
                    }
                }
                ICRL_MARK(16)
                // ---- (3w) wide mode: sum the pair sums of all clusters (and of all ranks) -- see the kernel's header comment
                bool exchanged = false;
                if constexpr (WIDE) {
                    constexpr int F = NTW2 * 4 + NT1 * 4 + 4 + 1 + 5;       // gradient floats + loss sums owned by a thread
                    auto G = [&](int k) -> float& {                           // k is a compile-time constant at every use
                        if (k < NTW2 * 4) return g_w2[k >> 2][k & 3];
                        k -= NTW2 * 4;
                        if (k < NT1 * 4) return g_w1[k >> 2][k & 3];
                        k -= NT1 * 4;
                        if (k < 4) return g_hw[k];
                        k -= 4;
                        if (k == 0) return g_s;
                        return tot[k - 1];
                    };
                    // grid-wide barrier among the CTAs of this trunk (2 per cluster): arrival counter + acquire spin
                    auto wide_barrier = [&](int which) {
                        __syncthreads();
                        if (tid == 0) {
                            unsigned int* ctr = a.wide_sync + role;
                            const unsigned int target = (unsigned int)(2 * step + which + 1) * (unsigned int)(2 * ncl);
                            __threadfence();
                            atomicAdd(ctr, 1u);
                            if (*(volatile float*)&XCH[31] == 0.f) {
                                const long long t0 = clock64();
                                for (;;) {
                                    unsigned int v;
                                    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
                                    if ((int)(v - target) >= 0) break;
                                    if (clock64() - t0 > 4000000000LL) { XCH[31] = 1.f; break; }   // ~2 s: clusters not co-resident
                                }
                            }
                        }
                        __syncthreads();
                    };
                    const int nred = 2 * ncl;                      // reducers of a trunk: (cluster, half)
                    const int S = (F + nred - 1) / nred;           // floats per reducer (<= WIDE_SMAX, checked by the host)
                    const int rid = cluster_id * 2 + half;
                    if (half == 0) {
                        float* mine = a.wide_part + (((size_t)role * ncl + cluster_id) * F) * NTT + tid;
#pragma unroll
                        for (int k = 0; k < F; ++k) __stcg(mine + (size_t)k * NTT, G(k));
                    }
                    wide_barrier(0);
                    {
                        float rs[WIDE_SMAX];
                        const float* pbase = a.wide_part + ((size_t)role * ncl * F) * NTT + tid;
                        // (latency bound: 4 clusters x S floats = up to 24 independent L2 loads in flight per round trip instead
                        //  of 8 -- the reduction was ~10 k cycles per step, 10 % of the samples of a 1 M-row launch)
#pragma unroll
                        for (int kk = 0; kk < WIDE_SMAX; ++kk) rs[kk] = 0.f;
                        for (int c0 = 0; c0 < ncl; c0 += 4) {
                            float v[4][WIDE_SMAX];
#pragma unroll
                            for (int cc = 0; cc < 4; ++cc)
#pragma unroll
                                for (int kk = 0; kk < WIDE_SMAX; ++kk) {
                                    const int k = rid * S + kk;
                                    v[cc][kk] = (c0 + cc < ncl && kk < S && k < F) ? __ldcg(pbase + ((size_t)(c0 + cc) * F + k) * NTT) : 0.f;
                                }
#pragma unroll
                            for (int cc = 0; cc < 4; ++cc)          // cluster order per float: identical bits on every replica
#pragma unroll
                                for (int kk = 0; kk < WIDE_SMAX; ++kk) rs[kk] += v[cc][kk];
                        }
                        if (DIST && a.world > 1) {
                            // data parallel: the same reducer of every rank holds the same slice -> one-hop exchange of
                            // {f0, f1, f2, seq ^ hash} words over NVLink peer memory, summed in rank order
                            const unsigned int want = a.flag_base + (unsigned int)step + 1u;
                            auto tag = [&](unsigned int x, unsigned int y, unsigned int z) {
                                return want ^ ((x ^ __funnelshift_l(y, y, 11) ^ __funnelshift_l(z, z, 22)) * 0x9E3779B1u);
                            };
                            auto slab = [&](float* base, int src) {
                                return reinterpret_cast<uint4*>(base) +
                                       ((((size_t)parity * ICRL_PPO_MAX_RANKS + src) * WIDE_MAXCTA + (cluster_id * NCTA + crank)) * 2) * NTT + tid;
                            };
                            const int nw = S > 3 ? 2 : 1;
                            for (int pr = 0; pr < a.world; ++pr) {
                                uint4* dst = slab(a.recv[pr], a.rank);
                                const unsigned int x0 = __float_as_uint(rs[0]), x1 = __float_as_uint(rs[1]), x2 = __float_as_uint(rs[2]);
                                dst[0] = make_uint4(x0, x1, x2, tag(x0, x1, x2));
                                if (nw > 1) {
                                    const unsigned int y0 = __float_as_uint(rs[3]), y1 = __float_as_uint(rs[4]), y2 = __float_as_uint(rs[5]);
                                    dst[NTT] = make_uint4(y0, y1, y2, tag(y0, y1, y2));
                                }
                            }
                            // ranks are polled one after the other (two words in flight): a few NVLink round trips per step are
                            // noise next to a wide step, and the big polling arrays of the single-cluster schemes would cost
                            // registers in the chunk loop
#pragma unroll
                            for (int kk = 0; kk < WIDE_SMAX; ++kk) rs[kk] = 0.f;
                            const long long tstart = clock64();
                            for (int src_rank = 0; src_rank < a.world; ++src_rank) {          // rank order: identical bits everywhere
                                const uint4* src = slab(a.recv[a.rank], src_rank);
                                uint4 x0, x1 = make_uint4(0u, 0u, 0u, 0u);
                                for (;;) {
                                    asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];"
                                                 : "=r"(x0.x), "=r"(x0.y), "=r"(x0.z), "=r"(x0.w) : "l"(src) : "memory");
                                    bool ok = (x0.w == tag(x0.x, x0.y, x0.z));
                                    if (nw > 1) {
                                        asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];"
                                                     : "=r"(x1.x), "=r"(x1.y), "=r"(x1.z), "=r"(x1.w) : "l"(src + NTT) : "memory");
                                        ok = ok && (x1.w == tag(x1.x, x1.y, x1.z));
                                    }
                                    if (ok) break;
                                    if (clock64() - tstart > 4000000000LL) { XCH[31] = 1.f; break; }   // ~2 s: a peer is gone
                                }
                                rs[0] += __uint_as_float(x0.x); rs[1] += __uint_as_float(x0.y); rs[2] += __uint_as_float(x0.z);
                                rs[3] += __uint_as_float(x1.x); rs[4] += __uint_as_float(x1.y); rs[5] += __uint_as_float(x1.z);
                            }
                        }
                        float* red = a.wide_red + ((size_t)role * F) * NTT + tid;
#pragma unroll
                        for (int kk = 0; kk < WIDE_SMAX; ++kk) {
                            const int k = rid * S + kk;
                            if (kk < S && k < F) __stcg(red + (size_t)k * NTT, rs[kk]);
                        }
                    }
                    wide_barrier(1);
                    {
                        const float* red = a.wide_red + ((size_t)role * F) * NTT + tid;
#pragma unroll
                        for (int k = 0; k < F; ++k) G(k) = __ldcg(red + (size_t)k * NTT);
                    }
                    exchanged = true;
                }
                // ---- (3) data parallel: all-reduce the pair sums across the ranks' matching CTAs over NVLink peer memory
                if (!WIDE && DIST && a.world > 1) {
                    // ---- (3a) 4 / 8 ranks: reduce-scatter + all-gather, both with self-validating words.
                    // The direct scheme below makes every thread read W full gradient copies one after the other (W x 2
                    // dependent L2 round trips, which is what made the exchange cost grow linearly with W).  Here the
                    // F floats a thread owns are cut into W slices; rank q sums slice q of every rank IN RANK ORDER (so all
                    // replicas see the same bits), then broadcasts the sum.  Per thread: W*NWD words in, W*NWD words out,
                    // each phase polled in one or two batches -> two NVLink hops, cost independent of W.  A word is
                    // {f0, f1, f2, seq ^ hash(f0, f1, f2)}: three payload floats ride with one self-validating tag, and a
                    // torn 16-byte store cannot pass for a whole one.  The two CTAs of
                    // a pair hold identical sums: half h sends only to the ranks of parity h, both poll the same slabs.
                    const unsigned int want = a.flag_base + (unsigned int)step + 1u;
                    constexpr int F = NTW2 * 4 + NT1 * 4 + 4 + 1 + 5;       // gradient floats + loss sums owned by a thread
                    auto G = [&](int k) -> float& {                           // k is a compile-time constant at every use
                        if (k < NTW2 * 4) return g_w2[k >> 2][k & 3];
                        k -= NTW2 * 4;
                        if (k < NT1 * 4) return g_w1[k >> 2][k & 3];
                        k -= NT1 * 4;
                        if (k < 4) return g_hw[k];
                        k -= 4;
                        if (k == 0) return g_s;
                        return tot[k - 1];
                    };
                    auto rsag = [&](auto wc) {
                        constexpr int W = decltype(wc)::value;
                        constexpr int S = (F + W - 1) / W;                  // floats per slice
                        constexpr int NWD = (S + 2) / 3;                    // words per slice
                        static_assert(NWD <= RSAG_MAXW, "RS/AG slab too small");
                        const int me = a.rank;
                        auto slab = [&](float* base, int region, int src) {
                            return reinterpret_cast<uint4*>(base) +
                                   ((((size_t)(region * 2 + parity) * ICRL_PPO_MAX_RANKS + src) * 3 + role) * RSAG_MAXW) * NTT + tid;
                        };
                        // the fourth lane is the sequence number XOR a hash of the payload: a word that arrived torn (old and
                        // new 8-byte halves mixed) fails the check unless the mixed-in old half equals the new one anyway
                        auto tag = [&](unsigned int x, unsigned int y, unsigned int z) {
                            return want ^ ((x ^ __funnelshift_l(y, y, 11) ^ __funnelshift_l(z, z, 22)) * 0x9E3779B1u);
                        };
                        auto put = [&](uint4* dst, int j, float x, float y, float z) {
                            const unsigned int xi = __float_as_uint(x), yi = __float_as_uint(y), zi = __float_as_uint(z);
                            dst[j * NTT] = make_uint4(xi, yi, zi, tag(xi, yi, zi));
                        };
                        // polls NW words (word w -> slab(region, w / NWD) + (w % NWD) * NTT), 16 per round trip, and hands
                        // each validated word to `sink(w, x, y, z)`
                        const long long tstart = clock64();
                        auto poll = [&](int region, auto sink) {
                            constexpr int NW = W * NWD;
#pragma unroll
                            for (int w0 = 0; w0 < NW; w0 += 16) {
                                uint4 x[16];
                                for (;;) {
                                    bool ok = true;
#pragma unroll
                                    for (int j = 0; j < 16; ++j)
                                        if (w0 + j < NW) {
                                            const uint4* src = slab(a.recv[me], region, (w0 + j) / NWD) + ((w0 + j) % NWD) * NTT;
                                            asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];"
                                                         : "=r"(x[j].x), "=r"(x[j].y), "=r"(x[j].z), "=r"(x[j].w)
                                                         : "l"(src) : "memory");
                                        }
#pragma unroll
                                    for (int j = 0; j < 16; ++j)
                                        if (w0 + j < NW) ok = ok && (x[j].w == tag(x[j].x, x[j].y, x[j].z));
                                    if (ok) break;
                                    if (clock64() - tstart > 4000000000LL) { XCH[31] = 1.f; break; }   // ~2 s: a peer is gone
                                }
#pragma unroll
                                for (int j = 0; j < 16; ++j)
                                    if (w0 + j < NW)
                                        sink(w0 + j, __uint_as_float(x[j].x), __uint_as_float(x[j].y), __uint_as_float(x[j].z));
                            }
                        };
                        // reduce-scatter: slice q of my floats -> rank q
#pragma unroll
                        for (int q = 0; q < W; ++q) {
                            if ((q & 1) != half) continue;
                            uint4* dst = slab(a.recv[q], 0, me);
#pragma unroll
                            for (int j = 0; j < NWD; ++j) {
                                const int k = q * S + 3 * j;
                                put(dst, j, (3 * j < S && k < F) ? G(k) : 0.f, (3 * j + 1 < S && k + 1 < F) ? G(k + 1) : 0.f,
                                    (3 * j + 2 < S && k + 2 < F) ? G(k + 2) : 0.f);
                            }
                        }
                        float red[S];
#pragma unroll
                        for (int i = 0; i < S; ++i) red[i] = 0.f;
                        poll(0, [&](int w, float x, float y, float z) {       // w ascending == rank ascending per element
                            const int i = 3 * (w % NWD);
                            if (i < S) red[i] += x;
                            if (i + 1 < S) red[i + 1] += y;
                            if (i + 2 < S) red[i + 2] += z;
                        });
                        // all-gather: my reduced slice -> every rank
#pragma unroll
                        for (int pr = 0; pr < W; ++pr) {
                            if ((pr & 1) != half) continue;
                            uint4* dst = slab(a.recv[pr], 1, me);
#pragma unroll
                            for (int j = 0; j < NWD; ++j)
                                put(dst, j, (3 * j < S) ? red[3 * j] : 0.f, (3 * j + 1 < S) ? red[3 * j + 1] : 0.f,
                                    (3 * j + 2 < S) ? red[3 * j + 2] : 0.f);
                        }
                        poll(1, [&](int w, float x, float y, float z) {
                            const int q = w / NWD, i = 3 * (w % NWD), k = q * S + i;
                            if (i < S && k < F) G(k) = x;
                            if (i + 1 < S && k + 1 < F) G(k + 1) = y;
                            if (i + 2 < S && k + 2 < F) G(k + 2) = z;
                        });
                    };
                    // ---- (3a') 2 and 4 ranks: one hop.  Every rank broadcasts its full gradient as tagged 3-float words (the two CTAs of
                    // a pair send alternate words, both read everything) and each thread adds the W copies in rank order:
                    // W * ceil(F / 3) words polled 16 at a time -- 24 words = two round trips for HalfCheetah, against four with
                    // the {value, seq, value, seq} words of (3b).
                    auto bcast_sum = [&](auto wc) {
                        constexpr int W = decltype(wc)::value;
                        constexpr int NWD = (F + 2) / 3;
                        static_assert(NWD <= RSAG_MAXW, "slab too small");
                        const int me = a.rank;
                        auto slab = [&](float* base, int src) {
                            return reinterpret_cast<uint4*>(base) +
                                   ((((size_t)(2 * 2 + parity) * ICRL_PPO_MAX_RANKS + src) * 3 + role) * RSAG_MAXW) * NTT + tid;
                        };
                        auto tag = [&](unsigned int x, unsigned int y, unsigned int z) {
                            return want ^ ((x ^ __funnelshift_l(y, y, 11) ^ __funnelshift_l(z, z, 22)) * 0x9E3779B1u);
                        };
                        // The own contribution never travels through global memory (narrow dW1 tiles, or two ranks): nothing is
                        // stored to or polled from the own slab, which cuts the bytes every polling round pulls through L2 (the
                        // rounds are bandwidth bound: 256 threads x words x 16 B per CTA) and the peer stores (~30 B / cycle per
                        // SM: 825 cycles for HalfCheetah's 24 KB per peer) by 1 / W.  Two ranks: it simply stays in the
                        // registers (a + b == b + a bit for bit, both ranks form the same sum).  More ranks: it is parked in the
                        // (idle) pair-exchange buffer and added when the rank-ordered sum reaches this rank's position, so every
                        // replica still adds the W contributions in rank order.
                        // (the wide dW1 tiles of NT1 > 2 have no registers to spare for that: own words go through the own slab.
                        //  Measured and rejected: staging the words in shared memory and sending them as 4 KB TMA bulk stores,
                        //  shared -> peer global -- send 1153 cycles against 825, profiles/dp2_timing_r02.txt)
                        constexpr bool SKIP = (W == 2) || (NT1 <= 2);
                        constexpr bool PARK = SKIP && (W > 2);
                        float* own = PAY + tid;                       // own[k * NTT]: conflict-free, thread private
#pragma unroll
                        for (int pr = 0; pr < W; ++pr) {
                            if (SKIP && pr == me) continue;
                            uint4* dst = slab(a.recv[pr], me);
#pragma unroll
                            for (int j = 0; j < NWD; ++j) {
                                if ((j & 1) != half) continue;
                                const unsigned int xi = __float_as_uint(3 * j < F ? G(3 * j) : 0.f),
                                                   yi = __float_as_uint(3 * j + 1 < F ? G(3 * j + 1) : 0.f),
                                                   zi = __float_as_uint(3 * j + 2 < F ? G(3 * j + 2) : 0.f);
                                dst[j * NTT] = make_uint4(xi, yi, zi, tag(xi, yi, zi));
                            }
                        }
                        if (PARK) {
#pragma unroll
                            for (int k = 0; k < F; ++k) { own[k * NTT] = G(k); G(k) = 0.f; }
                        } else if (!SKIP) {
#pragma unroll
                            for (int k = 0; k < F; ++k) G(k) = 0.f;
                        }
                        ICRL_MARK(17)
                        const long long tstart = clock64();
                        constexpr int NW = (SKIP ? W - 1 : W) * NWD;   // words of the (remote) ranks, ascending rank
                        // PW words in flight per polling round trip: every round after the first costs one more L2 round trip
                        constexpr int PW = NT1 >= 8 ? 16 : (NW <= 26) ? NW : ((NW + 1) / 2 <= 26 ? (NW + 1) / 2 : 16);   // (wide dW1 tiles: no registers to spare)
                        auto add_own = [&]() {
#pragma unroll
                            for (int k = 0; k < F; ++k) G(k) += own[k * NTT];
                        };
#pragma unroll
                        for (int w0 = 0; w0 < NW; w0 += PW) {
                            uint4 x[PW];
                            for (;;) {
                                bool ok = true;
#pragma unroll
                                for (int j = 0; j < PW; ++j)
                                    if (w0 + j < NW) {
                                        const int ri = (w0 + j) / NWD, src_rank = ri + ((SKIP && ri >= me) ? 1 : 0);
                                        const uint4* src = slab(a.recv[me], src_rank) + ((w0 + j) % NWD) * NTT;
                                        asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];"
                                                     : "=r"(x[j].x), "=r"(x[j].y), "=r"(x[j].z), "=r"(x[j].w)
                                                     : "l"(src) : "memory");
                                    }
#pragma unroll
                                for (int j = 0; j < PW; ++j)
                                    if (w0 + j < NW) ok = ok && (x[j].w == tag(x[j].x, x[j].y, x[j].z));
                                if (ok) break;
                                if (clock64() - tstart > 4000000000LL) { XCH[31] = 1.f; break; }   // ~2 s: a peer is gone
                            }
#pragma unroll
                            for (int j = 0; j < PW; ++j) {
                                if (w0 + j < NW) {
                                    // remote rank index ri stands for rank ri + (ri >= me): the own gradient goes in right before
                                    // the first word of remote index `me` (== rank me + 1)
                                    if (PARK && (w0 + j) % NWD == 0 && (w0 + j) / NWD == me) add_own();
                                    const int k = 3 * ((w0 + j) % NWD);
                                    if (k < F) G(k) += __uint_as_float(x[j].x);
                                    if (k + 1 < F) G(k + 1) += __uint_as_float(x[j].y);
                                    if (k + 2 < F) G(k + 2) += __uint_as_float(x[j].z);
                                }
                            }
                        }
                        if (PARK && me == W - 1) add_own();
                    };
                    // auto: broadcast + sum for 2 and 4 ranks (measured at 4 ranks: 434 vs 442 ms per iteration against RS/AG),
                    // reduce-scatter + all-gather for 8 (the broadcast would need six polling rounds there)
                    const bool want_bcast = a.dist_mode == 3 || (a.dist_mode == 0 && a.world <= 4);
                    if (want_bcast && a.world == 2) { bcast_sum(std::integral_constant<int, 2>{}); exchanged = true; }
                    else if (want_bcast && a.world == 4) { bcast_sum(std::integral_constant<int, 4>{}); exchanged = true; }
                    const bool want_rsag = a.dist_mode == 2 || (a.dist_mode == 0 && a.world >= 4);
                    if (exchanged) {}
                    else if (want_rsag && a.world == 8) { rsag(std::integral_constant<int, 8>{}); exchanged = true; }
                    else if (want_rsag && a.world == 4) { rsag(std::integral_constant<int, 4>{}); exchanged = true; }
                    else if (want_rsag && a.world == 2) { rsag(std::integral_constant<int, 2>{}); exchanged = true; }
                }
                if (!WIDE && DIST && a.world > 1 && !exchanged) {
                    // ---- (3b) any other world size: direct exchange.  "LL" protocol (as NCCL's low-latency path): every 16-byte store carries two values and two copies of
                    // this step's sequence number, so the data validates itself -- no fence, no separate flag, no barrier:
                    // the exchange costs one NVLink store latency.  (A torn 16-byte store is still two self-validating
                    // 8-byte halves.)  Buffers alternate by step parity and the sequence number grows monotonically, so a
                    // stale slot can never match.  Every rank also stores into its OWN slab and then sums all slabs in
                    // rank order from memory: identical order everywhere -> bit-identical replicated updates.
                    static_assert(NP <= DIST_SLOTS, "receive-buffer slab too small");
                    const unsigned int want = a.flag_base + (unsigned int)step + 1u;
                    const size_t slab16 = ((size_t)(parity * ICRL_PPO_MAX_RANKS + a.rank) * NCTA + crank) * (DIST_SLOTS / 2) * NTT;
                    const bool t0 = true;
                    for (int p = 0; p < a.world; ++p) {
                        uint4* dst = reinterpret_cast<uint4*>(a.recv[p]) + slab16 + tid;
                        auto put4 = [&](int v4, float x, float y, float z, float w) {
                            dst[(2 * v4) * NTT] = make_uint4(__float_as_uint(x), want, __float_as_uint(y), want);
                            dst[(2 * v4 + 1) * NTT] = make_uint4(__float_as_uint(z), want, __float_as_uint(w), want);
                        };
                        int v4 = 0;
#pragma unroll
                        for (int i = 0; i < NTW2; ++i) put4(v4++, g_w2[i][0], g_w2[i][1], g_w2[i][2], g_w2[i][3]);
#pragma unroll
                        for (int i = 0; i < NT1; ++i) put4(v4++, g_w1[i][0], g_w1[i][1], g_w1[i][2], g_w1[i][3]);
                        put4(v4++, g_hw[0], g_hw[1], g_hw[2], g_hw[3]);
                        put4(v4++, g_s, t0 ? tot[0] : 0.f, t0 ? tot[1] : 0.f, t0 ? tot[2] : 0.f);
                        put4(v4++, t0 ? tot[3] : 0.f, t0 ? tot[4] : 0.f, 0.f, 0.f);
                    }
#pragma unroll
                    for (int i = 0; i < NTW2; ++i)
#pragma unroll
                        for (int c = 0; c < 4; ++c) g_w2[i][c] = 0.f;
#pragma unroll
                    for (int i = 0; i < NT1; ++i)
#pragma unroll
                        for (int c = 0; c < 4; ++c) g_w1[i][c] = 0.f;
#pragma unroll
                    for (int i = 0; i < 4; ++i) g_hw[i] = 0.f;
                    g_s = 0.f;
#pragma unroll
                    for (int i = 0; i < 5; ++i) tot[i] = 0.f;
                    const long long tstart = clock64();
                    for (int r = 0; r < a.world; ++r) {
                        const uint4* src = reinterpret_cast<const uint4*>(a.recv[a.rank]) +
                                           ((size_t)(parity * ICRL_PPO_MAX_RANKS + r) * NCTA + crank) * (DIST_SLOTS / 2) * NTT + tid;
                        // 8 float4 groups (16 sixteen-byte words) in flight per polling round trip
                        auto get4x4 = [&](int v4, float4 (&o)[8], int n) {
                            uint4 x[16];
                            for (;;) {
                                bool ok = true;
#pragma unroll
                                for (int j = 0; j < 16; ++j)
                                    if (j < 2 * n)
                                        asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];"
                                                     : "=r"(x[j].x), "=r"(x[j].y), "=r"(x[j].z), "=r"(x[j].w)
                                                     : "l"(src + (2 * v4 + j) * NTT) : "memory");
#pragma unroll
                                for (int j = 0; j < 16; ++j)
                                    if (j < 2 * n) ok = ok && (x[j].y == want) && (x[j].w == want);
                                if (ok) break;
                                if (clock64() - tstart > 4000000000LL) { XCH[31] = 1.f; break; }   // ~2 s: a peer is gone
                            }
#pragma unroll
                            for (int j = 0; j < 8; ++j)
                                if (j < n)
                                    o[j] = make_float4(__uint_as_float(x[2 * j].x), __uint_as_float(x[2 * j].z),
                                                       __uint_as_float(x[2 * j + 1].x), __uint_as_float(x[2 * j + 1].z));
                        };
                        constexpr int NG = NTW2 + NT1 + 3;       // float4 groups
                        // walk the groups 4 at a time; the group -> register mapping is resolved at compile time
#pragma unroll
                        for (int g0 = 0; g0 < NG; g0 += 8) {
                            float4 o[8];
                            get4x4(g0, o, (NG - g0) < 8 ? (NG - g0) : 8);
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const int gi = g0 + j;
                                if (gi < NTW2) {
                                    g_w2[gi][0] += o[j].x; g_w2[gi][1] += o[j].y; g_w2[gi][2] += o[j].z; g_w2[gi][3] += o[j].w;
                                } else if (gi < NTW2 + NT1) {
                                    g_w1[gi - NTW2][0] += o[j].x; g_w1[gi - NTW2][1] += o[j].y;
                                    g_w1[gi - NTW2][2] += o[j].z; g_w1[gi - NTW2][3] += o[j].w;
                                } else if (gi == NTW2 + NT1) {
                                    g_hw[0] += o[j].x; g_hw[1] += o[j].y; g_hw[2] += o[j].z; g_hw[3] += o[j].w;
                                } else if (gi == NTW2 + NT1 + 1) {
                                    g_s += o[j].x; tot[0] += o[j].y; tot[1] += o[j].z; tot[2] += o[j].w;
                                } else if (gi == NTW2 + NT1 + 2) {
                                    tot[3] += o[j].x; tot[4] += o[j].y;
                                }
                            }
                        }
                    }
                }
            }
            ICRL_MARK(18)
            // ---- (4) norm of the reduced gradient (block reduction; also publishes the loss totals from scratch[120..124])
            {
                float r2[6] = {tot[0], tot[1], tot[2], tot[3], tot[4], local_sumsq()};
                block_reduce(r2);
#pragma unroll
                for (int i = 0; i < 6; ++i) red[i] = r2[i];
            }
            const float ss = red[5];
            const size_t so = (size_t)step * ICRL_PPO_STATS_PER_STEP;
            float kl_step = 0.f;
            if (role == 0 && working) {
                float pl = -(red[0] * invB);
                pl = pl + nu * (red[1] * invB);
                pl = pl / (1.f + nu);
                kl_step = red[3] * invB;
                if (tid == 0 && half == 0 && cluster_id == 0) {
                    a.stats[so + 0] = pl;
                    a.stats[so + 1] = red[2] * invB;
                    a.stats[so + 4] = -(red[4] * invB);
                    a.stats[so + 5] = kl_step;
                }
            } else if (working) {
                if (tid == 0 && half == 0 && cluster_id == 0) a.stats[so + (role == 1 ? 2 : 3)] = red[0] * invB;
            }
            ICRL_MARK(8)

            // ---- global gradient norm: every CTA publishes its trunk's sum of squares through DSMEM (st.async -> norm mbarrier)
            // epoch-level KL early stop is decided by the pi CTAs right here (they have this step's KL) and rides along
            float stop_flag = 0.f;
            if (role == 0 && working) {
                epoch_kl_sum += (double)kl_step;
                ++epoch_steps;
                const bool last_of_epoch = (mb == a.steps_per_epoch - 1);
                if (last_of_epoch && a.has_target_kl && (epoch_kl_sum / epoch_steps) > 1.5 * a.target_kl) stop_flag = 1.f;
                if (a.max_steps > 0 && (WIDE ? a.epoch_base * a.steps_per_epoch : 0) + step + 1 >= a.max_steps) stop_flag = 2.f;
            }
            if (tid < ncta && working) {
                uint32_t ra, rb;
                asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(smem_u32(XCH + (parity * 8 + crank) * 2)), "r"((uint32_t)tid));
                asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rb) : "r"(smem_u32(&BAR[3])), "r"((uint32_t)tid));
                asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f32 [%0], {%1, %2}, [%3];" ::"r"(ra),
                             "f"(ss), "f"(stop_flag), "r"(rb) : "memory");
            }
            // every CTA waits for the words of ALL six CTAs (it uses the even ranks' values): no CTA can run a step ahead of
            // a peer that is still reading this step's exchange buffers
            if (*(volatile float*)&XCH[31] == 0.f && !mbar_wait_bounded(&BAR[3], (uint32_t)(step & 1), 2000000000LL)) XCH[31] = 1.f;
            ICRL_MARK(9)
            const float total_ss = XCH[(parity * 8 + 0) * 2] + XCH[(parity * 8 + 2) * 2] + XCH[(parity * 8 + 4) * 2];
            const float stop_rx = XCH[(parity * 8 + 0) * 2 + 1];
            const float total_norm = sqrtf(total_ss);
            const float clip_coef = fminf(a.max_grad_norm / (total_norm + 1e-6f), 1.0f);
            if (crank == 0 && tid == 0 && cluster_id == 0) {
                a.stats[so + 7] = total_norm;
                a.stats[so + 6] = 0.f;   // total loss is assembled on the host from the parts (needs all three CTAs)
            }

            // ---- Adam (each thread updates the parameters it owns; the shared-memory weights are refreshed in place)
            if (working) {
                AdamConsts ac;
                ac.one_minus_b1 = (float)(1.0 - a.beta1);
                ac.b2 = (float)a.beta2;
                ac.one_minus_b2 = (float)(1.0 - a.beta2);
                ac.inv_bc2_sqrt = adam_inv_bc2_sqrt;
                ac.eps = (float)a.adam_eps;
                ac.neg_step_size = adam_neg_step;
                // padding entries of this CTA's trunk (j >= its h1, k >= its h0 / D) keep g = m = v = 0 and therefore stay
                // exactly 0: their weights and biases are 0, so tanh(0) = 0 and every gradient into them is a product with 0
#pragma unroll
                for (int nt = 0; nt < NTW2; ++nt) {
                    float2* pa = reinterpret_cast<float2*>(W2 + oj * LDH + w2_k(nt));
                    float2* pb = reinterpret_cast<float2*>(W2 + (oj + 8) * LDH + w2_k(nt));
                    const float2 wa = *pa, wb = *pb;
                    *pa = make_float2(adam_update(wa.x, g_w2[nt][0] * clip_coef, m_w2[nt][0], v_w2[nt][0], ac),
                                      adam_update(wa.y, g_w2[nt][1] * clip_coef, m_w2[nt][1], v_w2[nt][1], ac));
                    *pb = make_float2(adam_update(wb.x, g_w2[nt][2] * clip_coef, m_w2[nt][2], v_w2[nt][2], ac),
                                      adam_update(wb.y, g_w2[nt][3] * clip_coef, m_w2[nt][3], v_w2[nt][3], ac));
                }
#pragma unroll
                for (int i = 0; i < NT1; ++i) {
                    if (w1_k(i) < KP) {
                        float2* pa = reinterpret_cast<float2*>(W1 + oj * LDX + w1_k(i));
                        float2* pb = reinterpret_cast<float2*>(W1 + (oj + 8) * LDX + w1_k(i));
                        const float2 wa = *pa, wb = *pb;
                        *pa = make_float2(adam_update(wa.x, g_w1[i][0] * clip_coef, m_w1[i][0], v_w1[i][0], ac),
                                          adam_update(wa.y, g_w1[i][1] * clip_coef, m_w1[i][1], v_w1[i][1], ac));
                        *pb = make_float2(adam_update(wb.x, g_w1[i][2] * clip_coef, m_w1[i][2], v_w1[i][2], ac),
                                          adam_update(wb.y, g_w1[i][3] * clip_coef, m_w1[i][3], v_w1[i][3], ac));
                    }
                }
                if (hd < AOUT) {
                    float4* wp = reinterpret_cast<float4*>(HW + hd * WA_LD + 4 * hk4);
                    const float4 w4 = *wp;
                    *wp = make_float4(adam_update(w4.x, g_hw[0] * clip_coef, m_hw[0], v_hw[0], ac),
                                      adam_update(w4.y, g_hw[1] * clip_coef, m_hw[1], v_hw[1], ac),
                                      adam_update(w4.z, g_hw[2] * clip_coef, m_hw[2], v_hw[2], ac),
                                      adam_update(w4.w, g_hw[3] * clip_coef, m_hw[3], v_hw[3], ac));
                }
                if (s_kind >= 0 && flat_scalar() >= 0) {
                    float* slot = s_kind == 0 ? &B1[s_idx] : s_kind == 1 ? &B2[s_idx] : s_kind == 2 ? &HB[s_idx] : &LOGSTD[s_idx];
                    const float pnew = adam_update(*slot, g_s * clip_coef, m_s, v_s, ac);
                    *slot = pnew;
                    if (s_kind == 3) {
                        const float sigma = expf(pnew);
                        SIG[s_idx] = 1.f / (sigma * sigma);
                        SIG[AMAX + s_idx] = logf(sigma);
                    }
                }
            }
            ICRL_MARK(10)
            if (stop_rx == 1.f) { early_stop_epoch = (WIDE ? a.epoch_base : 0) + epoch; stop_all = true; kl_stopped = true; }
            if (stop_rx == 2.f) { stop_all = true; }
            // (the next chunk's leading __syncthreads orders these shared-memory weight updates before their first use)
        }  // minibatches
    }      // epochs
    if (working && cur_valid(cur)) mbar_wait(&BAR[q & 1], (uint32_t)((q >> 1) & 1));   // drain the in-flight prefetch
    __syncthreads();
    if (timed) {
        for (int i = 0; i < 20; ++i) a.timing[crank * 20 + i] = tacc[i];
    }
#undef ICRL_MARK

    // ---- write back parameters and moments (owner threads of the first CTA of each pair; the second holds identical copies)
    if (working && half == 0 && cluster_id == 0) {
#pragma unroll
        for (int nt = 0; nt < NTW2; ++nt)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int j = frag_j(c), k = w2_k(nt) + frag_dk(c), f = (SHARED && !own_l2) ? -1 : flat_w2(j, k);
                if (f >= 0) { a.params[f] = W2[j * LDH + k]; a.adam_m[f] = m_w2[nt][c]; a.adam_v[f] = v_w2[nt][c]; }
            }
#pragma unroll
        for (int i = 0; i < NT1; ++i)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int j = frag_j(c), k = w1_k(i) + frag_dk(c), f = (SHARED && !own_l1) ? -1 : flat_w1(j, k);
                if (f >= 0) { a.params[f] = W1[j * LDX + k]; a.adam_m[f] = m_w1[i][c]; a.adam_v[f] = v_w1[i][c]; }
            }
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            const int f = flat_hw(hd, 4 * hk4 + kk);
            if (f >= 0) { a.params[f] = HW[hd * WA_LD + 4 * hk4 + kk]; a.adam_m[f] = m_hw[kk]; a.adam_v[f] = v_hw[kk]; }
        }
        const int f = (SHARED && ((s_kind == 0 && !own_l1) || (s_kind == 1 && !own_l2))) ? -1 : flat_scalar();
        if (f >= 0) {
            const float* slot = s_kind == 0 ? &B1[s_idx] : s_kind == 1 ? &B2[s_idx] : s_kind == 2 ? &HB[s_idx] : &LOGSTD[s_idx];
            a.params[f] = *slot; a.adam_m[f] = m_s; a.adam_v[f] = v_s;
        }
    }
    if (crank == 0 && tid == 0 && cluster_id == 0) {
        if (WIDE) {        // one launch per epoch: the host presets result[0] = n_epochs, the steps accumulate over the launches
            if (stop_all) { a.result[3] = 1; if (kl_stopped) a.result[0] = early_stop_epoch; }
            a.result[1] = a.result[1] + step;
        } else {
            a.result[0] = early_stop_epoch;
            a.result[1] = step;
        }
    }
    // an exchange wait of ANY CTA hit its bound (lost cluster peer / data-parallel rank): the host zeroes result[2] before the
    // launch and raises when it comes back set (the parameters of such a launch are not valid)
    if (tid == 0 && *(volatile float*)&XCH[31] != 0.f) a.result[2] = 1;
    cluster_sync_all();   // nobody exits while a peer may still address its shared memory
}

// ---------------------------------------------------------------- host side

template <int NT1, bool WIDE>
static int launch_cfg(const PpoArgs& a, cudaStream_t st, int n_clusters, cudaLaunchConfig_t* cfg, cudaLaunchAttribute* attr,
                      void (**kern_out)(const PpoArgs)) {
    void (*kern)(const PpoArgs);
    if (a.timing != nullptr)
        kern = WIDE ? (a.world > 1 ? ppo_train_kernel<NT1, true, true, true> : ppo_train_kernel<NT1, false, true, true>)
                    : (a.world > 1 ? ppo_train_kernel<NT1, true, false, true> : ppo_train_kernel<NT1, false, false, true>);
    else
        kern = WIDE ? (a.world > 1 ? ppo_train_kernel<NT1, true, true, false> : ppo_train_kernel<NT1, false, true, false>)
                    : (a.world > 1 ? ppo_train_kernel<NT1, true, false, false> : ppo_train_kernel<NT1, false, false, false>);
    // shared trunk layers: separate instantiations, so the kernels of separate trunks stay as they are (single GPU, no
    // phase timing: the host refuses world > 1 and does not ask for timing with n_shared > 0)
    if (a.n_shared > 0)
        kern = WIDE ? ppo_train_kernel<NT1, false, true, false, true> : ppo_train_kernel<NT1, false, false, false, true>;
    const PpoSmem L = ppo_smem_layout(a.DP, ppo_pay_floats<NT1>(), a.n_shared > 0);
    if (L.total_bytes > 227 * 1024) {
        set_error("obs_dim %d needs %d bytes of shared memory (> 227 KB)", a.D, L.total_bytes);
        return ICRL_EUNSUPPORTED;
    }
    ICRL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total_bytes));
    *cfg = cudaLaunchConfig_t{};
    cfg->gridDim = dim3(NCTA * n_clusters);
    cfg->blockDim = dim3(NTT);
    cfg->dynamicSmemBytes = L.total_bytes;
    cfg->stream = st;
    attr[0].id = cudaLaunchAttributeClusterDimension;      // clusters of 6 CTAs: a CTA pair per trunk (pi, vf, cvf)
    attr[0].val.clusterDim.x = NCTA;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg->attrs = attr;
    cfg->numAttrs = 1;
    *kern_out = kern;
    return 0;
}

template <int NT1>
static int launch_ppo(const PpoArgs& a, cudaStream_t st) {
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr[1];
    void (*kern)(const PpoArgs);
    if (int rc = launch_cfg<NT1, false>(a, st, 1, &cfg, attr, &kern)) return rc;
    const cudaError_t err = cudaLaunchKernelEx(&cfg, kern, a);
    if (err != cudaSuccess) {
        set_error("ppo_train_kernel launch failed: %s", cudaGetErrorString(err));
        return (int)err;
    }
    count_launch();
    return 0;
}

// how many 6-CTA clusters of the wide kernel can be resident at once on this device (all of them spin on grid barriers, so
// the launch must never exceed it); cached per (device, instantiation)
template <int NT1>
static int wide_max_clusters(const PpoArgs& a, cudaStream_t st, int* out) {
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr[1];
    void (*kern)(const PpoArgs);
    if (int rc = launch_cfg<NT1, true>(a, st, 1, &cfg, attr, &kern)) return rc;
    cfg.gridDim = dim3(NCTA * 32);
    int n = 0;
    ICRL_CUDA(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
    *out = n;
    return 0;
}

// wide mode: one launch per epoch -- gather that epoch's minibatch-ordered streams, its per-step statistics, then the
// many-cluster kernel.  The device decides the target_kl stop (result[3]); later launches return at once.
template <int NT1>
static int launch_ppo_wide(PpoArgs a, cudaStream_t st, int n_clusters, float* xs, float* as, float* ss, float* advstats) {
    constexpr int F = ppo_frag_floats<NT1>();
    void *part, *sync;
    int rc;
    const size_t part_floats = ((size_t)3 * n_clusters * F + (size_t)3 * F) * NTT;
    if ((rc = device_scratch(SLOT_PPO4, part_floats * 4, &part))) return rc;
    if ((rc = device_scratch(SLOT_PPO5, 64, &sync))) return rc;
    const int n_epochs = a.n_epochs, spe = a.steps_per_epoch;
    const int* perm = a.perm;
    float* stats = a.stats;
    const double* advsums = a.advsums;
    const long long step_before = a.step_before;
    const unsigned int flag_base = a.flag_base;
    a.ncl = n_clusters;
    a.n_epochs_total = n_epochs;
    a.wide_part = (float*)part;
    a.wide_red = (float*)part + (size_t)3 * n_clusters * F * NTT;
    a.wide_sync = (unsigned int*)sync;
    a.xs = xs; a.as = as; a.ss = ss; a.advstats = advstats;
    {   // result[0] = n_epochs unless a launch stops early
        const int32_t init[4] = {n_epochs, 0, 0, 0};
        ICRL_CUDA(cudaMemcpyAsync(a.result, init, sizeof(init), cudaMemcpyHostToDevice, st));
    }
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr[1];
    void (*kern)(const PpoArgs);
    if ((rc = launch_cfg<NT1, true>(a, st, n_clusters, &cfg, attr, &kern))) return rc;
    const long long n_alloc = (long long)a.N + RB;
    const long long blocks = (n_alloc + 7) / 8;
    const int ggrid = (int)(blocks < 8LL * sm_count() ? blocks : 8LL * sm_count());
    for (int e = 0; e < n_epochs; ++e) {
        a.n_epochs = 1;
        a.epoch_base = e;
        a.perm = perm + (size_t)e * a.N;
        a.stats = stats + (size_t)e * spe * ICRL_PPO_STATS_PER_STEP;
        a.advsums = advsums ? advsums + (size_t)e * spe * 4 : nullptr;
        a.step_before = step_before + (long long)e * spe;
        a.flag_base = flag_base + (unsigned int)(e * spe);
        ppo_gather_kernel<<<ggrid, 256, 0, st>>>(a, xs, as, ss, (long long)a.N, n_alloc);
        ICRL_LAUNCH_CHECK();
        ppo_stats_kernel<<<spe, 128, 0, st>>>(ss, advstats, a.N, a.B, spe, a.beta1, a.beta2, a.lr, a.step_before, a.advsums);
        ICRL_LAUNCH_CHECK();
        ICRL_CUDA(cudaMemsetAsync(sync, 0, 64, st));
        const cudaError_t err = cudaLaunchKernelEx(&cfg, kern, a);
        if (err != cudaSuccess) {
            set_error("wide ppo_train_kernel launch failed: %s", cudaGetErrorString(err));
            return (int)err;
        }
        count_launch();
    }
    return 0;
}

}  // namespace icrl

extern "C" {

int64_t icrl_ppo_param_count(const icrl_ppo_cfg* cfg) {
    icrl::PpoArgs a = {};
    if (icrl::ppo_make_args(cfg, a)) return -1;
    return icrl::ppo_fill_offsets(a);
}

static void ppo_print_timing(unsigned long long* timing_dev, cudaStream_t st, double steps);

static int ppo_train_impl(const icrl_ppo_cfg* cfg, const icrl_ppo_data* data, float* params, float* adam_m, float* adam_v,
                          int64_t adam_step_before, float* step_stats, int32_t* result, const icrl_ppo_dist* dist,
                          void* stream) {
    icrl::PpoArgs a = {};
    int rc = icrl::ppo_make_args(cfg, a);
    if (rc) return rc;
    if (dist) {
        ICRL_CHECK_ARG(dist->world >= 1 && dist->world <= ICRL_PPO_MAX_RANKS && dist->rank >= 0 && dist->rank < dist->world,
                       "bad rank/world (%d/%d)", dist->rank, dist->world);
        ICRL_CHECK_ARG(dist->world == 1 || a.n_shared == 0,
                       "shared policy layers (n_shared = %d) are not supported in data-parallel training (world %d)",
                       a.n_shared, dist->world);
        a.rank = dist->rank; a.world = dist->world; a.flag_base = dist->flag_base; a.advsums = dist->advsums;
        for (int r = 0; r < dist->world; ++r) {
            ICRL_CHECK_ARG(dist->world == 1 || (dist->recv[r] && dist->flags[r]), "peer buffer %d is NULL", r);
            a.recv[r] = dist->recv[r]; a.flags[r] = dist->flags[r];
        }
        ICRL_CHECK_ARG(dist->world == 1 || dist->advsums, "data-parallel mode needs the all-reduced advsums table");
    }
    ICRL_CHECK_ARG(data && params && adam_m && adam_v && step_stats && result, "NULL pointer passed to icrl_ppo_train");
    ICRL_CHECK_ARG(a.N > 0 && a.n_epochs > 0, "empty rollout buffer or n_epochs <= 0");
    ICRL_CHECK_ARG(data->observations && data->actions && data->old_log_prob && data->reward_advantages &&
                       data->reward_returns && data->cost_advantages && data->cost_returns && data->perm,
                   "NULL rollout array");
    ICRL_CHECK_ARG((!a.has_clip_vf_r || data->old_reward_values) && (!a.has_clip_vf_c || data->old_cost_values),
                   "value clipping enabled but old values are NULL");
    a.obs = data->observations; a.act = data->actions; a.old_logp = data->old_log_prob;
    a.old_vr = data->old_reward_values ? data->old_reward_values : data->reward_returns;
    a.adv_r = data->reward_advantages; a.ret_r = data->reward_returns;
    a.old_vc = data->old_cost_values ? data->old_cost_values : data->cost_returns;
    a.adv_c = data->cost_advantages; a.ret_c = data->cost_returns;
    a.perm = data->perm;
    a.nu_dev = data->nu_device;
    a.params = params; a.adam_m = adam_m; a.adam_v = adam_v; a.stats = step_stats; a.result = result;
    a.step_before = adam_step_before;
    if (a.world < 1) { a.world = 1; a.rank = 0; }
    {
        const char* m = getenv("ICRL_PPO_DIST_MODE");      // 0 auto, 1 direct exchange, 2 reduce-scatter/all-gather
        a.dist_mode = m ? atoi(m) : 0;
    }
    cudaStream_t st = (cudaStream_t)stream;
    ICRL_CUDA(cudaMemsetAsync(result, 0, 4 * sizeof(int32_t), st));
    const int n_tiles = a.KP / 8;                 // n-tiles of dW1; each warp owns every second one
    const int nt1 = (n_tiles + 1) / 2;
    if (nt1 > 8) {
        icrl::set_error("obs_dim %d too large for the PPO kernel (max 128)", a.D);
        return ICRL_EUNSUPPORTED;
    }
    static unsigned long long* timing_dev = nullptr;
    const bool want_timing = getenv("ICRL_PPO_TIMING") != nullptr && a.n_shared == 0;   // (no timed shared-layer kernel)
    if (want_timing && !timing_dev) cudaMalloc(&timing_dev, 128 * sizeof(unsigned long long));
    a.timing = want_timing ? timing_dev : nullptr;
    auto print_timing = [&](double steps) { ppo_print_timing(timing_dev, st, steps); };
    // large batches run on many clusters (ICRL_PPO_WIDE=0/1 forces the choice, ICRL_PPO_WIDE_CLUSTERS caps the cluster count)
    bool wide = a.B >= icrl::WIDE_MIN_BATCH;
    if (const char* m = getenv("ICRL_PPO_WIDE")) wide = atoi(m) != 0;
    int n_clusters = 1;
    if (wide) {
        int cap = 0;
        if (nt1 <= 1) rc = icrl::wide_max_clusters<1>(a, st, &cap);
        else if (nt1 <= 2) rc = icrl::wide_max_clusters<2>(a, st, &cap);
        else if (nt1 <= 4) rc = icrl::wide_max_clusters<4>(a, st, &cap);
        else rc = icrl::wide_max_clusters<8>(a, st, &cap);
        if (rc) return rc;
        if (cap > icrl::WIDE_MAXCTA / icrl::NCTA) cap = icrl::WIDE_MAXCTA / icrl::NCTA;
        const int useful = (a.B + icrl::RB - 1) / icrl::RB;            // one 64-row chunk per cluster at least
        n_clusters = cap < useful ? cap : useful;
        if (const char* m = getenv("ICRL_PPO_WIDE_CLUSTERS")) {          // tests: exactly this many clusters (some may stay empty)
            const int c = atoi(m);
            if (c > 0) n_clusters = c < cap ? c : cap;
        }
        const int nt1r = nt1 <= 1 ? 1 : nt1 <= 2 ? 2 : nt1 <= 4 ? 4 : 8;
        const int F = icrl::NTW2 * 4 + nt1r * 4 + 4 + 1 + 5;
        if (n_clusters < 1 || 2 * n_clusters * icrl::WIDE_SMAX < F) wide = false;   // too few clusters to spread the reduction
    }
    {
        const int epochs_alloc = wide ? 1 : a.n_epochs;           // wide mode stages one epoch at a time
        const int total_steps = epochs_alloc * a.steps_per_epoch;
        const long long n_rows = (long long)epochs_alloc * a.N, n_alloc = n_rows + icrl::RB;
        const int aw = a.is_discrete ? 1 : a.A;
        a.AP = (aw + 3) / 4 * 4;
        void *xs, *as, *ss, *advstats;
        if ((rc = icrl::device_scratch(icrl::SLOT_PPO0, (size_t)n_alloc * a.DP * 4, &xs))) return rc;
        if ((rc = icrl::device_scratch(icrl::SLOT_PPO1, (size_t)total_steps * 8 * sizeof(float), &advstats))) return rc;
        if ((rc = icrl::device_scratch(icrl::SLOT_PPO2, (size_t)n_alloc * a.AP * 4, &as))) return rc;
        if ((rc = icrl::device_scratch(icrl::SLOT_PPO3, (size_t)n_alloc * 8 * 4, &ss))) return rc;
        if (wide) {
            if (nt1 <= 1) rc = icrl::launch_ppo_wide<1>(a, st, n_clusters, (float*)xs, (float*)as, (float*)ss, (float*)advstats);
            else if (nt1 <= 2) rc = icrl::launch_ppo_wide<2>(a, st, n_clusters, (float*)xs, (float*)as, (float*)ss, (float*)advstats);
            else if (nt1 <= 4) rc = icrl::launch_ppo_wide<4>(a, st, n_clusters, (float*)xs, (float*)as, (float*)ss, (float*)advstats);
            else rc = icrl::launch_ppo_wide<8>(a, st, n_clusters, (float*)xs, (float*)as, (float*)ss, (float*)advstats);
            if (rc == 0 && want_timing) {       // the last epoch's launch; per step of that launch
                fprintf(stderr, "[ppo timing] many-cluster kernel, %d clusters, last epoch (%d steps of %d rows):\n", n_clusters,
                        a.steps_per_epoch, a.B);
                print_timing((double)a.steps_per_epoch);
            }
            return rc;
        }
        const long long blocks = (n_alloc + 7) / 8;
        const int grid = (int)(blocks < 8LL * icrl::sm_count() ? blocks : 8LL * icrl::sm_count());
        icrl::ppo_gather_kernel<<<grid, 256, 0, st>>>(a, (float*)xs, (float*)as, (float*)ss, n_rows, n_alloc);
        ICRL_LAUNCH_CHECK();
        icrl::ppo_stats_kernel<<<total_steps, 128, 0, st>>>((const float*)ss, (float*)advstats, a.N, a.B, a.steps_per_epoch,
                                                            a.beta1, a.beta2, a.lr, a.step_before, a.advsums);
        ICRL_LAUNCH_CHECK();
        a.xs = (const float*)xs; a.as = (const float*)as; a.ss = (const float*)ss;
        a.advstats = (const float*)advstats;
    }
    if (nt1 <= 1) rc = icrl::launch_ppo<1>(a, st);
    else if (nt1 <= 2) rc = icrl::launch_ppo<2>(a, st);
    else if (nt1 <= 4) rc = icrl::launch_ppo<4>(a, st);
    else rc = icrl::launch_ppo<8>(a, st);
    if (rc == 0 && want_timing) print_timing((double)(a.max_steps > 0 ? a.max_steps : a.n_epochs * a.steps_per_epoch));
    return rc;
}

// profiling aid (ICRL_PPO_TIMING=1): per-phase cycles of thread 0 of each trunk's first CTA (cluster 0); synchronises!
static void ppo_print_timing(unsigned long long* timing_dev, cudaStream_t st, double steps) {
    unsigned long long h[128];
    cudaStreamSynchronize(st);
    cudaMemcpy(h, timing_dev, sizeof(h), cudaMemcpyDeviceToHost);
    const char* names[11] = {"wait+sync", "prefetch", "L1", "L2", "head", "headgrad+dH2", "dW2+dH1", "dW1", "blockreduce+stats",
                             "norm xchg", "adam"};
    for (int r = 0; r < icrl::NCTA; r += (r == 0 ? 1 : 2)) {
        const unsigned long long* t = h + r * 20;
        fprintf(stderr, "[ppo timing] cta %d cycles/step:", r);
        double tot = 0;
        for (int i = 0; i < 11; ++i) { fprintf(stderr, " %s=%.0f", names[i], t[i] / steps); tot += t[i] / steps; }
        for (int i = 11; i < 19; ++i) tot += t[i] / steps;
        fprintf(stderr, " | head: dot=%.0f logp=%.0f, headgrad: dHW=%.0f bias/logstd=%.0f dH2=%.0f | exchange: pair wait+add=%.0f "
                        "rank send=%.0f rank poll+sum=%.0f | total=%.0f\n",
                t[11] / steps, t[12] / steps, t[13] / steps, t[14] / steps, t[15] / steps, t[16] / steps, t[17] / steps,
                t[18] / steps, tot);
    }
}

int icrl_ppo_train(const icrl_ppo_cfg* cfg, const icrl_ppo_data* data, float* params, float* adam_m, float* adam_v,
                   int64_t adam_step_before, float* step_stats, int32_t* result, void* stream) {
    return ppo_train_impl(cfg, data, params, adam_m, adam_v, adam_step_before, step_stats, result, nullptr, stream);
}

int icrl_ppo_train_dist(const icrl_ppo_cfg* cfg, const icrl_ppo_data* data, float* params, float* adam_m, float* adam_v,
                        int64_t adam_step_before, float* step_stats, int32_t* result, const icrl_ppo_dist* dist,
                        void* stream) {
    ICRL_CHECK_ARG(dist != nullptr, "dist is NULL");
    return ppo_train_impl(cfg, data, params, adam_m, adam_v, adam_step_before, step_stats, result, dist, stream);
}

int icrl_ppo_local_advsums(const icrl_ppo_cfg* cfg, const icrl_ppo_data* data, double* advsums_out, void* stream) {
    icrl::PpoArgs a = {};
    int rc = icrl::ppo_make_args(cfg, a);
    if (rc) return rc;
    ICRL_CHECK_ARG(data && advsums_out && data->perm && data->reward_advantages && data->cost_advantages && a.N > 0,
                   "NULL pointer passed to icrl_ppo_local_advsums");
    icrl::ppo_local_advsums_kernel<<<a.n_epochs * a.steps_per_epoch, 128, 0, (cudaStream_t)stream>>>(
        data->perm, data->reward_advantages, data->cost_advantages, a.T, a.E, a.N, a.B, a.steps_per_epoch, advsums_out);
    ICRL_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
