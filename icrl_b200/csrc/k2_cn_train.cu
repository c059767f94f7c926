// K2 -- importance-sampling-weighted constraint-net training, replaces ConstraintNet.train + compute_is_weights +
// ConstraintNet.get + th.optim.Adam.step (icrl/constraint_net.py:137-256, 301-317).
//
// Per backward iteration, six launches on one stream and NO host synchronisation (the early-stop decision is a device flag
// every later kernel checks first).  Every kernel is multi-CTA; the cross-CTA steps use per-CTA partials + a "last block
// done" ticket, the cross-GPU steps (data-parallel mode) ride on the same tickets:
//   A   cn_forward (K1 kernel, out_kind = prediction) over this rank's nominal rows         -> current_preds
//   B1  cn_is_partial_kernel   sum of the IS ratios, per-episode products (float64 log-sum)            [exchange 0]
//   B2  cn_is_weights_kernel   mean ratio, normalised weights, both KLs, early-stop test (constraint_net.py:231-256,
//                              173-177), weight statistics                                               [exchange 1]
//   C   cn_grad_kernel         forward + backward over nominal and expert tiles; weight gradients are contractions over
//                              the rows of a tile (dW_l = dH_l^T A_{l-1}) accumulated in shared memory, one partial
//                              gradient per CTA (deterministic reduction, no float atomics)
//   D1  cn_reduce_kernel       per-parameter sum of the CTA partials                                     [exchange 2]
//   D2  cn_adam_kernel         sum over ranks in rank order, loss / prediction statistics, Adam (torch single-tensor
//                              rule, eps 1e-5)
// Data-parallel mode (SURVEY 8(e): "shard nominal rows by whole episodes and expert rows evenly"): every rank runs the same
// six kernels on ITS nominal episodes / expert rows.  An exchange is: every rank stores its partial result straight into
// every rank's exchange buffer (CUDA-IPC mapped peer memory, NVLink stores from inside the kernel), the last block to
// finish fences and publishes a sequence number in each peer's flag slot; the consuming kernel spins on its own flag slots
// (bounded) and then sums the W contributions in rank order, so all replicas apply bit-identical Adam updates.  With one
// rank the same code runs on a local buffer.  No NCCL call, no host round trip.
// Minibatch mode (`cn_batch_size`, constraint_net.py:304-317): the IS weights still come from the full nominal set; C / D1
// / D2 then run once per minibatch on rows gathered through the host-drawn numpy permutation (same indices for the nominal
// and the expert set, as the reference does).
// Quirk A (SURVEY 8 a16): in per-step IS mode the reference's [N,1,1] x [N,1] broadcast makes the nominal loss
// mean(w) * mean(log(p+eps)); we reproduce that value and gradient in O(N).
#include <math.h>

#include <algorithm>

#include "cn_common.cuh"

namespace icrl {

int cn_forward_device(const CnPlan& plan, const void* obs, int obs_is_f64, const float* acs, int64_t n_rows, float* out,
                      int out_kind, cudaStream_t st);

struct CnCtrl {          // device-resident control / result block
    int stopped;         // a KL threshold was exceeded: every later kernel returns at once
    int early_stop_itr;
    int steps_taken;
    int error;           // an exchange wait hit its bound (a peer rank is gone)
    int pending_stop;    // B2's block 0 decides, B2's last block publishes it as `stopped`
    unsigned int ticket[3];
    float mean_w;        // minibatch mode: mean of the IS weights over the minibatch's rows
    float is_mean, is_max, is_min, kl_old_new, kl_new_old;
    float m[14];         // loss / prediction metrics of the last completed step (icrl_cn_train_metrics order)
};

enum { ST_NLOG = 0, ST_NWLOG, ST_N1MP, ST_NSUM, ST_NMAX, ST_NMIN, ST_ELOG, ST_E1MP, ST_ESUM, ST_EMAX, ST_EMIN, ST_COUNT = 12 };

// ------------------------------------------------------------------------------------------------ exchange buffers
// One buffer per rank (local scratch when there is a single rank), identical layout everywhere:
//   CnXHeader | float grad[MAX_RANKS][gstride] | float prod_all[n_episodes_global]
struct CnXHeader {
    unsigned int flags[3][ICRL_PPO_MAX_RANKS];          // [exchange][source rank] = sequence number of the last complete push
    unsigned int pad[8];
    double sum_ratio[ICRL_PPO_MAX_RANKS];               // exchange 0
    double wstat[ICRL_PPO_MAX_RANKS][4];                // exchange 1: sum w, max w, min w, any NaN
    double stats[ICRL_PPO_MAX_RANKS][ST_COUNT];         // exchange 2
};
struct CnX {
    int rank, world;
    int gstride;                                         // floats per rank slot of the gradient area
    unsigned char* buf[ICRL_PPO_MAX_RANKS];
    __host__ __device__ CnXHeader* hdr(int r) const { return reinterpret_cast<CnXHeader*>(buf[r]); }
    __host__ __device__ float* grad(int r, int src) const {
        return reinterpret_cast<float*>(buf[r] + sizeof(CnXHeader)) + (size_t)src * gstride;
    }
    __host__ __device__ float* prod(int r) const {
        return reinterpret_cast<float*>(buf[r] + sizeof(CnXHeader)) + (size_t)ICRL_PPO_MAX_RANKS * gstride;
    }
};
static_assert(sizeof(CnXHeader) % 16 == 0, "exchange header must keep the float areas 16-byte aligned");
inline int cn_gstride(int n_params) { return (n_params + 3) / 4 * 4; }
inline size_t cn_xchg_bytes(int n_params, int n_episodes_global) {
    return sizeof(CnXHeader) + ((size_t)ICRL_PPO_MAX_RANKS * cn_gstride(n_params) + (size_t)(n_episodes_global > 0 ? n_episodes_global : 1)) * 4;
}

__device__ __forceinline__ void cn_st_release_sys(unsigned int* p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int cn_ld_acquire_sys(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// every thread of the block returns once all ranks have published `want` for exchange `e` (bounded: ~2 s)
__device__ __forceinline__ void cn_wait(const CnX& x, int e, unsigned int want, CnCtrl* ctrl) {
    if ((int)threadIdx.x < x.world) {
        const unsigned int* f = &x.hdr(x.rank)->flags[e][threadIdx.x];
        const long long t0 = clock64();
        while ((int)(cn_ld_acquire_sys(f) - want) < 0) {
            if (clock64() - t0 > 4000000000LL) { ctrl->error = 1; break; }
        }
    }
    __syncthreads();
}
// "last block done": true in every thread of the block that arrives last (all blocks' earlier global / peer stores are
// visible to it and, through its own later release stores, to the peers)
__device__ __forceinline__ bool cn_last_block(unsigned int* ticket) {
    __shared__ int is_last;
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    __syncthreads();
    if (is_last) __threadfence_system();
    return is_last != 0;
}
__device__ __forceinline__ double cn_block_sum(double v, double* red /* [32] shared */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    double t = 0.0;
    for (int i = 0; i < nwarp; ++i) t += red[i];
    return t;
}

// ------------------------------------------------------------------------------------------------ B1
// ratio_i = (p_new_i + eps) / (p_old_i + eps); prod_j = exp(sum_i log ratio_i) accumulated in float64 (overflow -> inf,
// underflow -> 0, as the reference's fp32 th.prod)
__global__ void __launch_bounds__(256) cn_is_partial_kernel(CnCtrl* ctrl, const CnX x, const float* __restrict__ p_old,
                                                            const float* __restrict__ p_new, const int* __restrict__ offsets,
                                                            int n_episodes, int episode_base, long long n, float eps,
                                                            unsigned int want, double* __restrict__ part) {
    __shared__ double red[32];
    if (ctrl->stopped) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
    double s = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + tid; i < n; i += (long long)gridDim.x * blockDim.x)
        s += (double)((p_new[i] + eps) / (p_old[i] + eps));
    s = cn_block_sum(s, red);
    if (tid == 0) part[blockIdx.x] = s;
    for (int j = blockIdx.x * nwarp + warp; j < n_episodes; j += gridDim.x * nwarp) {
        double ls = 0.0;
        for (int i = offsets[j] + lane; i < offsets[j + 1]; i += 32) ls += log((double)((p_new[i] + eps) / (p_old[i] + eps)));
        ls = warp_sum(ls);
        if (lane == 0) {
            const float pj = (float)exp(ls);
            for (int r = 0; r < x.world; ++r) x.prod(r)[episode_base + j] = pj;
        }
    }
    if (cn_last_block(&ctrl->ticket[0]) && tid < 32) {
        // warp 0 of the last block: lanes stride over the CTA partials (independent L2 loads), shuffle tree in a fixed order
        double tot = 0.0;
        for (unsigned int b = tid; b < gridDim.x; b += 32) tot += *(volatile double*)&part[b];
        tot = warp_sum(tot);
        if (tid == 0) {
            for (int r = 0; r < x.world; ++r) x.hdr(r)->sum_ratio[x.rank] = tot;
            __threadfence_system();
            for (int r = 0; r < x.world; ++r) cn_st_release_sys(&x.hdr(r)->flags[0][x.rank], want);
            ctrl->ticket[0] = 0;
        }
    }
}

// ------------------------------------------------------------------------------------------------ B2
__global__ void __launch_bounds__(256) cn_is_weights_kernel(CnCtrl* ctrl, const CnX x, const float* __restrict__ p_old,
                                                            const float* __restrict__ p_new, const int* __restrict__ offsets,
                                                            int n_episodes, int episode_base, long long n, double n_global,
                                                            int m_global, float eps, int use_is, int per_step, float tkon,
                                                            float tkno, int itr, unsigned int want, float* __restrict__ w,
                                                            double* __restrict__ part) {
    __shared__ double red[32];
    __shared__ float redf[2][8];
    if (ctrl->stopped) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
    double ws = 0.0;
    float wmax = -INFINITY, wmin = INFINITY;
    bool wnan = false;
    if (!use_is) {
        for (long long i = (long long)blockIdx.x * blockDim.x + tid; i < n; i += (long long)gridDim.x * blockDim.x) {
            w[i] = 1.f;
            ws += 1.0;
        }
        wmax = wmin = 1.f;
    } else {
        cn_wait(x, 0, want, ctrl);
        double sr = 0.0;
        for (int r = 0; r < x.world; ++r) sr += x.hdr(x.rank)->sum_ratio[r];
        const float mean_ratio = (float)(sr / n_global);
        const float* prod = x.prod(x.rank);
        double sp = 0.0;
        for (int j = tid; j < m_global; j += blockDim.x) sp += (double)prod[j];
        const float sum_prod = (float)cn_block_sum(sp, red);
        if (blockIdx.x == 0) {
            const float prod_mean = sum_prod / (float)m_global;
            double k1 = 0.0, k2 = 0.0;
            for (int j = tid; j < m_global; j += blockDim.x) {
                const float pj = prod[j], lg = logf(pj + eps);
                k1 += (double)(-lg);
                k2 += (double)((pj - prod_mean) * lg / (prod_mean + eps));
            }
            const float kl_old_new = (float)(cn_block_sum(k1, red) / m_global);
            const float kl_new_old = (float)(cn_block_sum(k2, red) / m_global);
            if (tid == 0) {
                ctrl->kl_old_new = kl_old_new; ctrl->kl_new_old = kl_new_old;
                // constraint_net.py:174-177 (NaN / -inf never compare greater)
                if ((tkon != -1.f && kl_old_new > tkon) || (tkno != -1.f && kl_new_old > tkno)) {
                    ctrl->pending_stop = 1;
                    ctrl->early_stop_itr = itr;
                }
            }
        }
        if (per_step) {
            for (long long i = (long long)blockIdx.x * blockDim.x + tid; i < n; i += (long long)gridDim.x * blockDim.x) {
                const float wi = ((p_new[i] + eps) / (p_old[i] + eps)) / mean_ratio;
                w[i] = wi; ws += (double)wi; wmax = fmaxf(wmax, wi); wmin = fminf(wmin, wi); wnan |= (wi != wi);
            }
        } else {
            for (int j = blockIdx.x * nwarp + warp; j < n_episodes; j += gridDim.x * nwarp) {
                const float wj = (float)m_global * prod[episode_base + j] / (sum_prod + eps);
                for (int i = offsets[j] + lane; i < offsets[j + 1]; i += 32) w[i] = wj;
                if (lane == 0) {
                    ws += (double)wj * (double)(offsets[j + 1] - offsets[j]);
                    wmax = fmaxf(wmax, wj); wmin = fminf(wmin, wj); wnan |= (wj != wj);
                }
            }
        }
    }
    ws = cn_block_sum(ws, red);
    wmax = warp_max(wmax); wmin = warp_min(wmin);
    const unsigned anynan = __ballot_sync(0xffffffffu, wnan);
    if (lane == 0) { redf[0][warp] = anynan ? NAN : wmax; redf[1][warp] = anynan ? NAN : wmin; }
    __syncthreads();
    if (tid == 0) {
        float mx = -INFINITY, mn = INFINITY;
        bool nn = false;
        for (int i = 0; i < nwarp; ++i) {
            nn |= (redf[0][i] != redf[0][i]);
            mx = fmaxf(mx, redf[0][i]); mn = fminf(mn, redf[1][i]);
        }
        double* o = part + (size_t)blockIdx.x * 4;
        o[0] = ws; o[1] = (double)mx; o[2] = (double)mn; o[3] = nn ? 1.0 : 0.0;
    }
    if (cn_last_block(&ctrl->ticket[1]) && tid < 32) {
        double tot = 0.0, mx = -INFINITY, mn = INFINITY, nn = 0.0;
        for (unsigned int b = tid; b < gridDim.x; b += 32) {
            const volatile double* o = part + (size_t)b * 4;
            tot += o[0]; mx = fmax(mx, o[1]); mn = fmin(mn, o[2]); nn += o[3];
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            tot += __shfl_xor_sync(0xffffffffu, tot, o);
            mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
            mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            nn += __shfl_xor_sync(0xffffffffu, nn, o);
        }
        if (tid != 0) return;
        for (int r = 0; r < x.world; ++r) {
            double* d = x.hdr(r)->wstat[x.rank];
            d[0] = tot; d[1] = mx; d[2] = mn; d[3] = nn;
        }
        __threadfence_system();
        for (int r = 0; r < x.world; ++r) cn_st_release_sys(&x.hdr(r)->flags[1][x.rank], want);
        // the logged is_mean / is_max / is_min are those of the LAST importance-weight evaluation, early stops included
        // (constraint_net.py:171-177, 214-216): combine all ranks' statistics here rather than in the Adam kernel
        const CnXHeader* h = x.hdr(x.rank);
        double sw = 0.0, wmx = -INFINITY, wmn = INFINITY, wnan = 0.0;
        const long long t0 = clock64();
        for (int r = 0; r < x.world; ++r) {
            while ((int)(cn_ld_acquire_sys(&h->flags[1][r]) - want) < 0) {
                if (clock64() - t0 > 4000000000LL) { ctrl->error = 1; break; }
            }
            sw += h->wstat[r][0]; wmx = fmax(wmx, h->wstat[r][1]); wmn = fmin(wmn, h->wstat[r][2]); wnan += h->wstat[r][3];
        }
        ctrl->is_mean = (float)(sw / n_global);
        ctrl->is_max = wnan > 0.0 ? NAN : (float)wmx;      // torch.max / min propagate NaN
        ctrl->is_min = wnan > 0.0 ? NAN : (float)wmn;
        ctrl->stopped = ctrl->pending_stop;
        ctrl->ticket[1] = 0;
    }
}

// minibatch mode, per-step IS: the mean of the weights over the minibatch's rows (what the reference's broadcast collapses to)
__global__ void __launch_bounds__(256) cn_batch_meanw_kernel(CnCtrl* ctrl, const float* __restrict__ w,
                                                             const int* __restrict__ idx, int n_batch) {
    __shared__ double red[32];
    if (ctrl->stopped) return;
    double s = 0.0;
    for (int i = threadIdx.x; i < n_batch; i += blockDim.x) s += (double)w[idx[i]];
    s = cn_block_sum(s, red);
    if (threadIdx.x == 0) ctrl->mean_w = (float)(s / (double)n_batch);
}

// ------------------------------------------------------------------------------------------------ C
struct GradSmem {
    int bar, mean, rstd, low, high, w[ICRL_MAX_HIDDEN], wb[ICRL_MAX_HIDDEN], b[ICRL_MAX_HIDDEN], wout, raw, acs, xp, hp, dz, g,
        total;
    int LD, KP0;
};

__host__ __device__ inline GradSmem grad_smem_layout(const CnPlan& p, int HP, int TILE, int obs_elem, int n_params) {
    GradSmem s;
    s.LD = TILE + 4;
    s.KP0 = align_up(p.n_select, 4);
    int off = 0;
    s.bar = off; off += 16;
    s.mean = off; off += p.has_norm ? p.obs_dim * 8 : 0;
    s.rstd = off; off += p.has_norm ? p.obs_dim * 8 : 0;
    s.low = off; off += p.has_clip_acs ? p.acs_dim * 4 : 0;
    s.high = off; off += p.has_clip_acs ? p.acs_dim * 4 : 0;
    off = align_up(off, 16);
    for (int l = 0; l < ICRL_MAX_HIDDEN; ++l) {
        s.w[l] = off;                                   // forward copy, k-major [K][HP]
        if (l < p.n_hidden) off += (l == 0 ? p.n_select : HP) * HP * 4;
        s.wb[l] = off;                                  // backward copy, [j][HP] (row j = output unit, cols = inputs), l >= 1
        if (l < p.n_hidden && l >= 1) off += HP * HP * 4;
        s.b[l] = off;
        if (l < p.n_hidden) off += HP * 4;
    }
    s.wout = off; off += (HP + 4) * 4;
    off = align_up(off, 16);
    const int raw_bytes = align_up(TILE * p.obs_dim * obs_elem, 16);
    const int dh_bytes = p.n_hidden * HP * s.LD * 4;    // dH planes alias the raw obs tile (dead after input preparation)
    s.raw = off; off += raw_bytes > dh_bytes ? raw_bytes : dh_bytes;
    s.acs = off; off += align_up(TILE * p.acs_w * 4, 16);
    s.xp = off; off += s.KP0 * s.LD * 4;                // prepared inputs, k-major planes [KP0][LD]
    s.hp = off; off += p.n_hidden * HP * s.LD * 4;      // activations per layer [l][HP][LD]
    s.dz = off; off += s.LD * 4;
    s.g = off; off += align_up(n_params, 4) * 4;        // per-CTA gradient accumulator, flat parameter order
    s.total = off;
    return s;
}

// `idx` != NULL (minibatch mode): the tile rows are gathered through idx[0 .. n_batch) from BOTH sets (the reference uses the
// same batch indices for the nominal and the expert batch, constraint_net.py:304-317) and n_nom == n_exp == n_batch.
// The 1/N factors of the loss means use the GLOBAL row counts (all ranks).
template <typename ObsT, int HP>
__global__ void __launch_bounds__(128) cn_grad_kernel(const __grid_constant__ CnPlan plan, CnCtrl* __restrict__ ctrl,
                                                      const CnX x, unsigned int want1, int need_meanw,
                                                      const ObsT* __restrict__ nobs, const float* __restrict__ nacs,
                                                      long long n_nom, const ObsT* __restrict__ eobs,
                                                      const float* __restrict__ eacs, long long n_exp,
                                                      double n_nom_global, double n_exp_global,
                                                      const int* __restrict__ idx,
                                                      const float* __restrict__ w, int per_step, int gail, float eps,
                                                      float reg, int n_params, int tma_ok, float* __restrict__ part_grad,
                                                      float* __restrict__ part_stats) {
    extern __shared__ __align__(16) unsigned char smem[];
    if (ctrl->stopped) return;
    const int TILE = blockDim.x, tid = threadIdx.x;
    const GradSmem L = grad_smem_layout(plan, HP, TILE, sizeof(ObsT), n_params);
    const int LD = L.LD, KP0 = L.KP0, NH = plan.n_hidden;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + L.bar);
    float* XP = reinterpret_cast<float*>(smem + L.xp);
    float* HPL = reinterpret_cast<float*>(smem + L.hp);
    float* DH = reinterpret_cast<float*>(smem + L.raw);
    float* DZ = reinterpret_cast<float*>(smem + L.dz);
    float* G = reinterpret_cast<float*>(smem + L.g);
    float* WO = reinterpret_cast<float*>(smem + L.wout);
    if (tid == 0) { mbar_init(bar, 1); fence_mbar_init(); }
    // weights: forward (k-major) copies via the shared loader layout, plus [j][k] copies for the backward pass
    {
        CnSmem F;   // reuse cn_load_weights with our offsets
        F.bar = L.bar; F.mean = L.mean; F.rstd = L.rstd; F.low = L.low; F.high = L.high; F.wout = L.wout;
        for (int l = 0; l < ICRL_MAX_HIDDEN; ++l) { F.w[l] = L.w[l]; F.b[l] = L.b[l]; }
        F.obs = L.raw; F.acs = L.acs; F.h = L.hp; F.total = L.total;
        cn_load_weights<HP>(plan, F, smem);
        const float* src = plan.params;
        int in_dim = plan.n_select;
        for (int l = 0; l < NH; ++l) {
            const int out_dim = plan.hidden[l];
            if (l >= 1) {
                float* WB = reinterpret_cast<float*>(smem + L.wb[l]);
                for (int i = tid; i < HP * HP; i += TILE) {
                    const int j = i / HP, k = i - j * HP;
                    WB[i] = (j < out_dim && k < in_dim) ? src[j * in_dim + k] : 0.f;
                }
            }
            src += out_dim * in_dim + out_dim;
            in_dim = out_dim;
        }
    }
    for (int i = tid; i < align_up(n_params, 4); i += TILE) G[i] = 0.f;
    __syncthreads();

    // per-step IS: mean(w) over the rows the loss mean runs over -- all ranks' nominal rows (exchange 1), or the minibatch
    float mean_w = 1.f;
    if (need_meanw) {
        if (idx != nullptr) {
            mean_w = ctrl->mean_w;
        } else {
            cn_wait(x, 1, want1, ctrl);
            double sw = 0.0;
            for (int r = 0; r < x.world; ++r) sw += x.hdr(x.rank)->wstat[r][0];
            mean_w = (float)(sw / n_nom_global);
        }
    }
    const long long tiles_nom = (n_nom + TILE - 1) / TILE, tiles_exp = (n_exp + TILE - 1) / TILE;
    const float inv_nn = (float)(1.0 / n_nom_global), inv_ne = (float)(1.0 / n_exp_global);
    float st[ST_COUNT];
#pragma unroll
    for (int i = 0; i < ST_COUNT; ++i) st[i] = 0.f;
    st[ST_NMAX] = -INFINITY; st[ST_NMIN] = INFINITY; st[ST_EMAX] = -INFINITY; st[ST_EMIN] = INFINITY;
    uint32_t phase = 0;

    CnSmem S;   // staging view for cn_stage_tile / cn_input
    S.bar = L.bar; S.mean = L.mean; S.rstd = L.rstd; S.low = L.low; S.high = L.high; S.obs = L.raw; S.acs = L.acs;

    for (long long tile = blockIdx.x; tile < tiles_nom + tiles_exp; tile += gridDim.x) {
        const bool is_nom = tile < tiles_nom;
        const long long t_in = is_nom ? tile : tile - tiles_nom;
        const long long n_set = is_nom ? n_nom : n_exp;
        const long long row0 = t_in * TILE;
        const int rows = (int)min((long long)TILE, n_set - row0);
        if (idx == nullptr) {
            cn_stage_tile<ObsT>(plan, S, smem, is_nom ? nobs : eobs, is_nom ? nacs : eacs, row0, rows,
                                tma_ok && rows == TILE, phase);
        } else {
            // gathered rows: warp per row, coalesced along the row
            const ObsT* go = is_nom ? nobs : eobs;
            const float* ga = is_nom ? nacs : eacs;
            ObsT* so = reinterpret_cast<ObsT*>(smem + L.raw);
            float* sa = reinterpret_cast<float*>(smem + L.acs);
            for (int rr = tid >> 5; rr < rows; rr += TILE >> 5) {
                const long long src = idx[row0 + rr];
                for (int c = tid & 31; c < plan.obs_dim; c += 32) so[rr * plan.obs_dim + c] = go[src * plan.obs_dim + c];
                for (int c = tid & 31; c < plan.acs_w; c += 32) sa[rr * plan.acs_w + c] = ga[src * plan.acs_w + c];
            }
            __syncthreads();
        }
        const int r = tid;
        const bool active = r < rows;
        // ---- prepared inputs -> k-major planes
        for (int k = 0; k < KP0; ++k) XP[k * LD + r] = (active && k < plan.n_select) ? cn_input<ObsT>(plan, S, smem, r, k) : 0.f;
        __syncthreads();   // raw tile is dead from here on (DH aliases it)

        // ---- forward, keeping every layer's activations
        float acc[HP];
        {
            const float* B = reinterpret_cast<const float*>(smem + L.b[0]);
#pragma unroll
            for (int j = 0; j < HP; ++j) acc[j] = B[j];
            const float* W = reinterpret_cast<const float*>(smem + L.w[0]);
#pragma unroll 2
            for (int k = 0; k < plan.n_select; ++k) cn_fma_row<HP>(acc, XP[k * LD + r], W + k * HP);
        }
        for (int l = 1; l < NH; ++l) {
            float* Hp = HPL + (l - 1) * HP * LD;
#pragma unroll
            for (int j = 0; j < HP; ++j) Hp[j * LD + r] = fmaxf(acc[j], 0.f);
            const float* B = reinterpret_cast<const float*>(smem + L.b[l]);
#pragma unroll
            for (int j = 0; j < HP; ++j) acc[j] = B[j];
            const float* W = reinterpret_cast<const float*>(smem + L.w[l]);
            const int kin = plan.hidden[l - 1];
#pragma unroll 4
            for (int k = 0; k < kin; ++k) cn_fma_row<HP>(acc, Hp[k * LD + r], W + k * HP);
        }
        float z = WO[HP];
        {
            float* Hp = HPL + (NH - 1) * HP * LD;
#pragma unroll
            for (int j = 0; j < HP; ++j) {
                const float a = fmaxf(acc[j], 0.f);
                Hp[j * LD + r] = a;
                z = fmaf(a, WO[j], z);
            }
        }
        // ---- loss terms and dL/dz for this row
        const float pr = sigmoidf_ref(z);
        float dz = 0.f;
        if (active) {
            float dLdp;
            if (is_nom) {
                const float wi = per_step ? mean_w : w[idx ? (long long)idx[row0 + r] : row0 + r];
                if (gail) {
                    const float l1 = fmaxf(logf(1.f - pr), -100.f);            // nn.BCELoss clamps log at -100
                    st[ST_NLOG] += logf(pr + eps);      // `unweighted_nominal_loss` is mean(log(p + eps)) in both modes (:211)
                    st[ST_NWLOG] += -l1;                // BCE(p, 0)
                    dLdp = pr / fmaxf((1.f - pr) * pr, 1e-12f) * inv_nn;           // BCELoss backward, y = 0
                } else {
                    const float lg = logf(pr + eps);
                    st[ST_NLOG] += lg; st[ST_NWLOG] += wi * lg;
                    dLdp = wi * inv_nn / (pr + eps) - reg * inv_nn;
                }
                st[ST_N1MP] += 1.f - pr; st[ST_NSUM] += pr;
                st[ST_NMAX] = fmaxf(st[ST_NMAX], pr); st[ST_NMIN] = fminf(st[ST_NMIN], pr);
            } else {
                if (gail) {
                    const float l1 = fmaxf(logf(pr), -100.f);
                    st[ST_ELOG] += -l1;
                    // BCELoss backward with y = 1: (p - 1) / max((1 - p) p, 1e-12), so the gradient fades out on rows the
                    // discriminator rejects with p < 1e-12 instead of pushing them at full strength (-1 / p)
                    dLdp = (pr - 1.f) / fmaxf((1.f - pr) * pr, 1e-12f) * inv_ne;
                } else {
                    st[ST_ELOG] += logf(pr + eps);
                    dLdp = -inv_ne / (pr + eps) - reg * inv_ne;
                }
                st[ST_E1MP] += 1.f - pr; st[ST_ESUM] += pr;
                st[ST_EMAX] = fmaxf(st[ST_EMAX], pr); st[ST_EMIN] = fminf(st[ST_EMIN], pr);
            }
            dz = dLdp * pr * (1.f - pr);
        }
        DZ[r] = dz;
        // ---- backward through the hidden layers (thread-per-row); dH planes [l][HP][LD]
        {
            float* Hp = HPL + (NH - 1) * HP * LD;
            float* Dp = DH + (NH - 1) * HP * LD;
#pragma unroll
            for (int j = 0; j < HP; ++j) Dp[j * LD + r] = (Hp[j * LD + r] > 0.f) ? dz * WO[j] : 0.f;
        }
        for (int l = NH - 1; l >= 1; --l) {
            const float* Dp = DH + l * HP * LD;
            const float* WB = reinterpret_cast<const float*>(smem + L.wb[l]);
            float dacc[HP];
#pragma unroll
            for (int k = 0; k < HP; ++k) dacc[k] = 0.f;
            const int jout = plan.hidden[l];
#pragma unroll 4
            for (int j = 0; j < jout; ++j) cn_fma_row<HP>(dacc, Dp[j * LD + r], WB + j * HP);
            const float* Hq = HPL + (l - 1) * HP * LD;
            float* Dq = DH + (l - 1) * HP * LD;
#pragma unroll
            for (int k = 0; k < HP; ++k) Dq[k * LD + r] = (Hq[k * LD + r] > 0.f) ? dacc[k] : 0.f;
        }
        __syncthreads();

        // ---- weight gradients: contractions over the tile's rows, accumulated into the CTA's flat gradient
        {
            int goff = 0, in_dim = plan.n_select;
            for (int l = 0; l < NH; ++l) {
                const int out_dim = plan.hidden[l];
                const float* Dp = DH + l * HP * LD;
                const float* Ap = (l == 0) ? XP : HPL + (l - 1) * HP * LD;
                const int ktiles = (in_dim + 3) / 4, jtiles = (out_dim + 3) / 4;
                for (int t = tid; t < ktiles * jtiles; t += TILE) {
                    const int tj = t % jtiles, tk = t / jtiles;
                    float a4[4][4];
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < 4; ++j) a4[i][j] = 0.f;
                    for (int rr = 0; rr < TILE; rr += 4) {
                        float4 d[4], x[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            d[i] = *reinterpret_cast<const float4*>(Dp + (4 * tj + i) * LD + rr);
                            x[i] = *reinterpret_cast<const float4*>(Ap + (4 * tk + i) * LD + rr);
                        }
#pragma unroll
                        for (int i = 0; i < 4; ++i)
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                a4[i][j] = fmaf(d[i].x, x[j].x, a4[i][j]);
                                a4[i][j] = fmaf(d[i].y, x[j].y, a4[i][j]);
                                a4[i][j] = fmaf(d[i].z, x[j].z, a4[i][j]);
                                a4[i][j] = fmaf(d[i].w, x[j].w, a4[i][j]);
                            }
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const int jo = 4 * tj + i, ki = 4 * tk + j;
                            if (jo < out_dim && ki < in_dim) G[goff + jo * in_dim + ki] += a4[i][j];
                        }
                }
                for (int j = tid; j < out_dim; j += TILE) {
                    float s = 0.f;
                    for (int rr = 0; rr < TILE; rr += 4) {
                        const float4 d = *reinterpret_cast<const float4*>(Dp + j * LD + rr);
                        s += (d.x + d.y) + (d.z + d.w);
                    }
                    G[goff + out_dim * in_dim + j] += s;
                }
                goff += out_dim * in_dim + out_dim;
                in_dim = out_dim;
            }
            // output layer: dw_out[j] = sum_r dz[r] * h_last[j][r], db_out = sum_r dz[r]
            const float* Hp = HPL + (NH - 1) * HP * LD;
            for (int j = tid; j <= in_dim; j += TILE) {
                float s = 0.f;
                if (j < in_dim) {
                    for (int rr = 0; rr < TILE; rr += 4) {
                        const float4 d = *reinterpret_cast<const float4*>(DZ + rr);
                        const float4 h = *reinterpret_cast<const float4*>(Hp + j * LD + rr);
                        s = fmaf(d.x, h.x, s); s = fmaf(d.y, h.y, s); s = fmaf(d.z, h.z, s); s = fmaf(d.w, h.w, s);
                    }
                } else {
                    for (int rr = 0; rr < TILE; ++rr) s += DZ[rr];
                }
                G[goff + j] += s;
            }
        }
        __syncthreads();   // planes are rewritten by the next tile
    }

    // ---- per-CTA partial gradient and statistics
    for (int i = tid; i < n_params; i += TILE) part_grad[(size_t)blockIdx.x * n_params + i] = G[i];
    __shared__ float sred[ST_COUNT][4];
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int i = 0; i < ST_COUNT; ++i) {
        float v = st[i];
        if (i == ST_NMAX || i == ST_EMAX) v = warp_max(v);
        else if (i == ST_NMIN || i == ST_EMIN) v = warp_min(v);
        else v = warp_sum(v);
        if (lane == 0) sred[i][warp] = v;
    }
    __syncthreads();
    if (tid < ST_COUNT) {
        const int nw = (TILE + 31) / 32;
        float v = sred[tid][0];
        for (int i = 1; i < nw; ++i) {
            if (tid == ST_NMAX || tid == ST_EMAX) v = fmaxf(v, sred[tid][i]);
            else if (tid == ST_NMIN || tid == ST_EMIN) v = fminf(v, sred[tid][i]);
            else v += sred[tid][i];
        }
        part_stats[(size_t)blockIdx.x * ST_COUNT + tid] = v;
    }
}

// ------------------------------------------------------------------------------------------------ D1
// per-parameter sum of the CTA partial gradients (fixed order) -> this rank's slot in EVERY rank's exchange buffer
__global__ void __launch_bounds__(256) cn_reduce_kernel(CnCtrl* ctrl, const CnX x, const float* __restrict__ part_grad,
                                                        const float* __restrict__ part_stats, int n_parts, int n_params,
                                                        unsigned int want) {
    if (ctrl->stopped) return;
    // a WARP per parameter: lane l adds the partials of CTAs l, l + 32, ... and a shuffle tree totals the lanes (a fixed order
    // for a given n_parts).  One thread per parameter walked the n_parts partials as one dependent chain of L2 loads:
    // 80 us per launch for 119 partials, more than the gradient kernel itself.
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int i = blockIdx.x * 8 + wib;
    if (i < n_params) {
        float g = 0.f;
        for (int b = lane; b < n_parts; b += 32) g += part_grad[(size_t)b * n_params + i];
        g = warp_sum(g);
        if (lane < x.world) x.grad(lane, x.rank)[i] = g;
    }
    if (blockIdx.x == 0) {
        for (int k = wib; k < ST_COUNT; k += 8) {
            const bool is_max = (k == ST_NMAX || k == ST_EMAX), is_min = (k == ST_NMIN || k == ST_EMIN);
            double v = is_max ? -INFINITY : is_min ? INFINITY : 0.0;
            for (int b = lane; b < n_parts; b += 32) {
                const double p = (double)part_stats[(size_t)b * ST_COUNT + k];
                v = is_max ? fmax(v, p) : is_min ? fmin(v, p) : v + p;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double q = __shfl_xor_sync(0xffffffffu, v, o);
                v = is_max ? fmax(v, q) : is_min ? fmin(v, q) : v + q;
            }
            if (lane < x.world) x.hdr(lane)->stats[x.rank][k] = v;
        }
    }
    if (cn_last_block(&ctrl->ticket[2]) && threadIdx.x == 0) {
        for (int r = 0; r < x.world; ++r) cn_st_release_sys(&x.hdr(r)->flags[2][x.rank], want);
        ctrl->ticket[2] = 0;
    }
}

// ------------------------------------------------------------------------------------------------ D2
__global__ void __launch_bounds__(256) cn_adam_kernel(CnCtrl* ctrl, const CnX x, float* __restrict__ params,
                                                      float* __restrict__ adam_m, float* __restrict__ adam_v, int n_params,
                                                      double n_nom_global, double n_exp_global, double n_is_global,
                                                      int use_is, int per_step,
                                                      int batch_mode, int gail, float reg, double lr, double beta1,
                                                      double beta2, double adam_eps, long long step, int step_index,
                                                      unsigned int want) {
    if (ctrl->stopped) return;
    cn_wait(x, 2, want, ctrl);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_params) {
        const double bc1 = 1.0 - pow(beta1, (double)step), bc2 = 1.0 - pow(beta2, (double)step);
        const float omb1 = (float)(1.0 - beta1), b2 = (float)beta2, omb2 = (float)(1.0 - beta2);
        const float bc2s = (float)sqrt(bc2), epsf = (float)adam_eps, nss = (float)(-(lr / bc1));
        float g = 0.f;
        for (int r = 0; r < x.world; ++r) g += x.grad(x.rank, r)[i];          // rank order: identical bits on every replica
        float m = adam_m[i], v = adam_v[i];
        m = fmaf(omb1, g - m, m);
        v = fmaf(omb2 * g, g, v * b2);
        const float denom = sqrtf(v) / bc2s + epsf;
        params[i] = fmaf(nss, m / denom, params[i]);
        adam_m[i] = m; adam_v[i] = v;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const CnXHeader* h = x.hdr(x.rank);
        double s[ST_COUNT];
        for (int k = 0; k < ST_COUNT; ++k) s[k] = 0.0;
        double nmax = -INFINITY, nmin = INFINITY, emax = -INFINITY, emin = INFINITY;
        for (int r = 0; r < x.world; ++r) {
            for (int k = 0; k < ST_COUNT; ++k) s[k] += h->stats[r][k];
            nmax = fmax(nmax, h->stats[r][ST_NMAX]); nmin = fmin(nmin, h->stats[r][ST_NMIN]);
            emax = fmax(emax, h->stats[r][ST_EMAX]); emin = fmin(emin, h->stats[r][ST_EMIN]);
        }
        const float is_mean = ctrl->is_mean;      // written by this iteration's cn_is_weights_kernel (all ranks' rows)
        const float mean_w = !(use_is && per_step) ? 1.f : (batch_mode ? ctrl->mean_w : is_mean);
        const double nn = n_nom_global, ne = n_exp_global;
        const float expert_loss = (float)(s[ST_ELOG] / ne), unweighted = (float)(s[ST_NLOG] / nn);
        float nominal_loss, reg_loss, loss;
        if (gail) {
            nominal_loss = (float)(s[ST_NWLOG] / nn); reg_loss = 0.f;
            loss = nominal_loss + expert_loss;
        } else {
            nominal_loss = (use_is && per_step) ? mean_w * unweighted : (float)(s[ST_NWLOG] / nn);
            reg_loss = reg * ((float)(s[ST_E1MP] / ne) + (float)(s[ST_N1MP] / nn));
            loss = (-expert_loss + nominal_loss) + reg_loss;
        }
        float* m = ctrl->m;
        m[0] = loss; m[1] = expert_loss; m[2] = unweighted; m[3] = nominal_loss; m[4] = reg_loss;
        m[8] = (float)nmax; m[9] = (float)nmin; m[10] = (float)(s[ST_NSUM] / nn);
        m[11] = (float)emax; m[12] = (float)emin; m[13] = (float)(s[ST_ESUM] / ne);
        ctrl->steps_taken = step_index + 1;
    }
}

struct GradCall {           // the per-launch extras of cn_grad_kernel
    CnX x;
    unsigned int want1;
    double n_nom_global, n_exp_global;
    const int* idx;
};

template <typename ObsT, int HP>
static int launch_grad(const CnPlan& plan, CnCtrl* ctrl, const GradCall& gc, const void* nobs, const float* nacs, int64_t n_nom,
                       const void* eobs, const float* eacs, int64_t n_exp, const float* w, const icrl_cn_train_cfg& cfg,
                       int n_params, float** part_grad, float** part_stats, int* n_parts, cudaStream_t st) {
    auto kern = cn_grad_kernel<ObsT, HP>;
    int tile = 128;
    GradSmem L = grad_smem_layout(plan, HP, tile, sizeof(ObsT), n_params);
    while (L.total > 220 * 1024 && tile > 32) {
        tile /= 2;
        L = grad_smem_layout(plan, HP, tile, sizeof(ObsT), n_params);
    }
    if (L.total > 220 * 1024) {
        set_error("constraint net too large for the training kernel's shared memory (%d bytes)", L.total);
        return ICRL_EUNSUPPORTED;
    }
    ICRL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total));
    int per_sm = 1;
    ICRL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, tile, L.total));
    if (per_sm < 1) per_sm = 1;
    const int64_t tiles = (n_nom + tile - 1) / tile + (n_exp + tile - 1) / tile;
    const int64_t cap = (int64_t)per_sm * sm_count();
    const int grid = (int)(tiles < cap ? tiles : cap);
    int rc;
    void *pg, *ps;
    if ((rc = device_scratch(SLOT_WORK0, (size_t)grid * n_params * 4, &pg))) return rc;
    if ((rc = device_scratch(SLOT_WORK1, (size_t)grid * ST_COUNT * 4, &ps))) return rc;
    *part_grad = (float*)pg; *part_stats = (float*)ps; *n_parts = grid;
    const int tma_ok = ((reinterpret_cast<uintptr_t>(nobs) | reinterpret_cast<uintptr_t>(nacs) |
                         reinterpret_cast<uintptr_t>(eobs) | reinterpret_cast<uintptr_t>(eacs)) & 15u) == 0;
    const int per_step = cfg.per_step_is && cfg.importance_sampling;
    kern<<<grid, tile, L.total, st>>>(plan, ctrl, gc.x, gc.want1, per_step && !cfg.train_gail_lambda, (const ObsT*)nobs, nacs,
                                      n_nom, (const ObsT*)eobs, eacs, n_exp, gc.n_nom_global, gc.n_exp_global, gc.idx, w,
                                      per_step, cfg.train_gail_lambda, cfg.eps, cfg.regularizer_coeff, n_params, tma_ok,
                                      *part_grad, *part_stats);
    ICRL_LAUNCH_CHECK();
    return 0;
}

template <typename ObsT>
static int dispatch_grad(const CnPlan& plan, CnCtrl* ctrl, const GradCall& gc, const void* nobs, const float* nacs, int64_t n_nom,
                         const void* eobs, const float* eacs, int64_t n_exp, const float* w, const icrl_cn_train_cfg& cfg,
                         int n_params, float** pg, float** ps, int* np, cudaStream_t st) {
#define ICRL_GRAD_CASE(W) \
    case W: return launch_grad<ObsT, W>(plan, ctrl, gc, nobs, nacs, n_nom, eobs, eacs, n_exp, w, cfg, n_params, pg, ps, np, st)
    switch (cn_padded_width(plan)) {
        ICRL_GRAD_CASE(8); ICRL_GRAD_CASE(16); ICRL_GRAD_CASE(24); ICRL_GRAD_CASE(32);
        ICRL_GRAD_CASE(40); ICRL_GRAD_CASE(48); ICRL_GRAD_CASE(64);
    }
#undef ICRL_GRAD_CASE
    set_error("unsupported constraint-net width");
    return ICRL_EUNSUPPORTED;
}

}  // namespace icrl

static int cn_train_impl(const icrl_cn_desc* d, const icrl_cn_train_cfg* cfg, const void* nominal_obs,
                         int32_t nominal_obs_is_f64, const float* nominal_acs, int64_t n_nominal,
                         const int32_t* episode_offsets, int32_t n_episodes, const void* expert_obs,
                         int32_t expert_obs_is_f64, const float* expert_acs, int64_t n_expert, float* adam_m,
                         float* adam_v, int64_t* adam_step, icrl_cn_train_metrics* metrics, const icrl_cn_dist* dist,
                         void* stream) {
    using namespace icrl;
    CnPlan plan;
    int rc = make_plan(d, &plan);
    if (rc) return rc;
    ICRL_CHECK_ARG(cfg && metrics && adam_m && adam_v && adam_step, "NULL pointer passed to icrl_cn_train");
    ICRL_CHECK_ARG(n_nominal > 0 && n_expert > 0 && nominal_obs && nominal_acs && expert_obs && expert_acs,
                   "empty nominal or expert batch");
    ICRL_CHECK_ARG(nominal_obs_is_f64 == expert_obs_is_f64, "nominal and expert observations must share a dtype");
    ICRL_CHECK_ARG(!cfg->importance_sampling || (episode_offsets && n_episodes > 0), "importance sampling needs episodes");
    ICRL_CHECK_ARG(cfg->iterations >= 0, "iterations < 0");
    const bool batch_mode = cfg->batch_size > 0;
    ICRL_CHECK_ARG(!batch_mode || cfg->perm, "minibatch mode needs the host-drawn permutations (cfg->perm)");
    const bool dp = dist != nullptr && dist->world > 1;
    if (dp && batch_mode) {
        set_error("cn_batch_size (minibatch mode) is not available in data-parallel mode");
        return ICRL_EUNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int n_params = (int)cn_param_count(plan);
    const int use_is = cfg->importance_sampling ? 1 : 0;
    const int per_step = (cfg->per_step_is && use_is) ? 1 : 0;

    // global shapes (all ranks) and this rank's place in them
    double n_nom_global = (double)n_nominal, n_exp_global = (double)n_expert;
    int m_global = n_episodes, episode_base = 0;
    CnX x = {};
    x.rank = 0; x.world = 1; x.gstride = cn_gstride(n_params);
    unsigned int seq_base = 0;
    if (dist != nullptr) {
        ICRL_CHECK_ARG(dist->world >= 1 && dist->world <= ICRL_PPO_MAX_RANKS && dist->rank >= 0 && dist->rank < dist->world,
                       "bad rank/world (%d/%d)", dist->rank, dist->world);
        ICRL_CHECK_ARG(dist->n_nominal_global >= n_nominal && dist->n_expert_global >= n_expert &&
                           dist->n_episodes_global >= n_episodes && dist->episode_base >= 0 &&
                           dist->episode_base + n_episodes <= dist->n_episodes_global,
                       "global counts are smaller than this rank's share");
        ICRL_CHECK_ARG(dist->buffer_bytes >= (int64_t)cn_xchg_bytes(n_params, dist->n_episodes_global),
                       "exchange buffers too small (%lld bytes, need %lld: icrl_cn_dist_bytes)", (long long)dist->buffer_bytes,
                       (long long)cn_xchg_bytes(n_params, dist->n_episodes_global));
        x.rank = dist->rank; x.world = dist->world;
        for (int r = 0; r < dist->world; ++r) {
            ICRL_CHECK_ARG(dist->recv[r] != nullptr, "peer buffer %d is NULL", r);
            x.buf[r] = (unsigned char*)dist->recv[r];
        }
        n_nom_global = (double)dist->n_nominal_global; n_exp_global = (double)dist->n_expert_global;
        m_global = dist->n_episodes_global; episode_base = dist->episode_base;
        seq_base = dist->seq_base;
    }
    void *wbuf, *misc, *xbuf = nullptr, *pbuf;
    // work buffer: start_preds | cur_preds | w  (each n_nominal); misc: CnCtrl
    if ((rc = device_scratch(SLOT_WORK2, (size_t)3 * n_nominal * 4, &wbuf))) return rc;
    if ((rc = device_scratch(SLOT_WORK3, sizeof(CnCtrl), &misc))) return rc;
    const int is_grid = (int)std::min<int64_t>((n_nominal + 1023) / 1024, 2LL * sm_count());
    if ((rc = device_scratch(SLOT_WORK5, (size_t)is_grid * 4 * sizeof(double), &pbuf))) return rc;
    if (dist == nullptr) {
        const size_t xb = cn_xchg_bytes(n_params, m_global);
        if ((rc = device_scratch(SLOT_WORK4, xb, &xbuf))) return rc;
        ICRL_CUDA(cudaMemsetAsync(xbuf, 0, sizeof(CnXHeader), st));     // flags restart at zero every call
        x.buf[0] = (unsigned char*)xbuf;
    }
    float* start_preds = (float*)wbuf;
    float* cur_preds = start_preds + n_nominal;
    float* w = cur_preds + n_nominal;
    double* part = (double*)pbuf;
    CnCtrl* ctrl = (CnCtrl*)misc;
    CnCtrl init = {};
    init.early_stop_itr = cfg->iterations;
    init.mean_w = 1.f;
    init.is_mean = init.is_max = init.is_min = 1.f;
    ICRL_CUDA(cudaMemcpyAsync(ctrl, &init, sizeof(CnCtrl), cudaMemcpyHostToDevice, st));

    if (use_is) {   // start_preds (constraint_net.py:159-162)
        if ((rc = cn_forward_device(plan, nominal_obs, nominal_obs_is_f64, nominal_acs, n_nominal, start_preds, 1, st)))
            return rc;
    }
    float *part_grad = nullptr, *part_stats = nullptr;
    int n_parts = 0;
    const int64_t batch_set = std::min(n_nominal, n_expert);       // constraint_net.py:305
    const int mb_per_itr = batch_mode ? (int)((batch_set + cfg->batch_size - 1) / cfg->batch_size) : 1;
    const int pgrid = (n_params + 255) / 256;
    int step_index = 0;
    for (int itr = 0; itr < cfg->iterations; ++itr) {
        const unsigned int want01 = seq_base + (unsigned int)itr + 1u;
        if (use_is) {
            if (itr == 0) {
                ICRL_CUDA(cudaMemcpyAsync(cur_preds, start_preds, (size_t)n_nominal * 4, cudaMemcpyDeviceToDevice, st));
            } else if ((rc = cn_forward_device(plan, nominal_obs, nominal_obs_is_f64, nominal_acs, n_nominal, cur_preds, 1,
                                               st))) {
                return rc;   // (a stopped run still pays this forward; it is tiny and keeps the host free of syncs)
            }
            cn_is_partial_kernel<<<is_grid, 256, 0, st>>>(ctrl, x, start_preds, cur_preds, episode_offsets, n_episodes,
                                                          episode_base, (long long)n_nominal, cfg->eps, want01, part);
            ICRL_LAUNCH_CHECK();
        }
        cn_is_weights_kernel<<<is_grid, 256, 0, st>>>(ctrl, x, start_preds, cur_preds, episode_offsets, n_episodes,
                                                      episode_base, (long long)n_nominal, n_nom_global, m_global, cfg->eps,
                                                      use_is, per_step, cfg->target_kl_old_new, cfg->target_kl_new_old, itr,
                                                      want01, w, part);
        ICRL_LAUNCH_CHECK();
        for (int mb = 0; mb < mb_per_itr; ++mb, ++step_index) {
            GradCall gc;
            gc.x = x; gc.want1 = want01; gc.n_nom_global = n_nom_global; gc.n_exp_global = n_exp_global; gc.idx = nullptr;
            int64_t nn = n_nominal, ne = n_expert;
            if (batch_mode) {
                const int64_t b0 = (int64_t)mb * cfg->batch_size;
                const int64_t nb = std::min<int64_t>(cfg->batch_size, batch_set - b0);
                gc.idx = cfg->perm + (size_t)itr * batch_set + b0;
                gc.n_nom_global = gc.n_exp_global = (double)nb;
                nn = ne = nb;
                if (per_step && !cfg->train_gail_lambda) {
                    cn_batch_meanw_kernel<<<1, 256, 0, st>>>(ctrl, w, gc.idx, (int)nb);
                    ICRL_LAUNCH_CHECK();
                }
            }
            rc = nominal_obs_is_f64
                     ? dispatch_grad<double>(plan, ctrl, gc, nominal_obs, nominal_acs, nn, expert_obs, expert_acs, ne, w, *cfg,
                                             n_params, &part_grad, &part_stats, &n_parts, st)
                     : dispatch_grad<float>(plan, ctrl, gc, nominal_obs, nominal_acs, nn, expert_obs, expert_acs, ne, w, *cfg,
                                            n_params, &part_grad, &part_stats, &n_parts, st);
            if (rc) return rc;
            const unsigned int want2 = seq_base + (unsigned int)step_index + 1u;
            cn_reduce_kernel<<<(n_params + 7) / 8, 256, 0, st>>>(ctrl, x, part_grad, part_stats, n_parts, n_params, want2);
            ICRL_LAUNCH_CHECK();
            cn_adam_kernel<<<pgrid, 256, 0, st>>>(ctrl, x, const_cast<float*>(plan.params), adam_m, adam_v, n_params,
                                                  gc.n_nom_global, gc.n_exp_global, n_nom_global, use_is, per_step,
                                                  batch_mode ? 1 : 0, cfg->train_gail_lambda, cfg->regularizer_coeff, cfg->lr,
                                                  cfg->adam_beta1, cfg->adam_beta2, cfg->adam_eps,
                                                  (long long)*adam_step + step_index + 1, step_index, want2);
            ICRL_LAUNCH_CHECK();
        }
    }
    CnCtrl out;
    ICRL_CUDA(cudaMemcpyAsync(&out, ctrl, sizeof(CnCtrl), cudaMemcpyDeviceToHost, st));
    ICRL_CUDA(cudaStreamSynchronize(st));
    if (out.error) {
        set_error("constraint-net training: an exchange wait timed out (a data-parallel rank did not deliver its partial sums)");
        return ICRL_EPEER;
    }
    *adam_step += out.steps_taken;
    metrics->cn_loss = out.m[0]; metrics->expert_loss = out.m[1]; metrics->unweighted_nominal_loss = out.m[2];
    metrics->nominal_loss = out.m[3]; metrics->regularizer_loss = out.m[4];
    metrics->is_mean = out.is_mean; metrics->is_max = out.is_max; metrics->is_min = out.is_min;
    metrics->nominal_preds_max = out.m[8]; metrics->nominal_preds_min = out.m[9]; metrics->nominal_preds_mean = out.m[10];
    metrics->expert_preds_max = out.m[11]; metrics->expert_preds_min = out.m[12]; metrics->expert_preds_mean = out.m[13];
    metrics->kl_old_new = out.kl_old_new; metrics->kl_new_old = out.kl_new_old;
    metrics->early_stop_itr = out.early_stop_itr; metrics->steps_taken = out.steps_taken;
    return 0;
}

extern "C" {

int64_t icrl_cn_dist_bytes(const icrl_cn_desc* d, int32_t n_episodes_global) {
    icrl::CnPlan plan;
    if (icrl::make_plan(d, &plan) != 0) return -1;
    return (int64_t)icrl::cn_xchg_bytes((int)icrl::cn_param_count(plan), n_episodes_global);
}

int icrl_cn_train(const icrl_cn_desc* d, const icrl_cn_train_cfg* cfg, const void* nominal_obs, int32_t nominal_obs_is_f64,
                  const float* nominal_acs, int64_t n_nominal, const int32_t* episode_offsets, int32_t n_episodes,
                  const void* expert_obs, int32_t expert_obs_is_f64, const float* expert_acs, int64_t n_expert, float* adam_m,
                  float* adam_v, int64_t* adam_step, icrl_cn_train_metrics* metrics, void* stream) {
    return cn_train_impl(d, cfg, nominal_obs, nominal_obs_is_f64, nominal_acs, n_nominal, episode_offsets, n_episodes,
                         expert_obs, expert_obs_is_f64, expert_acs, n_expert, adam_m, adam_v, adam_step, metrics, nullptr,
                         stream);
}

int icrl_cn_train_dist(const icrl_cn_desc* d, const icrl_cn_train_cfg* cfg, const void* nominal_obs,
                       int32_t nominal_obs_is_f64, const float* nominal_acs, int64_t n_nominal,
                       const int32_t* episode_offsets, int32_t n_episodes, const void* expert_obs, int32_t expert_obs_is_f64,
                       const float* expert_acs, int64_t n_expert, float* adam_m, float* adam_v, int64_t* adam_step,
                       icrl_cn_train_metrics* metrics, const icrl_cn_dist* dist, void* stream) {
    ICRL_CHECK_ARG(dist != nullptr, "dist is NULL");
    return cn_train_impl(d, cfg, nominal_obs, nominal_obs_is_f64, nominal_acs, n_nominal, episode_offsets, n_episodes,
                         expert_obs, expert_obs_is_f64, expert_acs, n_expert, adam_m, adam_v, adam_step, metrics, dist,
                         stream);
}

}  // extern "C"
