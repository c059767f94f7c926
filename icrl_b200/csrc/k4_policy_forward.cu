// Policy forward for rollout collection / evaluation (policies.py:716-731 without sampling): action mean or logits, reward
// value and cost value of every row.  grid = (row chunks, 3 trunks); each CTA keeps its trunk in shared memory and walks
// 64-row chunks with FP32 FFMA register tiles (4x4 outputs per thread, float4 broadcast operand reads).
#include "k4_common.cuh"

namespace icrl {

struct FwdSmem { int w1t, w2t, b1, b2, hw, hb, x, h1, h2, total_bytes; };
__host__ __device__ inline FwdSmem fwd_smem_layout(int DP4) {
    FwdSmem s;
    int o = 0;
    s.w1t = o; o += DP4 * H;
    s.w2t = o; o += H * H;
    s.b1 = o; o += H;
    s.b2 = o; o += H;
    s.hw = o; o += AMAX * WA_LD;
    s.hb = o; o += AMAX;
    s.x = o; o += RB * DP4;
    s.h1 = o; o += RB * H;
    s.h2 = o; o += RB * H;
    s.total_bytes = o * 4;
    return s;
}

// 64x64 += A[64 x K] * Bt[K x 64]  (A row-major lda, Bt k-major ld 64); thread tile rows 4ty.., cols 4tx..
// KC > 0: compile-time K (fully unrolled so operand loads run ahead of the FMAs); KC == 0: runtime K.
// SWZ: Bt's float4 column slots are XOR-swizzled with (k >> 2) & 15 (the W2t copy: lets the Adam phase write the
// transposed tile with conflict-free 128-bit stores while these row reads stay conflict-free).
template <int KC, bool SWZ = false>
__device__ __forceinline__ void gemm_tile_4x4(float (&acc)[4][4], const float* __restrict__ A, int lda,
                                              const float* __restrict__ Bt, int K, int ty, int tx) {
    const float* a0 = A + (4 * ty) * lda;
    const float* b0 = Bt + 4 * tx;
    const int kend = KC > 0 ? KC : K;
#pragma unroll (KC > 0 ? KC / 4 : 2)
    for (int k = 0; k < kend; k += 4) {
        float4 a[4], w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4*>(a0 + i * lda + k);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
            w[kk] = SWZ ? *reinterpret_cast<const float4*>(Bt + (k + kk) * H + 4 * (tx ^ ((k >> 2) & 15)))
                        : *reinterpret_cast<const float4*>(b0 + (k + kk) * H);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float av = kk == 0 ? a[i].x : kk == 1 ? a[i].y : kk == 2 ? a[i].z : a[i].w;
                acc[i][0] = fmaf(av, w[kk].x, acc[i][0]);
                acc[i][1] = fmaf(av, w[kk].y, acc[i][1]);
                acc[i][2] = fmaf(av, w[kk].z, acc[i][2]);
                acc[i][3] = fmaf(av, w[kk].w, acc[i][3]);
            }
        }
    }
}

// grid = (row chunks, 3 trunks).  Each CTA keeps its trunk in shared memory and walks 64-row chunks.
__global__ void __launch_bounds__(NTH) policy_forward_kernel(const __grid_constant__ PpoArgs a, const float* __restrict__ obs,
                                                             long long n, float* __restrict__ head,
                                                             float* __restrict__ values, float* __restrict__ cost_values) {
    extern __shared__ __align__(16) float sm[];
    const int DP = (a.D + 3) / 4 * 4;
    const FwdSmem L = fwd_smem_layout(DP);
    const int tid = threadIdx.x, trunk = blockIdx.y, D = a.D;
    const int AOUT = trunk == 0 ? a.A : 1;
    const int h0 = a.h0[trunk], h1 = a.h1[trunk];
    float* W1t = sm + L.w1t; float* W2t = sm + L.w2t; float* B1 = sm + L.b1; float* B2 = sm + L.b2;
    float* HW = sm + L.hw; float* HB = sm + L.hb; float* X = sm + L.x; float* H1 = sm + L.h1; float* H2 = sm + L.h2;
    for (int i = tid; i < DP * H; i += NTH) {
        const int k = i / H, j = i - k * H;
        W1t[i] = (k < D && j < h0) ? a.params[a.off_w1[trunk] + j * D + k] : 0.f;
    }
    for (int i = tid; i < H * H; i += NTH) {
        const int k = i / H, j = i - k * H;
        W2t[i] = (k < h0 && j < h1) ? a.params[a.off_w2[trunk] + j * h0 + k] : 0.f;
    }
    for (int i = tid; i < AMAX * WA_LD; i += NTH) {
        const int d = i / WA_LD, k = i - d * WA_LD;
        HW[i] = (d < AOUT && k < h1) ? a.params[a.off_hw[trunk] + d * h1 + k] : 0.f;
    }
    if (tid < H) {
        B1[tid] = tid < h0 ? a.params[a.off_b1[trunk] + tid] : 0.f;
        B2[tid] = tid < h1 ? a.params[a.off_b2[trunk] + tid] : 0.f;
    }
    if (tid < AMAX) HB[tid] = tid < AOUT ? a.params[a.off_hb[trunk] + tid] : 0.f;
    const int ty = tid >> 4, tx = tid & 15, hr = tid >> 2, hq = tid & 3;
    const long long n_chunks = (n + RB - 1) / RB;
    for (long long c = blockIdx.x; c < n_chunks; c += gridDim.x) {
        const long long row0 = c * RB;
        const int rows = (int)min((long long)RB, n - row0);
        __syncthreads();
        for (int i = tid; i < RB * DP; i += NTH) {
            const int r = i / DP, k = i - r * DP;
            X[i] = (r < rows && k < D) ? obs[(row0 + r) * D + k] : 0.f;
        }
        __syncthreads();
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = B1[4 * tx + j];
        gemm_tile_4x4<0>(acc, X, DP, W1t, DP, ty, tx);
#pragma unroll
        for (int i = 0; i < 4; ++i)
            *reinterpret_cast<float4*>(H1 + (4 * ty + i) * H + 4 * tx) =
                make_float4(tanhf(acc[i][0]), tanhf(acc[i][1]), tanhf(acc[i][2]), tanhf(acc[i][3]));
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = B2[4 * tx + j];
        gemm_tile_4x4<H>(acc, H1, H, W2t, H, ty, tx);
#pragma unroll
        for (int i = 0; i < 4; ++i)
            *reinterpret_cast<float4*>(H2 + (4 * ty + i) * H + 4 * tx) =
                make_float4(tanhf(acc[i][0]), tanhf(acc[i][1]), tanhf(acc[i][2]), tanhf(acc[i][3]));
        __syncthreads();
        for (int u = 0; u < 4; ++u) {
            const int d = hq + 4 * u;
            if (d < AOUT && hr < rows) {
                float o = HB[d];
                const float4* hrow = reinterpret_cast<const float4*>(H2 + hr * H);
                const float4* wrow = reinterpret_cast<const float4*>(HW + d * WA_LD);
#pragma unroll
                for (int k = 0; k < H / 4; ++k) {
                    const float4 h = hrow[k], w = wrow[k];
                    o = fmaf(h.x, w.x, o); o = fmaf(h.y, w.y, o); o = fmaf(h.z, w.z, o); o = fmaf(h.w, w.w, o);
                }
                if (trunk == 0) head[(row0 + hr) * a.A + d] = o;
                else if (trunk == 1) values[row0 + hr] = o;
                else cost_values[row0 + hr] = o;
            }
        }
    }
}


}  // namespace icrl

extern "C" int icrl_policy_forward(const icrl_ppo_cfg* cfg, const float* params, const float* obs, int64_t n, float* head,
                        float* values, float* cost_values, void* stream) {
    icrl::PpoArgs a = {};
    icrl_ppo_cfg c = *cfg;
    if (c.T <= 0) c.T = 1;
    if (c.E <= 0) c.E = 1;
    int rc = icrl::ppo_make_args(&c, a);
    if (rc) return rc;
    if (n == 0) return 0;
    ICRL_CHECK_ARG(params && obs && head && values && cost_values && n > 0, "NULL pointer passed to icrl_policy_forward");
    a.params = const_cast<float*>(params);
    const icrl::FwdSmem L = icrl::fwd_smem_layout((a.D + 3) / 4 * 4);
    ICRL_CUDA(cudaFuncSetAttribute(icrl::policy_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total_bytes));
    const int64_t chunks = (n + icrl::RB - 1) / icrl::RB;
    const int gx = (int)(chunks < icrl::sm_count() ? chunks : icrl::sm_count());
    icrl::policy_forward_kernel<<<dim3(gx, 3), icrl::NTH, L.total_bytes, (cudaStream_t)stream>>>(a, obs, n, head, values,
                                                                                                cost_values);
    ICRL_LAUNCH_CHECK();
    return 0;
}

