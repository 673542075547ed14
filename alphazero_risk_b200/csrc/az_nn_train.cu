// az_nn_train.cu — the training step of the policy/value network and TensorFlow-checkpoint exchange (SURVEY §8f N4).
//
// Reference: AlphaZeroNN::train (neural_network/alphazero_nn.cpp:351-410) runs, per batch of SETTINGS.BATCH_SIZE samples, the graph's
// "optimize" op with input_training = true; the graph is python/src/build_graph.py:54-106.  What that op computes (constants read from
// the shipped GraphDef python/model/model_txt_V2_5.pb, see oracle/nn_oracle.py for the restatement this file is checked against):
//   forward with FusedBatchNormV3(is_training = true): batch mean / biased batch variance, epsilon 0.001; moving statistics move to the
//   batch mean and the unbiased batch variance with momentum 0.99; the stem's BatchNorm runs over the board-row axis (7 groups);
//   loss = softmax cross-entropy(policy logits, target pi) [batch mean] + mean squared error(tanh value, target z) + 0.001 * sum of the
//   squared kernels (a six-output value head, SIXPLAYER.md §2: the mean over all n * 6 squared errors); Adam(lr 0.001, beta1 0.9, beta2 0.999, epsilon 1e-8) in TensorFlow's formulation.
// AlphaZeroNN::saveCheckpoint / loadCheckpoint (alphazero_nn.cpp:189-214) exchange the 163 tensors of the graph's Saver: variables, BN
// moving statistics, Adam slots "<var>/optimize" (m) and "<var>/optimize_1" (v), beta1_power, beta2_power (az_ckpt.cpp holds the format).
//
// Everything here is fp32 on CUDA cores: a training step is 3x the forward FLOPs on a batch of 512 and runs a few times per thousand
// self-play games, it is not on the self-play hot path.  Activations [rows = boards * 42][256 channels] row-major, as in az_nn.cu.
//   forward   k_tr_conv (raw 3x3 convolution, also used for the data gradient with the flipped + transposed kernel) ->
//             k_tr_stats / k_tr_stats_final (batch statistics, double accumulation, fixed reduction order) -> k_tr_bn_apply (+skip, ReLU)
//   heads     1x1 convolutions, 3-channel batch statistics, one block per board for the dense layers + losses + their backward
//   backward  k_tr_bwd_stats (sum g, sum g*xhat with g = dOut * [a > 0]) -> k_tr_bn_bwd (dz) -> k_tr_wgrad (split over boards, partials
//             reduced in a fixed order) and k_tr_conv (data gradient)
//   update    k_tr_adam per trainable variable (L2 term added to the kernels' gradients)
// Results are deterministic: no floating-point atomics anywhere.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "az_common.cuh"
#include "az_nn.cuh"
#include "az_samples6.cuh"
#include "az_tc_gemm.cuh"

#define TR_CH AZ_NN_CH
#define TR_BN_MOMENTUM 0.99f
#define TR_L2 0.001f
#define TR_LR 0.001f
#define TR_BETA1 0.9f
#define TR_BETA2 0.999f
#define TR_ADAM_EPS 1e-8f
#define TR_STAT_CHUNKS 296         // row chunks of the column reductions (2 per SM)
#define TR_WG_SPLITS 16            // board splits of the weight-gradient reduction

static inline size_t tr_mp(int rows) { return ((size_t)rows + 127) / 128 * 128; }     // rows of a GEMM output, 128-row tiles
static inline size_t tr_kp(int k) { return ((size_t)k + 63) / 64 * 64; }            // K of a GEMM, 64-element blocks

struct az_ckpt;
extern "C" int az_ckpt_open(const char* prefix, az_ckpt** out);
extern "C" int az_ckpt_close(az_ckpt* c);
extern "C" int az_ckpt_find(const az_ckpt* c, const char* name);
extern "C" int az_ckpt_tensor_info(const az_ckpt* c, int i, const char** name, int* dtype, int* rank, int64_t* shape8, size_t* bytes);
extern "C" int az_ckpt_read(az_ckpt* c, const char* name, void* h_out, size_t bytes);
extern "C" int az_ckpt_write(const char* prefix, int n, const char* const* names, const int* ranks, const int64_t* const* shapes,
                             const float* const* data);
int az_nn_sync_host(az_nn* nn);      // az_nn.cu

struct AzTrainState {
    int cap = 0;                                       // boards the work buffers are sized for
    bool dz_prepared = false;                          // the current layer's dz sits converted in conv.d_in3 (weight gradient done, data gradient next)
    int precision = AZ_NN_FP32;                        // AZ_NN_BF16: the three contractions run on the tensor cores (az_tc_gemm.cu)
    __nv_bfloat16 *d_colA = nullptr, *d_colB = nullptr;   // GEMM operands: im2col / transposed im2col, weights / transposed gradient
    AzTcConvScratch conv;                              // 256-channel convolutions of the tensor-core mode run on the tower kernel
    uint8_t* d_kind = nullptr;                         // per blob element: 0 not trainable, 1 plain, 2 kernel (L2 term)
    __nv_bfloat16* d_src16 = nullptr;                  // bf16 chunked copy of the tensor being unrolled
    float *d_grad = nullptr, *d_m = nullptr, *d_v = nullptr;      // blob-sized: gradient of the total loss, Adam slots
    std::vector<float> h_m, h_v;                       // host mirrors (checkpoints)
    bool slots_on_device = false, host_slots_stale = false;
    float beta1_power = TR_BETA1, beta2_power = TR_BETA2;
    uint64_t steps = 0;
    float* d_x = nullptr;                              // [cap][42][input_planes]
    std::vector<float*> z, a;                          // per conv layer (0 = stem, 1 + 2i / 2 + 2i = block i): raw output, activation
    float* d_stats = nullptr;                          // [layers + 2][4][256]: mean, invstd, c1 = sum(g)/N, c2 = sum(g*xhat)/N
    double* d_part = nullptr;                          // [TR_STAT_CHUNKS][256][2]
    float* d_g[3] = { nullptr, nullptr, nullptr };     // gradient buffers [cap][42][256]
    float* d_wT = nullptr;                             // [9][256][256] flipped + transposed kernel of the layer being back-propagated
    float* d_wpart = nullptr;                          // [TR_WG_SPLITS][9][256][256]
    float *d_hz = nullptr, *d_hg = nullptr;            // heads: raw 1x1 outputs / gradients [cap*42][4] (pi0, pi1, v, unused)
    float *d_hfeat = nullptr;                          // per board: s_pi[84] dlogit[43] s_v[42] h[256] dh[256] dout[vo <= 6] loss[2]
    float *d_hpart = nullptr;                          // [TR_STAT_CHUNKS][256][3] 1x1 kernel gradient partials
    float *d_tp = nullptr, *d_tv = nullptr, *d_loss = nullptr;   // d_tv: [cap][value outputs]
};
#define HF_STRIDE 696
#define HF_SPI 0
#define HF_DLOGIT 84
#define HF_SV 128
#define HF_H 172
#define HF_DH 428
#define HF_DOUT 684      // [vo]
#define HF_LOSS 690

__constant__ int8_t c_tnb[42 * 9];       // neighbour of board cell p for tap t, -1 outside the board (SAME padding)

// ---------------------------------------------------------------- convolution (forward and data gradient)
// out[r][co] = sum_t sum_ci in[nb(r, t)][ci] * w[t][ci][co], raw (no BN).  Block = 4 boards x 64 output channels, 128 threads,
// thread = 21 rows x 4 channels, input channels in chunks of 32 (same tiling as k_nn_conv_fp32).
#define TC_BOARDS 4
#define TC_ROWS (TC_BOARDS * 42)
#define TC_CO 64
#define TC_CI 32
#define TC_SMEM_FLOATS ((TC_ROWS + 1) * TC_CI + 9 * TC_CI * TC_CO)

__global__ void __launch_bounds__(128) k_tr_conv(const float* __restrict__ in, int n, int cin, const float* __restrict__ w, float* __restrict__ out)
{
    extern __shared__ float sm[];
    float* s_in = sm;
    float* s_w = sm + (TC_ROWS + 1) * TC_CI;
    const int b0 = blockIdx.x * TC_BOARDS, co0 = blockIdx.y * TC_CO;
    const int cg = threadIdx.x & 15, rg = threadIdx.x >> 4;
    const int rows_valid = min(TC_BOARDS, n - b0) * 42;
    float acc[21][4];
#pragma unroll
    for (int j = 0; j < 21; ++j) { acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.0f; }
    if (threadIdx.x < TC_CI) s_in[TC_ROWS * TC_CI + threadIdx.x] = 0.0f;
    for (int c0 = 0; c0 < cin; c0 += TC_CI) {
        __syncthreads();
        for (int i = threadIdx.x; i < TC_ROWS * TC_CI; i += 128) {
            int r = i / TC_CI, ci = i - r * TC_CI;
            s_in[i] = (r < rows_valid && c0 + ci < cin) ? in[((size_t)b0 * 42 + r) * cin + c0 + ci] : 0.0f;
        }
        for (int i = threadIdx.x; i < 9 * TC_CI * TC_CO; i += 128) {
            int t = i / (TC_CI * TC_CO), rem = i - t * (TC_CI * TC_CO), ci = rem / TC_CO, co = rem - ci * TC_CO;
            s_w[i] = c0 + ci < cin ? w[((size_t)t * cin + c0 + ci) * TR_CH + co0 + co] : 0.0f;
        }
        __syncthreads();
        for (int t = 0; t < 9; ++t) {
            int src[21];
#pragma unroll
            for (int j = 0; j < 21; ++j) {
                int r = rg * 21 + j, bi = r / 42, p = r - bi * 42;
                int q = c_tnb[p * 9 + t];
                src[j] = (q < 0 ? TC_ROWS : bi * 42 + q) * TC_CI;
            }
            const float* wt = s_w + t * TC_CI * TC_CO + cg * 4;
#pragma unroll 4
            for (int ci = 0; ci < TC_CI; ++ci) {
                float4 w4 = *reinterpret_cast<const float4*>(wt + ci * TC_CO);
#pragma unroll
                for (int j = 0; j < 21; ++j) {
                    float av = s_in[src[j] + ci];
                    acc[j][0] = fmaf(av, w4.x, acc[j][0]); acc[j][1] = fmaf(av, w4.y, acc[j][1]);
                    acc[j][2] = fmaf(av, w4.z, acc[j][2]); acc[j][3] = fmaf(av, w4.w, acc[j][3]);
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 21; ++j) {
        int r = rg * 21 + j;
        if (r < rows_valid)
            *reinterpret_cast<float4*>(out + ((size_t)b0 * 42 + r) * TR_CH + co0 + cg * 4) = make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]);
    }
}

// wT[t][co][ci] = w[8 - t][ci][co]: the data gradient of a SAME 3x3 convolution is the convolution of dz with this kernel
__global__ void k_tr_flip_transpose(const float* __restrict__ w, float* __restrict__ wT)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 9 * TR_CH * TR_CH) return;
    int t = i / (TR_CH * TR_CH), rem = i - t * TR_CH * TR_CH, co = rem / TR_CH, ci = rem - co * TR_CH;
    wT[i] = w[((size_t)(8 - t) * TR_CH + ci) * TR_CH + co];
}

// ---------------------------------------------------------------- batch statistics (column reductions)
// mode 0: sum z, sum z^2           (forward statistics)
// mode 1: sum g, sum g * xhat      (backward), g = dout * [a > 0], xhat = (z - mean) * invstd
// stem = 1: the statistic group of element (r, c) is the board row y = (r % 42) / 6 instead of the channel c.
// grid = TR_STAT_CHUNKS blocks of 256 threads = 64 channel quads (16-byte loads) x 4 row lanes; partials in double, the row lanes are
// combined in lane order here and the chunks in chunk order by k_tr_stats_final.  (The stem variant keeps thread = channel.)
__global__ void __launch_bounds__(256) k_tr_stats(const float* __restrict__ z, const float* __restrict__ dout, const float* __restrict__ a,
                                                   const float* __restrict__ stats, int rows, int mode, int stem, double* __restrict__ part)
{
    __shared__ double s_red[8][7][2];
    __shared__ double s_lane[3][TR_CH][2];
    const int c = threadIdx.x, chunk = blockIdx.x;
    const int per = ((rows / 42 + TR_STAT_CHUNKS - 1) / TR_STAT_CHUNKS) * 42;           // whole boards per chunk
    const int r0 = min(rows, chunk * per), r1 = min(rows, r0 + per);
    if (!stem) {
        const int cq = threadIdx.x & 63, rl = threadIdx.x >> 6;
        double s0[4] = { 0.0, 0.0, 0.0, 0.0 }, s1[4] = { 0.0, 0.0, 0.0, 0.0 };
        float mean[4] = { 0, 0, 0, 0 }, inv[4] = { 0, 0, 0, 0 };
        if (mode) {
#pragma unroll
            for (int e = 0; e < 4; ++e) { mean[e] = stats[cq * 4 + e]; inv[e] = stats[TR_CH + cq * 4 + e]; }
        }
#pragma unroll 2
        for (int r = r0 + rl; r < r1; r += 4) {
            const size_t o = (size_t)r * TR_CH + cq * 4;
            const float4 zv = *reinterpret_cast<const float4*>(z + o);
            const float zz[4] = { zv.x, zv.y, zv.z, zv.w };
            if (mode == 0) {
#pragma unroll
                for (int e = 0; e < 4; ++e) { s0[e] += (double)zz[e]; s1[e] += (double)zz[e] * (double)zz[e]; }
            } else {
                const float4 av = *reinterpret_cast<const float4*>(a + o), dv = *reinterpret_cast<const float4*>(dout + o);
                const float aa[4] = { av.x, av.y, av.z, av.w }, dd[4] = { dv.x, dv.y, dv.z, dv.w };
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float g = aa[e] > 0.0f ? dd[e] : 0.0f;
                    s0[e] += (double)g; s1[e] += (double)g * (double)((zz[e] - mean[e]) * inv[e]);
                }
            }
        }
        if (rl > 0) {
#pragma unroll
            for (int e = 0; e < 4; ++e) { s_lane[rl - 1][cq * 4 + e][0] = s0[e]; s_lane[rl - 1][cq * 4 + e][1] = s1[e]; }
        }
        __syncthreads();
        if (rl == 0) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                double v0 = s0[e], v1 = s1[e];
                for (int l = 0; l < 3; ++l) { v0 += s_lane[l][cq * 4 + e][0]; v1 += s_lane[l][cq * 4 + e][1]; }
                part[((size_t)chunk * TR_CH + cq * 4 + e) * 2 + 0] = v0; part[((size_t)chunk * TR_CH + cq * 4 + e) * 2 + 1] = v1;
            }
        }
    } else {
        double s0[7], s1[7];
#pragma unroll
        for (int y = 0; y < 7; ++y) { s0[y] = 0.0; s1[y] = 0.0; }
        for (int b = r0; b < r1; b += 42) {
#pragma unroll
            for (int y = 0; y < 7; ++y) {
                const float mean = mode ? stats[y] : 0.0f, inv = mode ? stats[TR_CH + y] : 0.0f;
#pragma unroll
                for (int x = 0; x < 6; ++x) {
                    const size_t o = (size_t)(b + y * 6 + x) * TR_CH + c;
                    if (mode == 0) { const float v = z[o]; s0[y] += (double)v; s1[y] += (double)v * (double)v; }
                    else { const float g = a[o] > 0.0f ? dout[o] : 0.0f; s0[y] += (double)g; s1[y] += (double)g * (double)((z[o] - mean) * inv); }
                }
            }
        }
        // reduce the 256 channels of the block in a fixed order: warp shuffles, then warp 0 over the 8 warp sums
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
        for (int y = 0; y < 7; ++y) {
            double v0 = s0[y], v1 = s1[y];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { v0 += __shfl_xor_sync(0xffffffffu, v0, o); v1 += __shfl_xor_sync(0xffffffffu, v1, o); }
            if (lane == 0) { s_red[warp][y][0] = v0; s_red[warp][y][1] = v1; }
        }
        __syncthreads();
        if (threadIdx.x < 7) {
            double v0 = 0.0, v1 = 0.0;
            for (int w8 = 0; w8 < 8; ++w8) { v0 += s_red[w8][threadIdx.x][0]; v1 += s_red[w8][threadIdx.x][1]; }
            part[((size_t)chunk * TR_CH + threadIdx.x) * 2 + 0] = v0; part[((size_t)chunk * TR_CH + threadIdx.x) * 2 + 1] = v1;
        }
    }
}

// mode 0: mean, invstd into stats[0..1], moving statistics updated (FusedBatchNormV3 training outputs + AssignMovingAvg)
// mode 1: c1 = sum(g)/N, c2 = sum(g*xhat)/N into stats[2..3]; dgamma = sum(g*xhat), dbeta = sum(g) into the gradient blob
__global__ void __launch_bounds__(256) k_tr_stats_final(const double* __restrict__ part, int groups, double count, int mode, float* __restrict__ stats,
                                                         float* __restrict__ moving_mean, float* __restrict__ moving_var,
                                                         float* __restrict__ dgamma, float* __restrict__ dbeta)
{
    // grid = 8 blocks of 32 groups; 256 threads = 8 chunk lanes x 32 groups; each lane sums its chunks in order, then the lanes in order
    __shared__ double s_q[7][32][2];
    const int cl = threadIdx.x & 31, q = threadIdx.x >> 5, c = blockIdx.x * 32 + cl;
    double s0 = 0.0, s1 = 0.0;
    constexpr int QN = TR_STAT_CHUNKS / 8;
    static_assert(TR_STAT_CHUNKS % 8 == 0, "chunk count must split into eight lanes");
    if (c < groups) {
#pragma unroll 8
        for (int k = q * QN; k < (q + 1) * QN; ++k) { s0 += part[((size_t)k * TR_CH + c) * 2 + 0]; s1 += part[((size_t)k * TR_CH + c) * 2 + 1]; }
    }
    if (q > 0) { s_q[q - 1][cl][0] = s0; s_q[q - 1][cl][1] = s1; }
    __syncthreads();
    if (q > 0 || c >= groups) return;
    for (int l = 0; l < 7; ++l) { s0 += s_q[l][cl][0]; s1 += s_q[l][cl][1]; }
    if (mode == 0) {
        const double mean = s0 / count;
        double var = s1 / count - mean * mean; if (var < 0.0) var = 0.0;
        stats[c] = (float)mean; stats[TR_CH + c] = (float)(1.0 / sqrt(var + (double)AZ_NN_BN_EPS));
        const float mm = moving_mean[c], mv = moving_var[c];
        moving_mean[c] = mm - (mm - (float)mean) * (1.0f - TR_BN_MOMENTUM);
        moving_var[c] = mv - (mv - (float)(var * count / (count - 1.0))) * (1.0f - TR_BN_MOMENTUM);
    } else {
        stats[2 * TR_CH + c] = (float)(s0 / count); stats[3 * TR_CH + c] = (float)(s1 / count);
        dgamma[c] = (float)s1; dbeta[c] = (float)s0;
    }
}

// a = relu(gamma * (z - mean) * invstd + beta [+ skip])
__global__ void __launch_bounds__(256) k_tr_bn_apply(const float* __restrict__ z, const float* __restrict__ stats, const float* __restrict__ gamma,
                                                      const float* __restrict__ beta, const float* __restrict__ skip, float* __restrict__ a,
                                                      size_t total, int stem)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = (int)(i % TR_CH);
    const int grp = stem ? (int)((i / TR_CH) % 42) / 6 : c;
    float v = (z[i] - stats[grp]) * stats[TR_CH + grp] * gamma[grp] + beta[grp];
    if (skip) v += skip[i];
    a[i] = v > 0.0f ? v : 0.0f;
}

// dz = gamma * invstd * (g - c1 - xhat * c2), g = dout * [a > 0]
__global__ void __launch_bounds__(256) k_tr_bn_bwd(const float* __restrict__ z, const float* __restrict__ dout, const float* __restrict__ a,
                                                    const float* __restrict__ stats, const float* __restrict__ gamma, float* __restrict__ dz,
                                                    size_t total, int stem)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = (int)(i % TR_CH);
    const int grp = stem ? (int)((i / TR_CH) % 42) / 6 : c;
    const float inv = stats[TR_CH + grp];
    const float g = a[i] > 0.0f ? dout[i] : 0.0f;
    const float xh = (z[i] - stats[grp]) * inv;
    dz[i] = gamma[grp] * inv * (g - stats[2 * TR_CH + grp] - xh * stats[3 * TR_CH + grp]);
}

// dst += dout * [a > 0]   (the skip connection's share of a block's input gradient)
__global__ void __launch_bounds__(256) k_tr_add_masked(float* __restrict__ dst, const float* __restrict__ dout, const float* __restrict__ a, size_t total)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < total && a[i] > 0.0f) dst[i] += dout[i];
}

// ---------------------------------------------------------------- tensor-core mode: BatchNorm passes that also emit the bf16 operands
// Block = 32 rows x 256 channels, thread = (row, 8-channel chunk) four times over; the chunk values go through shared memory so that the
// chunked bf16 board layout of the tower kernel ([chunk][AZ_TC_HALO + board * AZ_TC_RPB + cell][8]) is written in contiguous runs.
__device__ __forceinline__ void ld8(const float* __restrict__ p, float (&v)[8])
{
    const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p + 4));
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
// k_tr_bn_apply_rpb: a = relu(gamma * (z - mean) * invstd + beta [+ skip]) as fp32 AND as the next convolution's operand.
__global__ void __launch_bounds__(256) k_tr_bn_apply_rpb(const float* __restrict__ z, const float* __restrict__ stats, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, const float* __restrict__ skip, float* __restrict__ a,
                                                        int rows, int stem, __nv_bfloat16* __restrict__ a_rpb, int r_alloc)
{
    __shared__ uint4 tile[32][33];
    const int r0 = blockIdx.x * 32;
    for (int j = threadIdx.x; j < 1024; j += 256) {
        const int rl = j >> 5, cc = j & 31, r = r0 + rl;
        if (r < rows) {
            const size_t o = (size_t)r * TR_CH + cc * 8;
            const float4 z0 = *reinterpret_cast<const float4*>(z + o), z1 = *reinterpret_cast<const float4*>(z + o + 4);
            float v[8] = { z0.x, z0.y, z0.z, z0.w, z1.x, z1.y, z1.z, z1.w };
            if (stem) {
                const int grp = (r % 42) / 6;
                const float mu = stats[grp], inv = stats[TR_CH + grp], ga = gamma[grp], be = beta[grp];
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = (v[e] - mu) * inv * ga + be;
            } else {
                float mu[8], inv[8], ga[8], be[8];
                ld8(stats + cc * 8, mu); ld8(stats + TR_CH + cc * 8, inv); ld8(gamma + cc * 8, ga); ld8(beta + cc * 8, be);
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = (v[e] - mu[e]) * inv[e] * ga[e] + be[e];
            }
            if (skip) {
                const float4 s0 = *reinterpret_cast<const float4*>(skip + o), s1 = *reinterpret_cast<const float4*>(skip + o + 4);
                v[0] += s0.x; v[1] += s0.y; v[2] += s0.z; v[3] += s0.w; v[4] += s1.x; v[5] += s1.y; v[6] += s1.z; v[7] += s1.w;
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] = v[e] > 0.0f ? v[e] : 0.0f;
            *reinterpret_cast<float4*>(a + o) = make_float4(v[0], v[1], v[2], v[3]);
            *reinterpret_cast<float4*>(a + o + 4) = make_float4(v[4], v[5], v[6], v[7]);
            uint4 pk;
            __nv_bfloat162* p2 = reinterpret_cast<__nv_bfloat162*>(&pk);
#pragma unroll
            for (int e = 0; e < 4; ++e) p2[e] = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
            tile[rl][cc] = pk;
        }
    }
    __syncthreads();
    uint4* o4 = reinterpret_cast<uint4*>(a_rpb);
    for (int j = threadIdx.x; j < 1024; j += 256) {
        const int cl = j >> 5, rl = j & 31, r = r0 + rl;
        if (r < rows) { const int bb = r / 42; o4[(size_t)cl * r_alloc + AZ_TC_HALO + (size_t)bb * AZ_TC_RPB + (r - bb * 42)] = tile[rl][cl]; }
    }
}

// k_tr_bn_bwd_rpb: dz = gamma * invstd * (g - c1 - xhat * c2), g = dout * [a > 0], written as the data gradient's / weight gradient's
// bf16 operand: plain, cells with x = 0 zeroed, cells with x = 5 zeroed (var_stride_u4 apart); the fp32 copy only if dz32 != NULL.
__global__ void __launch_bounds__(256) k_tr_bn_bwd_rpb(const float* __restrict__ z, const float* __restrict__ dout, const float* __restrict__ a,
                                                      const float* __restrict__ stats, const float* __restrict__ gamma, float* __restrict__ dz32,
                                                      int rows, __nv_bfloat16* __restrict__ dz_rpb, int r_alloc, size_t var_stride_u4)
{
    __shared__ uint4 tile[32][33];
    const int r0 = blockIdx.x * 32;
    for (int j = threadIdx.x; j < 1024; j += 256) {
        const int rl = j >> 5, cc = j & 31, r = r0 + rl;
        if (r < rows) {
            const size_t o = (size_t)r * TR_CH + cc * 8;
            const float4 z0 = *reinterpret_cast<const float4*>(z + o), z1 = *reinterpret_cast<const float4*>(z + o + 4);
            const float4 d0 = *reinterpret_cast<const float4*>(dout + o), d1 = *reinterpret_cast<const float4*>(dout + o + 4);
            const float4 a0 = *reinterpret_cast<const float4*>(a + o), a1 = *reinterpret_cast<const float4*>(a + o + 4);
            const float zz[8] = { z0.x, z0.y, z0.z, z0.w, z1.x, z1.y, z1.z, z1.w }, dd[8] = { d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w };
            const float aa[8] = { a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w };
            float v[8], mu[8], inv[8], c1[8], c2[8], ga[8];
            ld8(stats + cc * 8, mu); ld8(stats + TR_CH + cc * 8, inv); ld8(stats + 2 * TR_CH + cc * 8, c1); ld8(stats + 3 * TR_CH + cc * 8, c2);
            ld8(gamma + cc * 8, ga);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const float g = aa[e] > 0.0f ? dd[e] : 0.0f;
                const float xh = (zz[e] - mu[e]) * inv[e];
                v[e] = ga[e] * inv[e] * (g - c1[e] - xh * c2[e]);
            }
            if (dz32) {
                *reinterpret_cast<float4*>(dz32 + o) = make_float4(v[0], v[1], v[2], v[3]);
                *reinterpret_cast<float4*>(dz32 + o + 4) = make_float4(v[4], v[5], v[6], v[7]);
            }
            uint4 pk;
            __nv_bfloat162* p2 = reinterpret_cast<__nv_bfloat162*>(&pk);
#pragma unroll
            for (int e = 0; e < 4; ++e) p2[e] = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
            tile[rl][cc] = pk;
        }
    }
    __syncthreads();
    uint4* o4 = reinterpret_cast<uint4*>(dz_rpb);
    for (int j = threadIdx.x; j < 1024; j += 256) {
        const int cl = j >> 5, rl = j & 31, r = r0 + rl;
        if (r < rows) {
            const int bb = r / 42, p = r - bb * 42, x = p % 6;
            const size_t at = (size_t)cl * r_alloc + AZ_TC_HALO + (size_t)bb * AZ_TC_RPB + p;
            const uint4 v = tile[rl][cl], zero = make_uint4(0u, 0u, 0u, 0u);
            o4[at] = v; o4[var_stride_u4 + at] = x == 0 ? zero : v; o4[2 * var_stride_u4 + at] = x == 5 ? zero : v;
        }
    }
}

// ---------------------------------------------------------------- weight gradient of a 3x3 convolution
// dW[t][ci][co] = sum_r in[nb(r, t)][ci] * dz[r][co].  Block = (32 input channels) x (64 output channels) x all 9 taps for one split of
// the boards; 256 threads, thread = 2 ci x 4 co x 9 taps = 72 accumulators; one board (42 rows) staged in shared memory per iteration.
__global__ void __launch_bounds__(256) k_tr_wgrad(const float* __restrict__ in, int cin, const float* __restrict__ dz, int n, float* __restrict__ part)
{
    __shared__ float s_in[43][TC_CI];       // row 42 = zeros (taps outside the board)
    __shared__ float s_dz[42][TC_CO];
    const int ci0 = blockIdx.x * TC_CI, co0 = blockIdx.y * TC_CO, split = blockIdx.z;
    const int tci = (threadIdx.x >> 4) * 2, tco = (threadIdx.x & 15) * 4;
    float acc[9][2][4];
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
        for (int i = 0; i < 2; ++i) { acc[t][i][0] = acc[t][i][1] = acc[t][i][2] = acc[t][i][3] = 0.0f; }
    if (threadIdx.x < TC_CI) s_in[42][threadIdx.x] = 0.0f;
    const int per = (n + TR_WG_SPLITS - 1) / TR_WG_SPLITS;
    const int b_end = min(n, (split + 1) * per);
    for (int b = split * per; b < b_end; ++b) {
        __syncthreads();
        for (int i = threadIdx.x; i < 42 * TC_CI; i += 256) {
            int r = i / TC_CI, ci = i - r * TC_CI;
            s_in[r][ci] = ci0 + ci < cin ? in[((size_t)b * 42 + r) * cin + ci0 + ci] : 0.0f;
        }
        for (int i = threadIdx.x; i < 42 * TC_CO; i += 256) {
            int r = i / TC_CO, co = i - r * TC_CO;
            s_dz[r][co] = dz[((size_t)b * 42 + r) * TR_CH + co0 + co];
        }
        __syncthreads();
        for (int r = 0; r < 42; ++r) {
            const float4 d4 = *reinterpret_cast<const float4*>(&s_dz[r][tco]);
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                int q = c_tnb[r * 9 + t]; q = q < 0 ? 42 : q;
                const float2 a2 = *reinterpret_cast<const float2*>(&s_in[q][tci]);
                acc[t][0][0] = fmaf(a2.x, d4.x, acc[t][0][0]); acc[t][0][1] = fmaf(a2.x, d4.y, acc[t][0][1]);
                acc[t][0][2] = fmaf(a2.x, d4.z, acc[t][0][2]); acc[t][0][3] = fmaf(a2.x, d4.w, acc[t][0][3]);
                acc[t][1][0] = fmaf(a2.y, d4.x, acc[t][1][0]); acc[t][1][1] = fmaf(a2.y, d4.y, acc[t][1][1]);
                acc[t][1][2] = fmaf(a2.y, d4.z, acc[t][1][2]); acc[t][1][3] = fmaf(a2.y, d4.w, acc[t][1][3]);
            }
        }
    }
    float* dst = part + (size_t)split * 9 * cin * TR_CH;
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
        for (int i = 0; i < 2; ++i)
            if (ci0 + tci + i < cin)
                *reinterpret_cast<float4*>(dst + ((size_t)t * cin + ci0 + tci + i) * TR_CH + co0 + tco) =
                    make_float4(acc[t][i][0], acc[t][i][1], acc[t][i][2], acc[t][i][3]);
}

__global__ void __launch_bounds__(256) k_tr_wgrad_reduce(const float* __restrict__ part, size_t count, float* __restrict__ grad)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    float s = 0.0f;
    for (int k = 0; k < TR_WG_SPLITS; ++k) s += part[(size_t)k * count + i];
    grad[i] = s;
}

// ---------------------------------------------------------------- heads
__device__ __forceinline__ float tr_warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// the two 1x1 convolutions: hz[r] = (a[r] . pi_w[:, 0], a[r] . pi_w[:, 1], a[r] . v_w, 0); one warp per row
__global__ void __launch_bounds__(256) k_tr_head_conv(const float* __restrict__ act, int rows, const float* __restrict__ pi_w, const float* __restrict__ v_w,
                                                       float* __restrict__ hz)
{
    const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (r >= rows) return;
    const float* arow = act + (size_t)r * TR_CH;
    float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f;
    for (int c = lane; c < TR_CH; c += 32) {
        const float x = arow[c];
        s0 = fmaf(x, pi_w[c * 2 + 0], s0); s1 = fmaf(x, pi_w[c * 2 + 1], s1); s2 = fmaf(x, v_w[c], s2);
    }
    s0 = tr_warp_sum(s0); s1 = tr_warp_sum(s1); s2 = tr_warp_sum(s2);
    if (lane == 0) *reinterpret_cast<float4*>(hz + (size_t)r * 4) = make_float4(s0, s1, s2, 0.0f);
}

// statistics of the three head channels over all rows: one block, double accumulation, fixed order.
// mode 0: from hz -> mean, invstd (+ moving statistics); mode 1: from hg, hz -> c1, c2, dgamma, dbeta.
// hstats layout: [4][4] = mean[3], invstd[3], c1[3], c2[3] (stride 4)
__global__ void __launch_bounds__(256) k_tr_head_stats(const float* __restrict__ hz, const float* __restrict__ hg, int rows, int mode, float* __restrict__ hstats,
                                                        float* __restrict__ pi_mm, float* __restrict__ pi_mv, float* __restrict__ v_mm, float* __restrict__ v_mv,
                                                        float* __restrict__ pi_dgamma, float* __restrict__ pi_dbeta, float* __restrict__ v_dgamma, float* __restrict__ v_dbeta)
{
    __shared__ double s_red[256][6];
    double s[6] = { 0.0, 0.0, 0.0, 0.0, 0.0, 0.0 };
    for (int r = threadIdx.x; r < rows; r += 256) {
        const float4 zv = *reinterpret_cast<const float4*>(hz + (size_t)r * 4);
        const float zz[3] = { zv.x, zv.y, zv.z };
        if (mode == 0) { for (int k = 0; k < 3; ++k) { s[k] += (double)zz[k]; s[3 + k] += (double)zz[k] * (double)zz[k]; } }
        else {
            const float4 gv = *reinterpret_cast<const float4*>(hg + (size_t)r * 4);
            const float gg[3] = { gv.x, gv.y, gv.z };
            for (int k = 0; k < 3; ++k) { s[k] += (double)gg[k]; s[3 + k] += (double)gg[k] * (double)((zz[k] - hstats[k]) * hstats[4 + k]); }
        }
    }
    for (int k = 0; k < 6; ++k) s_red[threadIdx.x][k] = s[k];
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) for (int k = 0; k < 6; ++k) s_red[threadIdx.x][k] += s_red[threadIdx.x + o][k];
        __syncthreads();
    }
    if (threadIdx.x < 3) {
        const int k = threadIdx.x;
        const double count = (double)rows, s0 = s_red[0][k], s1 = s_red[0][3 + k];
        if (mode == 0) {
            const double mean = s0 / count;
            double var = s1 / count - mean * mean; if (var < 0.0) var = 0.0;
            hstats[k] = (float)mean; hstats[4 + k] = (float)(1.0 / sqrt(var + (double)AZ_NN_BN_EPS));
            float* mm = k < 2 ? pi_mm + k : v_mm; float* mv = k < 2 ? pi_mv + k : v_mv;
            *mm = *mm - (*mm - (float)mean) * (1.0f - TR_BN_MOMENTUM);
            *mv = *mv - (*mv - (float)(var * count / (count - 1.0))) * (1.0f - TR_BN_MOMENTUM);
        } else {
            hstats[8 + k] = (float)(s0 / count); hstats[12 + k] = (float)(s1 / count);
            *(k < 2 ? pi_dgamma + k : v_dgamma) = (float)s1; *(k < 2 ? pi_dbeta + k : v_dbeta) = (float)s0;
        }
    }
}

// one block per board: BN + ReLU of the three head channels, dense layers, softmax / tanh, the two losses, and the backward pass down to
// the gradient with respect to the BN outputs (masked by the ReLU) -> hg.  The per-board vectors the weight gradients need go to hfeat.
// hp.vo value outputs: tv [n][vo], the value loss is the mean over the n * vo squared errors, dh = sum_k dout_k * dense_2[:, k]
__global__ void __launch_bounds__(256) k_tr_head_board(const float* __restrict__ hz, const float* __restrict__ hstats, AzHeadParams hp, const float* __restrict__ tp,
                                                        const float* __restrict__ tv, int n, float* __restrict__ hg, float* __restrict__ hfeat)
{
    __shared__ float s_pi[84], s_v[42], s_h[256], s_dh[256], s_logit[43], s_dlogit[43], s_red[6][8], s_do[6], s_d2[6];
    const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* hf = hfeat + (size_t)b * HF_STRIDE;
    if (threadIdx.x < 42) {
        const int p = threadIdx.x;
        const float4 zv = *reinterpret_cast<const float4*>(hz + ((size_t)b * 42 + p) * 4);
        const float y0 = (zv.x - hstats[0]) * hstats[4] * hp.bn_pi[0] + hp.bn_pi[2];
        const float y1 = (zv.y - hstats[1]) * hstats[5] * hp.bn_pi[1] + hp.bn_pi[3];
        const float yv = (zv.z - hstats[2]) * hstats[6] * hp.bn_v[0] + hp.bn_v[1];
        s_pi[p * 2 + 0] = fmaxf(y0, 0.0f); s_pi[p * 2 + 1] = fmaxf(y1, 0.0f); s_v[p] = fmaxf(yv, 0.0f);
    }
    __syncthreads();
    if (threadIdx.x < 43) {
        float s = hp.dense_b[threadIdx.x];
        for (int k = 0; k < 84; ++k) s = fmaf(s_pi[k], hp.dense_w[k * 43 + threadIdx.x], s);
        s_logit[threadIdx.x] = s;
    }
    {
        float s = hp.dense1_b[threadIdx.x];
        for (int k = 0; k < 42; ++k) s = fmaf(s_v[k], hp.dense1_w[k * 256 + threadIdx.x], s);
        s_h[threadIdx.x] = fmaxf(s, 0.0f);
    }
    __syncthreads();
    const int vo = hp.vo;
    for (int k = 0; k < vo; ++k) {
        const float part = tr_warp_sum(s_h[threadIdx.x] * hp.dense2_w[threadIdx.x * vo + k]);
        if (lane == 0) s_red[k][warp] = part;
    }
    __syncthreads();
    const float inv_n = 1.0f / (float)n, inv_nv = 1.0f / (float)(n * vo);
    if (threadIdx.x < vo) {
        const int k = threadIdx.x;
        float s = hp.dense2_b[k];
        for (int i = 0; i < 8; ++i) s += s_red[k][i];
        const float v = tanhf(s), d = v - tv[(size_t)b * vo + k];
        s_do[k] = 2.0f * d * inv_nv * (1.0f - v * v);           // d(mean squared error) / d(pre-tanh output)
        s_d2[k] = d * d;
        hf[HF_DOUT + k] = s_do[k];
    }
    if (warp == 1) {                                             // softmax cross-entropy of this board and its logit gradient
        const float l0 = s_logit[lane], l1 = lane < 11 ? s_logit[32 + lane] : -INFINITY;
        float m = fmaxf(l0, l1);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        const float e0 = expf(l0 - m), e1 = lane < 11 ? expf(l1 - m) : 0.0f;
        const float sum = tr_warp_sum(e0 + e1), lse = m + logf(sum);
        const float t0 = tp[(size_t)b * 43 + lane], t1 = lane < 11 ? tp[(size_t)b * 43 + 32 + lane] : 0.0f;
        const float tsum = tr_warp_sum(t0 + t1);
        const float loss = tr_warp_sum(t0 * (lse - l0) + (lane < 11 ? t1 * (lse - l1) : 0.0f));
        s_dlogit[lane] = (e0 / sum * tsum - t0) * inv_n;
        if (lane < 11) s_dlogit[32 + lane] = (e1 / sum * tsum - t1) * inv_n;
        if (lane == 0) hf[HF_LOSS] = loss;
    }
    __syncthreads();
    if (threadIdx.x == 0) {                                      // this board's squared errors, in component order
        float l = s_d2[0];
        for (int k = 1; k < vo; ++k) l += s_d2[k];
        hf[HF_LOSS + 1] = l;
    }
    {
        float g = s_do[0] * hp.dense2_w[threadIdx.x * vo];
        for (int k = 1; k < vo; ++k) g += s_do[k] * hp.dense2_w[threadIdx.x * vo + k];
        s_dh[threadIdx.x] = s_h[threadIdx.x] > 0.0f ? g : 0.0f;
    }
    __syncthreads();
    if (threadIdx.x < 84) {                                      // gradient w.r.t. the flattened policy features
        float s = 0.0f;
        for (int j = 0; j < 43; ++j) s = fmaf(s_dlogit[j], hp.dense_w[threadIdx.x * 43 + j], s);
        hg[((size_t)b * 42 + threadIdx.x / 2) * 4 + (threadIdx.x & 1)] = s_pi[threadIdx.x] > 0.0f ? s : 0.0f;
    } else if (threadIdx.x >= 96 && threadIdx.x < 96 + 42) {     // ... and the value features
        const int k = threadIdx.x - 96;
        float s = 0.0f;
        for (int j = 0; j < 256; ++j) s = fmaf(s_dh[j], hp.dense1_w[k * 256 + j], s);
        hg[((size_t)b * 42 + k) * 4 + 2] = s_v[k] > 0.0f ? s : 0.0f;
        hg[((size_t)b * 42 + k) * 4 + 3] = 0.0f;
    }
    if (threadIdx.x < 84) hf[HF_SPI + threadIdx.x] = s_pi[threadIdx.x];
    if (threadIdx.x < 43) hf[HF_DLOGIT + threadIdx.x] = s_dlogit[threadIdx.x];
    if (threadIdx.x < 42) hf[HF_SV + threadIdx.x] = s_v[threadIdx.x];
    hf[HF_H + threadIdx.x] = s_h[threadIdx.x];
    hf[HF_DH + threadIdx.x] = s_dh[threadIdx.x];
}

// gradients of the dense layers: one thread per output element, boards summed in order; vo value outputs (dense_2 is [256][vo])
#define TR_HEAD_D1_END (84 * 43 + 43 + 42 * 256 + 256)
__global__ void __launch_bounds__(256) k_tr_head_dense_grad(const float* __restrict__ hfeat, int n, int vo, float* __restrict__ g_dense_w, float* __restrict__ g_dense_b,
                                                             float* __restrict__ g_d1_w, float* __restrict__ g_d1_b, float* __restrict__ g_d2_w, float* __restrict__ g_d2_b,
                                                             float* __restrict__ loss2)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int a_off, b_off; float* dst;
    if (i < 84 * 43) { a_off = HF_SPI + i / 43; b_off = HF_DLOGIT + i % 43; dst = g_dense_w + i; }
    else if (i < 84 * 43 + 43) { a_off = -1; b_off = HF_DLOGIT + (i - 84 * 43); dst = g_dense_b + (i - 84 * 43); }
    else if (i < 84 * 43 + 43 + 42 * 256) { const int k = i - (84 * 43 + 43); a_off = HF_SV + k / 256; b_off = HF_DH + k % 256; dst = g_d1_w + k; }
    else if (i < TR_HEAD_D1_END) { const int k = i - (84 * 43 + 43 + 42 * 256); a_off = -1; b_off = HF_DH + k; dst = g_d1_b + k; }
    else if (i < TR_HEAD_D1_END + 256 * vo) { const int k = i - TR_HEAD_D1_END; a_off = HF_H + k / vo; b_off = HF_DOUT + k % vo; dst = g_d2_w + k; }
    else if (i < TR_HEAD_D1_END + 257 * vo) { const int k = i - (TR_HEAD_D1_END + 256 * vo); a_off = -1; b_off = HF_DOUT + k; dst = g_d2_b + k; }
    else if (i < TR_HEAD_D1_END + 257 * vo + 2) {                // the two batch losses (means: over n boards, over n * vo value errors)
        const int k = i - (TR_HEAD_D1_END + 257 * vo);
        float s = 0.0f;
        for (int b = 0; b < n; ++b) s += hfeat[(size_t)b * HF_STRIDE + HF_LOSS + k];
        loss2[k] = s / (float)(k == 1 ? n * vo : n);
        return;
    } else return;
    float s = 0.0f;
    for (int b = 0; b < n; ++b) {
        const float* hf = hfeat + (size_t)b * HF_STRIDE;
        s = fmaf(a_off < 0 ? 1.0f : hf[a_off], hf[b_off], s);
    }
    *dst = s;
}
static inline int tr_head_dense_elems(int vo) { return TR_HEAD_D1_END + 257 * vo + 2; }

// BN backward of the head channels per row, then the gradient into the tower output: dA[r][c] = sum_k dz[r][k] * W[c][k].
// dz overwrites hg (the 1x1 kernels' gradient needs it).  One warp per row.
__global__ void __launch_bounds__(256) k_tr_head_back(const float* __restrict__ hz, float* __restrict__ hg, const float* __restrict__ hstats, const float* __restrict__ bn_pi,
                                                       const float* __restrict__ bn_v, const float* __restrict__ pi_w, const float* __restrict__ v_w, int rows,
                                                       float* __restrict__ dact)
{
    const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (r >= rows) return;
    const float4 zv = *reinterpret_cast<const float4*>(hz + (size_t)r * 4);
    const float4 gv = *reinterpret_cast<const float4*>(hg + (size_t)r * 4);
    const float zz[3] = { zv.x, zv.y, zv.z }, gg[3] = { gv.x, gv.y, gv.z };
    const float gam[3] = { bn_pi[0], bn_pi[1], bn_v[0] };
    float dz[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float inv = hstats[4 + k], xh = (zz[k] - hstats[k]) * inv;
        dz[k] = gam[k] * inv * (gg[k] - hstats[8 + k] - xh * hstats[12 + k]);
    }
    __syncwarp();
    if (lane == 0) *reinterpret_cast<float4*>(hg + (size_t)r * 4) = make_float4(dz[0], dz[1], dz[2], 0.0f);
    float* drow = dact + (size_t)r * TR_CH;
    for (int c = lane; c < TR_CH; c += 32) drow[c] = dz[0] * pi_w[c * 2 + 0] + dz[1] * pi_w[c * 2 + 1] + dz[2] * v_w[c];
}

// gradient of the 1x1 kernels: part[chunk][c][k] = sum over the chunk's rows of a[r][c] * dz[r][k]; thread = channel
__global__ void __launch_bounds__(256) k_tr_head_wgrad(const float* __restrict__ act, const float* __restrict__ hdz, int rows, float* __restrict__ part)
{
    const int c = threadIdx.x, chunk = blockIdx.x;
    const int per = (rows + TR_STAT_CHUNKS - 1) / TR_STAT_CHUNKS;
    const int r0 = chunk * per, r1 = min(rows, r0 + per);
    float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f;
    for (int r = r0; r < r1; ++r) {
        const float x = act[(size_t)r * TR_CH + c];
        const float4 d = *reinterpret_cast<const float4*>(hdz + (size_t)r * 4);
        s0 = fmaf(x, d.x, s0); s1 = fmaf(x, d.y, s1); s2 = fmaf(x, d.z, s2);
    }
    float* p = part + ((size_t)chunk * TR_CH + c) * 3;
    p[0] = s0; p[1] = s1; p[2] = s2;
}
__global__ void __launch_bounds__(256) k_tr_head_wgrad_final(const float* __restrict__ part, float* __restrict__ g_pi_w, float* __restrict__ g_v_w)
{
    const int c = threadIdx.x;
    float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f;
    for (int k = 0; k < TR_STAT_CHUNKS; ++k) { const float* p = part + ((size_t)k * TR_CH + c) * 3; s0 += p[0]; s1 += p[1]; s2 += p[2]; }
    g_pi_w[c * 2 + 0] = s0; g_pi_w[c * 2 + 1] = s1; g_v_w[c] = s2;
}

// ---------------------------------------------------------------- Adam (TensorFlow's ResourceApplyAdam), L2 term for kernels
// one launch over the whole variable blob; kind[i]: 0 = not trainable (moving statistics), 1 = plain, 2 = kernel (carries the L2 term)
__global__ void __launch_bounds__(256) k_tr_adam(float* __restrict__ w, float* __restrict__ grad, float* __restrict__ m, float* __restrict__ v, size_t count,
                                                  const uint8_t* __restrict__ kind, float l2_scale, float lr_t)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint8_t kd = kind[i];
    if (kd == 0) return;
    const float g = grad[i] + (kd == 2 ? l2_scale : 0.0f) * w[i];   // d(0.001 * sum w^2)/dw = 0.002 * w
    grad[i] = g;
    const float mi = m[i] + (g - m[i]) * (1.0f - TR_BETA1);
    const float vi = v[i] + (g * g - v[i]) * (1.0f - TR_BETA2);
    m[i] = mi; v[i] = vi;
    w[i] = w[i] - (mi * lr_t) / (sqrtf(vi) + TR_ADAM_EPS);
}

// epoch means without a host round trip per batch: the two batch losses are added, in batch order, to double accumulators
__global__ void k_tr_loss_accum(const float* __restrict__ loss2, double* __restrict__ acc2)
{
    if (threadIdx.x < 2) acc2[threadIdx.x] += (double)loss2[threadIdx.x];
}

// NNInputData images (88 bytes, alphazero_nn_data.h:73-101) -> input planes [n][7][6][13] (setInStateTensor, alphazero_nn.cpp:31-67);
// sample record = 1 + 88 + 4 + 43 * 4 bytes (alphazero_nn_data.cpp:115-138): also unpacks the value and policy targets
__global__ void __launch_bounds__(64) k_tr_unpack_samples(const uint8_t* __restrict__ rec, const uint32_t* __restrict__ order, int n, float* __restrict__ x,
                                                           float* __restrict__ tp, float* __restrict__ tv)
{
    const int b = blockIdx.x;
    if (b >= n) return;
    const uint8_t* r = rec + (size_t)order[b] * AZ_SAMPLE_BYTES + 1;     // NNInputData
    __shared__ float f[10];
    if (threadIdx.x < 10) { uint32_t u = 0; for (int k = 0; k < 4; ++k) u |= (uint32_t)r[48 + 4 * threadIdx.x + k] << (8 * k); f[threadIdx.x] = __uint_as_float(u); }
    __syncthreads();
    const int me = r[42];
    if (threadIdx.x < 42) {
        const int p = threadIdx.x;
        const uint32_t v = r[p], owner = v >> 6; const float army = (float)(v & 63u) / 32.0f;
        float* o = x + ((size_t)b * 42 + p) * 13;
        o[0] = owner == (uint32_t)me ? army : 0.0f;
        o[1] = (owner != (uint32_t)me && owner < 2u) ? army : 0.0f;
        o[2] = owner >= 2u ? army : 0.0f;
        o[3] = f[9];                                            // armyShare
        o[4] = f[0]; o[5] = f[1]; o[6] = f[2];                  // reinforcementShare, attackFrequency, canDrawCard
        for (int k = 0; k < 6; ++k) o[7 + k] = f[3 + k];        // phase one-hot
    }
    if (threadIdx.x == 42) { uint32_t u = 0; for (int k = 0; k < 4; ++k) u |= (uint32_t)r[88 + k] << (8 * k); tv[b] = __uint_as_float(u); }
    if (threadIdx.x < 43) { uint32_t u = 0; for (int k = 0; k < 4; ++k) u |= (uint32_t)r[92 + 4 * threadIdx.x + k] << (8 * k); tp[(size_t)b * 43 + threadIdx.x] = __uint_as_float(u); }
}

// six-player records (az_samples6.cuh) -> the six-seat input planes of each record's image (e6_encode_position, the encoding the
// six-player search evaluates its leaves with) + value and policy targets; one thread per sample.  vo = 6: tv [n][6], target k =
// s6_value(status, (cur + k) % 6) (component 0 is the record's stored value).  P = the network's input planes (13, or 16 seat planes)
template <int P>
__global__ void __launch_bounds__(128) k_tr_unpack_samples6(const uint8_t* __restrict__ rec, const uint32_t* __restrict__ order, int n,
                                                            float* __restrict__ x, float* __restrict__ tp, float* __restrict__ tv, int vo)
{
    const int b = blockIdx.x * 128 + threadIdx.x;
    if (b >= n) return;
    const uint8_t* r = rec + (size_t)order[b] * S6_BYTES;
    e6_encode_position<P>(r, r + AZ_LANDS, r[S6_CUR], r[S6_PHASE], r[S6_ATTACKS], r[S6_ALLOW_DRAW], x + (size_t)b * 42 * P);
    const float* f = (const float*)r;                       // records are 4-byte aligned (288-byte stride)
    if (vo == 1) tv[b] = f[S6_VALUE / 4];
    else for (int k = 0; k < vo; ++k) tv[(size_t)b * vo + k] = s6_value((int8_t)r[S6_STATUS], (r[S6_CUR] + (uint32_t)k) % E6_PLAYERS);
    for (int i = 0; i < AZ_MOVES; ++i) tp[(size_t)b * AZ_MOVES + i] = f[S6_PI / 4 + i];
}

// ---------------------------------------------------------------- host side
static bool is_moving(const std::string& name)
{
    auto ends = [&](const char* s) { size_t l = strlen(s); return name.size() >= l && name.compare(name.size() - l, l, s) == 0; };
    return ends("/moving_mean") || ends("/moving_variance");
}
static bool is_kernel(const std::string& name) { const char* s = "/kernel"; return name.size() >= 7 && name.compare(name.size() - 7, 7, s) == 0; }

static AzTrainState* train_state(az_nn* nn)
{
    if (!nn->train) {
        nn->train = new (std::nothrow) AzTrainState();
        if (nn->train) { nn->train->h_m.assign(nn->blob.size(), 0.0f); nn->train->h_v.assign(nn->blob.size(), 0.0f); }
    }
    return nn->train;
}

void az_nn_train_release(az_nn* nn)
{
    AzTrainState* t = nn->train;
    if (!t) return;
    cudaFree(t->d_grad); cudaFree(t->d_m); cudaFree(t->d_v); cudaFree(t->d_x);
    for (float* p : t->z) cudaFree(p);
    for (float* p : t->a) cudaFree(p);
    cudaFree(t->d_stats); cudaFree(t->d_part); for (int i = 0; i < 3; ++i) cudaFree(t->d_g[i]);
    cudaFree(t->d_wT); cudaFree(t->d_wpart); cudaFree(t->d_hz); cudaFree(t->d_hg); cudaFree(t->d_hfeat); cudaFree(t->d_hpart);
    cudaFree(t->d_tp); cudaFree(t->d_tv); cudaFree(t->d_loss); cudaFree(t->d_colA); cudaFree(t->d_colB); cudaFree(t->d_src16); cudaFree(t->d_kind);
    az_tc_conv_raw_release(&t->conv);
    delete t;
    nn->train = nullptr;
}

static int slots_to_device(az_nn* nn, AzTrainState* t)
{
    const size_t np = nn->blob.size();
    if (!t->d_grad) {
        AZ_CUDA(cudaMalloc(&t->d_grad, sizeof(float) * np)); AZ_CUDA(cudaMalloc(&t->d_m, sizeof(float) * np)); AZ_CUDA(cudaMalloc(&t->d_v, sizeof(float) * np));
        AZ_CUDA(cudaMemset(t->d_grad, 0, sizeof(float) * np));
        std::vector<uint8_t> kind(np, 0);
        for (const AzVar& v : nn->vars)
            if (!is_moving(v.name)) std::fill(kind.begin() + (ptrdiff_t)v.offset, kind.begin() + (ptrdiff_t)(v.offset + v.count), (uint8_t)(is_kernel(v.name) ? 2 : 1));
        AZ_CUDA(cudaMalloc(&t->d_kind, np));
        AZ_CUDA(cudaMemcpy(t->d_kind, kind.data(), np, cudaMemcpyHostToDevice));
    }
    if (!t->slots_on_device) {
        AZ_CUDA(cudaMemcpy(t->d_m, t->h_m.data(), sizeof(float) * np, cudaMemcpyHostToDevice));
        AZ_CUDA(cudaMemcpy(t->d_v, t->h_v.data(), sizeof(float) * np, cudaMemcpyHostToDevice));
        t->slots_on_device = true; t->host_slots_stale = false;
    }
    return AZ_OK;
}

static int slots_to_host(az_nn* nn, AzTrainState* t)
{
    if (t->slots_on_device && t->host_slots_stale) {
        const size_t np = nn->blob.size();
        AZ_CUDA(cudaMemcpy(t->h_m.data(), t->d_m, sizeof(float) * np, cudaMemcpyDeviceToHost));
        AZ_CUDA(cudaMemcpy(t->h_v.data(), t->d_v, sizeof(float) * np, cudaMemcpyDeviceToHost));
        t->host_slots_stale = false;
    }
    return AZ_OK;
}

static int train_reserve(az_nn* nn, AzTrainState* t, int n)
{
    if (n <= t->cap) return AZ_OK;
    const int layers = 2 * nn->blocks + 1;
    const size_t act = tr_mp(n * 42) * TR_CH;                   // rows padded to the GEMM's 128-row tiles (the tensor-core path writes whole tiles)
    for (float* p : t->z) cudaFree(p);
    for (float* p : t->a) cudaFree(p);
    t->z.assign((size_t)layers, nullptr); t->a.assign((size_t)layers, nullptr);
    cudaFree(t->d_x); cudaFree(t->d_hz); cudaFree(t->d_hg); cudaFree(t->d_hfeat); cudaFree(t->d_tp); cudaFree(t->d_tv);
    cudaFree(t->d_colA); cudaFree(t->d_colB); cudaFree(t->d_src16); t->d_colA = t->d_colB = t->d_src16 = nullptr;
    for (int i = 0; i < 3; ++i) { cudaFree(t->d_g[i]); t->d_g[i] = nullptr; }
    t->d_x = t->d_hz = t->d_hg = t->d_hfeat = t->d_tp = t->d_tv = nullptr; t->cap = 0;
    for (int L = 0; L < layers; ++L) { AZ_CUDA(cudaMalloc(&t->z[(size_t)L], sizeof(float) * act)); AZ_CUDA(cudaMalloc(&t->a[(size_t)L], sizeof(float) * act)); }
    for (int i = 0; i < 3; ++i) AZ_CUDA(cudaMalloc(&t->d_g[i], sizeof(float) * act));
    AZ_CUDA(cudaMalloc(&t->d_x, sizeof(float) * (size_t)n * 42 * nn->input_planes));
    AZ_CUDA(cudaMalloc(&t->d_hz, sizeof(float) * (size_t)n * 42 * 4)); AZ_CUDA(cudaMalloc(&t->d_hg, sizeof(float) * (size_t)n * 42 * 4));
    AZ_CUDA(cudaMalloc(&t->d_hfeat, sizeof(float) * (size_t)n * HF_STRIDE));
    AZ_CUDA(cudaMalloc(&t->d_tp, sizeof(float) * (size_t)n * 43)); AZ_CUDA(cudaMalloc(&t->d_tv, sizeof(float) * (size_t)n * nn->value_outputs));
    {   // GEMM operands of the tensor-core path: A = max(im2col [Mp][9*256], transposed im2col [9*256][Kp]), B = max(weights, dz^T)
        const size_t mp = tr_mp(n * 42), kpw = tr_kp(n * 42);
        const size_t a_elems = (size_t)9 * TR_CH * (mp > kpw ? mp : kpw), b_elems = (size_t)TR_CH * (kpw > (size_t)9 * TR_CH ? kpw : (size_t)9 * TR_CH);
        AZ_CUDA(cudaMalloc(&t->d_colA, a_elems * sizeof(__nv_bfloat16))); AZ_CUDA(cudaMalloc(&t->d_colB, b_elems * sizeof(__nv_bfloat16)));
        AZ_CUDA(cudaMalloc(&t->d_src16, (size_t)n * 42 * TR_CH * sizeof(__nv_bfloat16)));
    }
    if (!t->d_stats) {
        AZ_CUDA(cudaMalloc(&t->d_stats, sizeof(float) * (size_t)(layers + 1) * 4 * TR_CH));
        AZ_CUDA(cudaMalloc(&t->d_part, sizeof(double) * TR_STAT_CHUNKS * TR_CH * 2));
        AZ_CUDA(cudaMalloc(&t->d_wT, sizeof(float) * 9 * TR_CH * TR_CH));
        AZ_CUDA(cudaMalloc(&t->d_wpart, sizeof(float) * (size_t)TR_WG_SPLITS * 9 * TR_CH * TR_CH));
        AZ_CUDA(cudaMalloc(&t->d_hpart, sizeof(float) * TR_STAT_CHUNKS * TR_CH * 3));
        AZ_CUDA(cudaMalloc(&t->d_loss, sizeof(float) * 2));
        AZ_CUDA(cudaFuncSetAttribute(k_tr_conv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(TC_SMEM_FLOATS * sizeof(float))));
        int8_t nb[42 * 9];
        for (int p = 0; p < 42; ++p)
            for (int k = 0; k < 9; ++k) {
                int y = p / 6 + k / 3 - 1, x = p % 6 + k % 3 - 1;
                nb[p * 9 + k] = (y < 0 || y >= 7 || x < 0 || x >= 6) ? (int8_t)-1 : (int8_t)(y * 6 + x);
            }
        AZ_CUDA(cudaMemcpyToSymbol(c_tnb, nb, sizeof nb));
    }
    t->cap = n;
    return AZ_OK;
}

// one raw 3x3 convolution out[r][256] = conv(in[r][cin], w[9][cin][256]) (flip: the data-gradient kernel w[8-t] transposed)
static int conv_any(az_nn* nn, AzTrainState* t, const float* in, int n, int cin, const float* w, int flip, float* out, cudaStream_t s,
                    const __nv_bfloat16* in_rpb = nullptr)
{
    if (t->precision == AZ_NN_BF16 && cin == TR_CH) {       // implicit GEMM on the tower kernel (no unrolled operand in HBM)
        if (flip && t->dz_prepared) { t->dz_prepared = false; return az_tc_dgrad_prepared(&t->conv, n, w, out, s); }
        if (!flip && in_rpb) return az_tc_conv_raw_rpb(&t->conv, in_rpb, n, w, 0, out, s);
        return az_tc_conv_raw(&t->conv, in, n, w, flip, out, s);
    }
    if (t->precision == AZ_NN_BF16) {                       // the 13- or 16-channel stem: chunked im2col + k_tc_gemm
        const int rows = n * 42, mp = (int)tr_mp(rows), cpad = (cin + 7) / 8 * 8, kp = (int)tr_kp(9 * cpad);
        int rc = az_tg_im2col(in, rows, cin, cpad, mp, kp, t->d_src16, t->d_colA, s); if (rc) return rc;
        rc = az_tg_weights(w, cin, cpad, kp, flip, t->d_colB, s); if (rc) return rc;
        return az_tg_gemm(t->d_colA, t->d_colB, out, mp, kp, 1, s);
    }
    const float* wk = w;
    if (flip) {
        k_tr_flip_transpose<<<(9 * TR_CH * TR_CH + 255) / 256, 256, 0, s>>>(w, t->d_wT);
        wk = t->d_wT;
    }
    const dim3 cgrid((unsigned)((n + TC_BOARDS - 1) / TC_BOARDS), TR_CH / TC_CO);
    k_tr_conv<<<cgrid, 128, TC_SMEM_FLOATS * sizeof(float), s>>>(in, n, cin, wk, out);
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

// the fused tensor-core route: tower kernel + k_tc_wgrad with the bf16 operands written by the BatchNorm passes themselves
static bool tr_tower(const AzTrainState* t) { return t->precision == AZ_NN_BF16; }

static std::string tr_block_sfx(int i) { return std::to_string(i) + std::string(1, (char)('a' + i)); }
// layer L >= 1 of the tower: block (L - 1) / 2, branch 2a for odd L, 2b for even L
static std::string tr_conv_name(int L) { return L == 0 ? "conv" : "res" + tr_block_sfx((L - 1) / 2) + ((L & 1) ? "_branch2a" : "_branch2b"); }
static std::string tr_bn_name(int L) { return L == 0 ? "conv_bn" : "bn" + tr_block_sfx((L - 1) / 2) + ((L & 1) ? "_branch2a" : "_branch2b"); }

static float* dvar(az_nn* nn, const std::string& name) { return const_cast<float*>(az_nn_dev_var(nn, name)); }
static float* gvar(az_nn* nn, AzTrainState* t, const std::string& name) { return t->d_grad + nn->vars[(size_t)nn->index.at(name)].offset; }

// forward statistics + activation of conv layer L
static int bn_forward(az_nn* nn, AzTrainState* t, int L, int n, const float* skip, cudaStream_t s)
{
    const int rows = n * 42, stem = L == 0;
    const size_t total = (size_t)rows * TR_CH;
    float* st = t->d_stats + (size_t)L * 4 * TR_CH;
    const std::string bn = tr_bn_name(L);
    k_tr_stats<<<TR_STAT_CHUNKS, 256, 0, s>>>(t->z[(size_t)L], nullptr, nullptr, st, rows, 0, stem, t->d_part);
    k_tr_stats_final<<<8, 256, 0, s>>>(t->d_part, stem ? 7 : TR_CH, stem ? (double)n * 6 * TR_CH : (double)rows, 0, st,
                                       dvar(nn, bn + "/moving_mean"), dvar(nn, bn + "/moving_variance"), nullptr, nullptr);
    if (tr_tower(t) && L + 1 < 2 * nn->blocks + 1)          // the next 256-channel convolution (and its weight gradient) read the chunked bf16 copy
        k_tr_bn_apply_rpb<<<(unsigned)((rows + 31) / 32), 256, 0, s>>>(t->z[(size_t)L], st, dvar(nn, bn + "/gamma"), dvar(nn, bn + "/beta"), skip,
                                                                  t->a[(size_t)L], rows, stem, t->conv.a_rpb[(size_t)L], t->conv.r_alloc);
    else
        k_tr_bn_apply<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(t->z[(size_t)L], st, dvar(nn, bn + "/gamma"), dvar(nn, bn + "/beta"), skip, t->a[(size_t)L], total, stem);
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

// dz of conv layer L from dout (gradient w.r.t. the layer's activation output); writes dgamma / dbeta
static int bn_backward(az_nn* nn, AzTrainState* t, int L, int n, const float* dout, float* dz, cudaStream_t s)
{
    const int rows = n * 42, stem = L == 0;
    const size_t total = (size_t)rows * TR_CH;
    float* st = t->d_stats + (size_t)L * 4 * TR_CH;
    const std::string bn = tr_bn_name(L);
    k_tr_stats<<<TR_STAT_CHUNKS, 256, 0, s>>>(t->z[(size_t)L], dout, t->a[(size_t)L], st, rows, 1, stem, t->d_part);
    k_tr_stats_final<<<8, 256, 0, s>>>(t->d_part, stem ? 7 : TR_CH, stem ? (double)n * 6 * TR_CH : (double)rows, 1, st, nullptr, nullptr,
                                       gvar(nn, t, bn + "/gamma"), gvar(nn, t, bn + "/beta"));
    t->dz_prepared = false;
    if (tr_tower(t) && L >= 1) {                            // dz goes straight into the operand buffers of k_tc_wgrad and the data gradient; no fp32 copy
        __nv_bfloat16* dz3 = nullptr; size_t vs = 0;
        int rc = az_tc_dz_target(&t->conv, n, s, &dz3, &vs); if (rc) return rc;
        k_tr_bn_bwd_rpb<<<(unsigned)((rows + 31) / 32), 256, 0, s>>>(t->z[(size_t)L], dout, t->a[(size_t)L], st, dvar(nn, bn + "/gamma"), nullptr, rows,
                                                                dz3, t->conv.r_alloc, vs);
        t->dz_prepared = true;
    } else
        k_tr_bn_bwd<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(t->z[(size_t)L], dout, t->a[(size_t)L], st, dvar(nn, bn + "/gamma"), dz, total, stem);
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

static int conv_wgrad(az_nn* nn, AzTrainState* t, int L, int n, const float* in, int cin, const float* dz, cudaStream_t s)
{
    if (tr_tower(t) && cin == TR_CH) {
        // nine GEMMs over the board rows with both operands read in place from the chunked bf16 buffers (k_tc_wgrad): dz was written
        // by k_tr_bn_bwd_rpb, the layer's input activation by k_tr_bn_apply_rpb during the forward pass
        AZ_REQUIRE(t->dz_prepared && L >= 1, "weight gradient before its dz");
        int splits = 1;
        int rc = az_tc_wgrad_rpb(&t->conv, t->conv.a_rpb[(size_t)L - 1], n, t->d_wpart, TR_WG_SPLITS, &splits, s); if (rc) return rc;
        return az_tg_reduce(t->d_wpart, splits, 9 * TR_CH, 9 * TR_CH, gvar(nn, t, tr_conv_name(L) + "/kernel"), s);
    }
    if (t->precision == AZ_NN_BF16) {                          // the stem: dW[t*cin + ci][co] = im2col(in)^T . dz, K = board cells, split over K
        const int rows = n * 42, mp = (int)tr_mp(9 * cin), kp = (int)tr_kp(rows);
        const int splits = az_tg_splits(kp, 148 / (mp / 128) > TR_WG_SPLITS ? TR_WG_SPLITS : 148 / (mp / 128));
        int rc = az_tg_im2col_t(in, rows, cin, mp, kp, t->d_src16, t->d_colA, s); if (rc) return rc;
        rc = az_tg_rows_t(dz, rows, kp, t->d_colB, s); if (rc) return rc;
        rc = az_tg_gemm(t->d_colA, t->d_colB, t->d_wpart, mp, kp, splits, s); if (rc) return rc;
        return az_tg_reduce(t->d_wpart, splits, mp, 9 * cin, gvar(nn, t, tr_conv_name(L) + "/kernel"), s);
    }
    dim3 grid((unsigned)((cin + TC_CI - 1) / TC_CI), TR_CH / TC_CO, TR_WG_SPLITS);
    k_tr_wgrad<<<grid, 256, 0, s>>>(in, cin, dz, n, t->d_wpart);
    const size_t count = (size_t)9 * cin * TR_CH;
    k_tr_wgrad_reduce<<<(unsigned)((count + 255) / 256), 256, 0, s>>>(t->d_wpart, count, gvar(nn, t, tr_conv_name(L) + "/kernel"));
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

static int train_step_dev(az_nn* nn, const float* d_x, const float* d_tp, const float* d_tv, int n, float* h_loss2, cudaStream_t s)
{
    AzTrainState* t = train_state(nn);
    AZ_REQUIRE(t != nullptr, "out of host memory");
    int rc = AZ_OK;
    if (!nn->host_stale) { rc = az_nn_finalize(nn); if (rc) return rc; }      // device copy of the weights is current (or already ahead)
    rc = slots_to_device(nn, t); if (rc) return rc;
    rc = train_reserve(nn, t, n); if (rc) return rc;
    if (t->precision == AZ_NN_BF16) { rc = az_tg_init(); if (rc) return rc; }
    if (tr_tower(t)) { rc = az_tc_layers_reserve(&t->conv, n, 2 * nn->blocks); if (rc) return rc; }
    const int layers = 2 * nn->blocks + 1, rows = n * 42;
    const size_t total = (size_t)rows * TR_CH;
    const unsigned egrid = (unsigned)((total + 255) / 256);
    // ---- forward
    rc = conv_any(nn, t, d_x, n, nn->input_planes, dvar(nn, "conv/kernel"), 0, t->z[0], s); if (rc) return rc;
    rc = bn_forward(nn, t, 0, n, nullptr, s); if (rc) return rc;
    for (int L = 1; L < layers; ++L) {
        rc = conv_any(nn, t, t->a[(size_t)L - 1], n, TR_CH, dvar(nn, tr_conv_name(L) + "/kernel"), 0, t->z[(size_t)L], s,
                      tr_tower(t) ? t->conv.a_rpb[(size_t)L - 1] : nullptr); if (rc) return rc;
        rc = bn_forward(nn, t, L, n, (L & 1) ? nullptr : t->a[(size_t)L - 2], s); if (rc) return rc;      // 2b adds the block input
    }
    const float* act = t->a[(size_t)layers - 1];
    float* hst = t->d_stats + (size_t)layers * 4 * TR_CH;
    const AzHeadParams hp = az_nn_head_params(nn);
    k_tr_head_conv<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(act, rows, hp.pi_w, hp.v_w, t->d_hz);
    k_tr_head_stats<<<1, 256, 0, s>>>(t->d_hz, nullptr, rows, 0, hst, dvar(nn, "bn_pi/moving_mean"), dvar(nn, "bn_pi/moving_variance"),
                                      dvar(nn, "bn_v/moving_mean"), dvar(nn, "bn_v/moving_variance"), nullptr, nullptr, nullptr, nullptr);
    k_tr_head_board<<<(unsigned)n, 256, 0, s>>>(t->d_hz, hst, hp, d_tp, d_tv, n, t->d_hg, t->d_hfeat);
    // ---- backward: heads
    k_tr_head_dense_grad<<<(tr_head_dense_elems(hp.vo) + 255) / 256, 256, 0, s>>>(t->d_hfeat, n, hp.vo, gvar(nn, t, "dense/kernel"), gvar(nn, t, "dense/bias"),
                                                                           gvar(nn, t, "dense_1/kernel"), gvar(nn, t, "dense_1/bias"),
                                                                           gvar(nn, t, "dense_2/kernel"), gvar(nn, t, "dense_2/bias"), t->d_loss);
    k_tr_head_stats<<<1, 256, 0, s>>>(t->d_hz, t->d_hg, rows, 1, hst, nullptr, nullptr, nullptr, nullptr,
                                      gvar(nn, t, "bn_pi/gamma"), gvar(nn, t, "bn_pi/beta"), gvar(nn, t, "bn_v/gamma"), gvar(nn, t, "bn_v/beta"));
    float *G0 = t->d_g[0], *G1 = t->d_g[1], *G2 = t->d_g[2];
    k_tr_head_back<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(t->d_hz, t->d_hg, hst, hp.bn_pi, hp.bn_v, hp.pi_w, hp.v_w, rows, G0);
    k_tr_head_wgrad<<<TR_STAT_CHUNKS, 256, 0, s>>>(act, t->d_hg, rows, t->d_hpart);
    k_tr_head_wgrad_final<<<1, 256, 0, s>>>(t->d_hpart, gvar(nn, t, "pi/kernel"), gvar(nn, t, "v/kernel"));
    AZ_CUDA(cudaGetLastError());
    // ---- backward: tower.  G0 = gradient w.r.t. the output of block i
    for (int i = nn->blocks - 1; i >= 0; --i) {
        const int La = 1 + 2 * i, Lb = 2 + 2 * i;
        rc = bn_backward(nn, t, Lb, n, G0, G1, s); if (rc) return rc;                                   // dz of 2b
        rc = conv_wgrad(nn, t, Lb, n, t->a[(size_t)La], TR_CH, G1, s); if (rc) return rc;
        rc = conv_any(nn, t, G1, n, TR_CH, dvar(nn, tr_conv_name(Lb) + "/kernel"), 1, G2, s); if (rc) return rc;   // gradient w.r.t. the 2a activation
        rc = bn_backward(nn, t, La, n, G2, G1, s); if (rc) return rc;                                   // dz of 2a
        rc = conv_wgrad(nn, t, La, n, t->a[(size_t)La - 1], TR_CH, G1, s); if (rc) return rc;
        rc = conv_any(nn, t, G1, n, TR_CH, dvar(nn, tr_conv_name(La) + "/kernel"), 1, G2, s); if (rc) return rc;   // gradient w.r.t. the block input ...
        k_tr_add_masked<<<egrid, 256, 0, s>>>(G2, G0, t->a[(size_t)Lb], total);                         // ... plus the skip connection's share
        float* tmp = G0; G0 = G2; G2 = tmp;
    }
    rc = bn_backward(nn, t, 0, n, G0, G1, s); if (rc) return rc;
    rc = conv_wgrad(nn, t, 0, n, d_x, nn->input_planes, G1, s); if (rc) return rc;
    // ---- Adam
    const float lr_t = (float)((double)TR_LR * sqrt(1.0 - (double)t->beta2_power) / (1.0 - (double)t->beta1_power));
    const size_t np = nn->blob.size();
    k_tr_adam<<<(unsigned)((np + 255) / 256), 256, 0, s>>>(nn->d_blob, t->d_grad, t->d_m, t->d_v, np, t->d_kind, 2.0f * TR_L2, lr_t);
    AZ_CUDA(cudaGetLastError());
    t->beta1_power *= TR_BETA1; t->beta2_power *= TR_BETA2; t->steps++;
    t->host_slots_stale = true;
    nn->host_stale = true; nn->finalized = false;               // the device weights are ahead of nn->blob and of the packed bf16 tiles
    if (h_loss2) {
        AZ_CUDA(cudaMemcpyAsync(h_loss2, t->d_loss, sizeof(float) * 2, cudaMemcpyDeviceToHost, s));
        AZ_CUDA(cudaStreamSynchronize(s));
    }
    return AZ_OK;
}

extern "C" int az_nn_train_step(az_nn* nn, const float* h_x, const float* h_target_policy, const float* h_target_value, int n,
                                float* loss_policy, float* loss_value, void* stream)
{
    AZ_REQUIRE(nn && h_x && h_target_policy && h_target_value, "NULL argument");
    AZ_REQUIRE(n >= 2, "a training batch needs at least 2 samples (batch statistics)");
    AzDeviceGuard guard(nn->device);
    cudaStream_t s = (cudaStream_t)stream;
    AzTrainState* t = train_state(nn);
    AZ_REQUIRE(t != nullptr, "out of host memory");
    int rc = train_reserve(nn, t, n); if (rc) return rc;
    AZ_CUDA(cudaMemcpyAsync(t->d_x, h_x, sizeof(float) * (size_t)n * 42 * nn->input_planes, cudaMemcpyHostToDevice, s));
    AZ_CUDA(cudaMemcpyAsync(t->d_tp, h_target_policy, sizeof(float) * (size_t)n * 43, cudaMemcpyHostToDevice, s));
    AZ_CUDA(cudaMemcpyAsync(t->d_tv, h_target_value, sizeof(float) * (size_t)n * nn->value_outputs, cudaMemcpyHostToDevice, s));
    float loss[2] = { 0.0f, 0.0f };
    rc = train_step_dev(nn, t->d_x, t->d_tp, t->d_tv, n, loss, s); if (rc) return rc;
    if (loss_policy) *loss_policy = loss[0];
    if (loss_value) *loss_value = loss[1];
    return AZ_OK;
}

// the record -> (input planes, targets) step of a training loop: batch b of an epoch unpacks the n records order[0..n) of d_rec
// (tv holds vo values per record, x `planes` input planes per board cell)
typedef void (*TrUnpack)(const uint8_t* d_rec, const uint32_t* d_order, int n, float* x, float* tp, float* tv, int vo, int planes, cudaStream_t s);
static void tr_unpack_samples(const uint8_t* d_rec, const uint32_t* d_order, int n, float* x, float* tp, float* tv, int, int, cudaStream_t s)
{
    k_tr_unpack_samples<<<(unsigned)n, 64, 0, s>>>(d_rec, d_order, n, x, tp, tv);
}
static void tr_unpack_samples6(const uint8_t* d_rec, const uint32_t* d_order, int n, float* x, float* tp, float* tv, int vo, int planes,
                               cudaStream_t s)
{
    if (planes == AZ_NN_IN_CH6) k_tr_unpack_samples6<AZ_NN_IN_CH6><<<(unsigned)((n + 127) / 128), 128, 0, s>>>(d_rec, d_order, n, x, tp, tv, vo);
    else k_tr_unpack_samples6<AZ_NN_IN_CH><<<(unsigned)((n + 127) / 128), 128, 0, s>>>(d_rec, d_order, n, x, tp, tv, vo);
}

// AlphaZeroNN::train (alphazero_nn.cpp:351-410): `epochs` passes over the samples in shuffled order, whole batches of batch_size only
// (:372 batchCount = size / BATCH_SIZE), on records of rec_bytes each that `unpack` turns into a batch.
// The reference shuffles with its process-wide std engine (irreproducible, src/rng.h:16); here: Fisher-Yates on splitmix64(seed).
static int train_records(az_nn* nn, const char* who, const uint8_t* h_records, size_t n_records, size_t rec_bytes, TrUnpack unpack,
                         int epochs, int batch_size, uint64_t seed, float* h_epoch_loss_policy, float* h_epoch_loss_value, cudaStream_t s)
{
    AzTrainState* t = train_state(nn);
    AZ_REQUIRE(t != nullptr, "out of host memory");
    int rc = train_reserve(nn, t, batch_size); if (rc) return rc;
    uint8_t* d_rec = nullptr; uint32_t* d_order = nullptr; double* d_acc = nullptr;
    AZ_CUDA(cudaMalloc(&d_rec, n_records * rec_bytes));
    if (cudaMalloc(&d_order, sizeof(uint32_t) * n_records) != cudaSuccess || cudaMalloc(&d_acc, 2 * sizeof(double)) != cudaSuccess) {
        cudaFree(d_rec); cudaFree(d_order); az_set_error("out of device memory"); return AZ_ERR_CUDA;
    }
    cudaError_t ce = cudaMemcpyAsync(d_rec, h_records, n_records * rec_bytes, cudaMemcpyHostToDevice, s);
    std::vector<uint32_t> order(n_records);
    for (size_t i = 0; i < n_records; ++i) order[i] = (uint32_t)i;
    uint64_t st = seed;
    const size_t batches = n_records / (size_t)batch_size;
    for (int e = 0; e < epochs && ce == cudaSuccess && rc == AZ_OK; ++e) {
        for (size_t i = n_records - 1; i > 0; --i) {
            st += 0x9E3779B97F4A7C15ull;
            uint64_t z = st; z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; z ^= z >> 31;
            const size_t j = (size_t)(z % (uint64_t)(i + 1));
            const uint32_t tmp = order[i]; order[i] = order[j]; order[j] = tmp;
        }
        ce = cudaMemcpyAsync(d_order, order.data(), sizeof(uint32_t) * n_records, cudaMemcpyHostToDevice, s);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
        // the batches of an epoch are enqueued back to back; the losses are accumulated on the device and read once per epoch
        if (ce == cudaSuccess) ce = cudaMemsetAsync(d_acc, 0, 2 * sizeof(double), s);
        for (size_t b = 0; b < batches && ce == cudaSuccess && rc == AZ_OK; ++b) {
            unpack(d_rec, d_order + b * (size_t)batch_size, batch_size, t->d_x, t->d_tp, t->d_tv, nn->value_outputs, nn->input_planes, s);
            rc = train_step_dev(nn, t->d_x, t->d_tp, t->d_tv, batch_size, nullptr, s);
            if (rc == AZ_OK) k_tr_loss_accum<<<1, 32, 0, s>>>(t->d_loss, d_acc);
        }
        double acc[2] = { 0.0, 0.0 };
        if (ce == cudaSuccess && rc == AZ_OK) ce = cudaMemcpyAsync(acc, d_acc, sizeof acc, cudaMemcpyDeviceToHost, s);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
        if (h_epoch_loss_policy) h_epoch_loss_policy[e] = (float)(acc[0] / (double)batches);
        if (h_epoch_loss_value) h_epoch_loss_value[e] = (float)(acc[1] / (double)batches);
    }
    cudaStreamSynchronize(s);
    cudaFree(d_rec); cudaFree(d_order); cudaFree(d_acc);
    if (ce != cudaSuccess) { az_set_error("%s: %s", who, cudaGetErrorString(ce)); return AZ_ERR_CUDA; }
    return rc;
}

// Samples are the packed records az_selfplay_samples returns (the reference's file layout).
extern "C" int az_nn_train(az_nn* nn, const uint8_t* h_records, size_t n_records, int epochs, int batch_size, uint64_t seed,
                           float* h_epoch_loss_policy, float* h_epoch_loss_value, void* stream)
{
    AZ_REQUIRE(nn && h_records, "NULL argument");
    AZ_REQUIRE(epochs >= 1 && batch_size >= 2, "epochs must be >= 1 and batch_size >= 2");
    AZ_REQUIRE(n_records >= (size_t)batch_size, "fewer samples than one batch");
    AZ_REQUIRE(nn->value_outputs == 1, "az_nn_train: two-player records hold one value target; the network has six value outputs");
    AZ_REQUIRE(nn->input_planes == AZ_NN_IN_CH, "az_nn_train: two-player records encode 13 input planes; the network has 16 (the six-player seat planes)");
    AzDeviceGuard guard(nn->device);
    return train_records(nn, "az_nn_train", h_records, n_records, AZ_SAMPLE_BYTES, tr_unpack_samples, epochs, batch_size, seed,
                         h_epoch_loss_policy, h_epoch_loss_value, (cudaStream_t)stream);
}

// The same loop on six-player records (az_selfplay6_samples); the input planes are the six-seat encoding of each record's image, with
// the network's plane count.
extern "C" int az_nn_train6(az_nn* nn, const uint8_t* h_records, size_t n_records, int epochs, int batch_size, uint64_t seed,
                            float* h_epoch_loss_policy, float* h_epoch_loss_value, void* stream)
{
    AZ_REQUIRE(nn && h_records, "NULL argument");
    AZ_REQUIRE(epochs >= 1 && batch_size >= 2, "epochs must be >= 1 and batch_size >= 2");
    AZ_REQUIRE(n_records >= (size_t)batch_size, "fewer samples than one batch");
    for (size_t i = 0; i < n_records; ++i) {                // the encoder indexes per-seat tables with these bytes
        const uint8_t* r = h_records + i * S6_BYTES;
        bool ok = r[S6_CUR] < E6_PLAYERS;
        for (int l = 0; l < AZ_LANDS; ++l) ok = ok && r[AZ_LANDS + l] < E6_PLAYERS;
        if (!ok) { az_set_error("az_nn_train6: record %zu holds a seat outside 0..5", i); return AZ_ERR_INVALID_ARG; }
    }
    AzDeviceGuard guard(nn->device);
    return train_records(nn, "az_nn_train6", h_records, n_records, S6_BYTES, tr_unpack_samples6, epochs, batch_size, seed,
                         h_epoch_loss_policy, h_epoch_loss_value, (cudaStream_t)stream);
}

// AZ_NN_FP32 (default): every contraction on the fp32 pipes — the parity path.  AZ_NN_BF16: forward convolutions, data gradients and
// weight gradients as bf16 tcgen05 GEMMs with fp32 accumulation (az_tc_gemm.cu); statistics, BatchNorm, heads, losses, Adam stay fp32.
extern "C" int az_nn_train_precision(az_nn* nn, int precision)
{
    AZ_REQUIRE(nn != nullptr, "nn is NULL");
    AZ_REQUIRE(precision == AZ_NN_FP32 || precision == AZ_NN_BF16, "precision must be AZ_NN_FP32 or AZ_NN_BF16");
    AzTrainState* t = train_state(nn);
    AZ_REQUIRE(t != nullptr, "out of host memory");
    t->precision = precision;
    return AZ_OK;
}

// gradient of the total loss (L2 term included) w.r.t. a trainable variable, as of the last step (test introspection)
extern "C" int az_nn_train_get_grad(az_nn* nn, const char* name, float* h_out, size_t count)
{
    AZ_REQUIRE(nn && name && h_out, "NULL argument");
    AZ_REQUIRE(nn->train && nn->train->d_grad, "no training step has run on this network");
    auto it = nn->index.find(name);
    if (it == nn->index.end()) { az_set_error("unknown variable '%s'", name); return AZ_ERR_INVALID_ARG; }
    const AzVar& v = nn->vars[(size_t)it->second];
    AZ_REQUIRE(v.count == count, "element count mismatch");
    AzDeviceGuard guard(nn->device);
    AZ_CUDA(cudaMemcpy(h_out, nn->train->d_grad + v.offset, sizeof(float) * count, cudaMemcpyDeviceToHost));
    return AZ_OK;
}

// raw convolution output z (which = 0) or activation a (which = 1) of tower layer `layer` (0 = stem, 2i+1 / 2i+2 = branch 2a / 2b of
// block i) as of the last step, [boards][42][256] (test introspection: per-layer forward parity of the two precisions)
extern "C" int az_nn_train_get_layer(az_nn* nn, int layer, int which, float* h_out, size_t count)
{
    AZ_REQUIRE(nn && h_out && (which == 0 || which == 1), "bad argument");
    AZ_REQUIRE(nn->train && nn->train->cap > 0, "no training step has run on this network");
    AzTrainState* t = nn->train;
    AZ_REQUIRE(layer >= 0 && layer < (int)t->z.size(), "layer out of range");
    AZ_REQUIRE(count <= (size_t)t->cap * 42 * TR_CH, "more elements than the last batch holds");
    AzDeviceGuard guard(nn->device);
    AZ_CUDA(cudaMemcpy(h_out, (which ? t->a : t->z)[(size_t)layer], sizeof(float) * count, cudaMemcpyDeviceToHost));
    return AZ_OK;
}

// Adam state of a variable: which = 0 -> m ("<var>/optimize"), 1 -> v ("<var>/optimize_1")
extern "C" int az_nn_optimizer_get(az_nn* nn, const char* name, int which, float* h_out, size_t count)
{
    AZ_REQUIRE(nn && name && h_out && (which == 0 || which == 1), "bad argument");
    AzTrainState* t = train_state(nn);
    AZ_REQUIRE(t != nullptr, "out of host memory");
    auto it = nn->index.find(name);
    if (it == nn->index.end()) { az_set_error("unknown variable '%s'", name); return AZ_ERR_INVALID_ARG; }
    const AzVar& v = nn->vars[(size_t)it->second];
    AZ_REQUIRE(v.count == count, "element count mismatch");
    AzDeviceGuard guard(nn->device);
    int rc = slots_to_host(nn, t); if (rc) return rc;
    memcpy(h_out, (which ? t->h_v : t->h_m).data() + v.offset, sizeof(float) * count);
    return AZ_OK;
}

extern "C" int az_nn_optimizer_powers(az_nn* nn, float* beta1_power, float* beta2_power, uint64_t* steps)
{
    AZ_REQUIRE(nn != nullptr, "nn is NULL");
    AzTrainState* t = train_state(nn);
    AZ_REQUIRE(t != nullptr, "out of host memory");
    if (beta1_power) *beta1_power = t->beta1_power;
    if (beta2_power) *beta2_power = t->beta2_power;
    if (steps) *steps = t->steps;
    return AZ_OK;
}

// ---------------------------------------------------------------- replica hand-off
// AlphaZeroNNGroup::train (alphazero_gpu_cluster.cpp:221-231) trains the first network of a group, saves a temporary checkpoint and
// loads it into the group's copies on the other GPUs.  Here the same state (every variable, both Adam slots of every trainable
// variable, the beta powers — what the graph's Saver writes) goes from `src` to `dst` by peer copies over NVLink when it lives on
// the device, by a host copy when it does not; no file in between.  dst must have the same number of residual blocks.
extern "C" int az_nn_copy_state(az_nn* dst, az_nn* src, void* stream)
{
    AZ_REQUIRE(dst && src, "NULL argument");
    AZ_REQUIRE(dst->blocks == src->blocks && dst->blob.size() == src->blob.size(), "networks differ in architecture");
    if (dst == src) return AZ_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t np = src->blob.size(), bytes = sizeof(float) * np;
    AzTrainState* ts = src->train;
    AzTrainState* td = ts ? train_state(dst) : dst->train;
    AZ_REQUIRE(!ts || td, "out of host memory");
    {
        AzDeviceGuard guard(dst->device);
        if (src->host_stale) {                                   // the device copy is the current one: peer copy, dst is then "ahead" too
            if (!dst->d_blob) AZ_CUDA(cudaMalloc(&dst->d_blob, bytes));
            AZ_CUDA(cudaMemcpyPeerAsync(dst->d_blob, dst->device, src->d_blob, src->device, bytes, s));
            dst->host_stale = true; dst->finalized = false;
        } else {
            dst->blob = src->blob; dst->host_stale = false; dst->finalized = false;
        }
        if (ts) {
            if (ts->slots_on_device) {
                int rc = slots_to_device(dst, td); if (rc) return rc;          // allocates dst's slot buffers
                AZ_CUDA(cudaMemcpyPeerAsync(td->d_m, dst->device, ts->d_m, src->device, bytes, s));
                AZ_CUDA(cudaMemcpyPeerAsync(td->d_v, dst->device, ts->d_v, src->device, bytes, s));
                td->host_slots_stale = true;
            } else {
                td->h_m = ts->h_m; td->h_v = ts->h_v; td->slots_on_device = false; td->host_slots_stale = false;
            }
            td->beta1_power = ts->beta1_power; td->beta2_power = ts->beta2_power; td->steps = ts->steps;
        } else if (td) {                                         // src never trained: dst goes back to a fresh optimizer
            std::fill(td->h_m.begin(), td->h_m.end(), 0.0f); std::fill(td->h_v.begin(), td->h_v.end(), 0.0f);
            td->slots_on_device = false; td->host_slots_stale = false;
            td->beta1_power = TR_BETA1; td->beta2_power = TR_BETA2; td->steps = 0;
        }
        AZ_CUDA(cudaStreamSynchronize(s));
    }
    return AZ_OK;
}

// ---------------------------------------------------------------- checkpoints
// TF_OP_SAVE (alphazero_nn.cpp:207-214): every tensor of the graph's Saver
extern "C" int az_nn_save_checkpoint(az_nn* nn, const char* prefix)
{
    AZ_REQUIRE(nn && prefix, "NULL argument");
    AzDeviceGuard guard(nn->device);
    AzTrainState* t = train_state(nn);
    AZ_REQUIRE(t != nullptr, "out of host memory");
    int rc = az_nn_sync_host(nn); if (rc) return rc;
    rc = slots_to_host(nn, t); if (rc) return rc;
    std::vector<std::string> names; std::vector<int> ranks; std::vector<std::vector<int64_t>> shapes; std::vector<const float*> data;
    auto add = [&](const std::string& nm, const std::vector<int>& shp, const float* p) {
        names.push_back(nm); ranks.push_back((int)shp.size()); shapes.emplace_back(shp.begin(), shp.end()); data.push_back(p);
    };
    for (const AzVar& v : nn->vars) {
        add(v.name, v.shape, nn->blob.data() + v.offset);
        if (!is_moving(v.name)) { add(v.name + "/optimize", v.shape, t->h_m.data() + v.offset); add(v.name + "/optimize_1", v.shape, t->h_v.data() + v.offset); }
    }
    add("beta1_power", {}, &t->beta1_power); add("beta2_power", {}, &t->beta2_power);
    std::vector<const char*> cn; std::vector<const int64_t*> cs;
    for (size_t i = 0; i < names.size(); ++i) { cn.push_back(names[i].c_str()); cs.push_back(shapes[i].data()); }
    return az_ckpt_write(prefix, (int)names.size(), cn.data(), ranks.data(), cs.data(), data.data());
}

// TF_OP_RESTORE (alphazero_nn.cpp:189-204): every variable must be in the checkpoint with the graph's shape (restore_all fails
// otherwise); the optimizer tensors are restored when present (a checkpoint written by the graph's Saver always has them)
extern "C" int az_nn_load_checkpoint(az_nn* nn, const char* prefix)
{
    AZ_REQUIRE(nn && prefix, "NULL argument");
    AzDeviceGuard guard(nn->device);
    AzTrainState* t = train_state(nn);
    AZ_REQUIRE(t != nullptr, "out of host memory");
    az_ckpt* c = nullptr;
    int rc = az_ckpt_open(prefix, &c); if (rc) return rc;
    auto check = [&](const std::string& nm, const std::vector<int>& shp) -> int {
        const int i = az_ckpt_find(c, nm.c_str());
        if (i < 0) { az_set_error("checkpoint %s has no tensor '%s'", prefix, nm.c_str()); return AZ_ERR_INVALID_ARG; }
        int dtype = 0, rank = 0; int64_t s8[8];
        az_ckpt_tensor_info(c, i, nullptr, &dtype, &rank, s8, nullptr);
        bool ok = dtype == 1 && rank == (int)shp.size();
        for (int k = 0; ok && k < rank; ++k) ok = s8[k] == (int64_t)shp[(size_t)k];
        if (!ok) { az_set_error("checkpoint %s: tensor '%s' has a different dtype/shape than the graph's variable", prefix, nm.c_str()); return AZ_ERR_INVALID_ARG; }
        return AZ_OK;
    };
    std::vector<float> blob(nn->blob.size()), m(nn->blob.size(), 0.0f), v(nn->blob.size(), 0.0f);
    float b1 = TR_BETA1, b2 = TR_BETA2;
    for (const AzVar& var : nn->vars) {
        rc = check(var.name, var.shape); if (rc) break;
        rc = az_ckpt_read(c, var.name.c_str(), blob.data() + var.offset, var.count * sizeof(float)); if (rc) break;
        if (is_moving(var.name)) continue;
        const std::string sm = var.name + "/optimize", sv = var.name + "/optimize_1";
        if (az_ckpt_find(c, sm.c_str()) >= 0 && az_ckpt_find(c, sv.c_str()) >= 0) {
            rc = check(sm, var.shape); if (rc) break;
            rc = check(sv, var.shape); if (rc) break;
            rc = az_ckpt_read(c, sm.c_str(), m.data() + var.offset, var.count * sizeof(float)); if (rc) break;
            rc = az_ckpt_read(c, sv.c_str(), v.data() + var.offset, var.count * sizeof(float)); if (rc) break;
        }
    }
    if (!rc && az_ckpt_find(c, "beta1_power") >= 0 && az_ckpt_find(c, "beta2_power") >= 0) {
        rc = az_ckpt_read(c, "beta1_power", &b1, sizeof(float));
        if (!rc) rc = az_ckpt_read(c, "beta2_power", &b2, sizeof(float));
    }
    az_ckpt_close(c);
    if (rc) return rc;
    nn->blob = blob; nn->finalized = false; nn->host_stale = false;
    t->h_m = m; t->h_v = v; t->slots_on_device = false; t->host_slots_stale = false;
    t->beta1_power = b1; t->beta2_power = b2;
    return AZ_OK;
}
