// az_nn_tc_value6.cu — the translation unit of the bf16 tensor-core forward: az_nn_tc.cu itself (included byte for byte: the ncu capture
// of its tower kernel in profiles/traffic.json is keyed by that file's hash) plus the value tail of a network with six value outputs
// (SIXPLAYER.md §2, az_nn_create_value).
//
// A six-output network shares everything with the one-output graph up to dense_1: the same tower, the same 1x1 head convolutions (whose
// per-cell sums the last tower layer's epilogue writes to d_head_z) and the same policy head.  So its forward is az_nn_tc_forward
// unchanged — policy bit for bit what a one-output network with the same shared weights gives — followed by k_nn_value6_tail, which
// reads d_head_z again and writes value [n][6] over the scalar the one-output tail left in the first n entries.
#include "az_nn_tc.cu"

// value [n][6] for HB boards per block: BatchNorm + ReLU of the v channel, dense 42 -> 256 + ReLU, dense 256 -> 6, tanh; the
// arithmetic of k_nn_heads_tail's value head, once per output column
__global__ void __launch_bounds__(256) k_nn_value6_tail(const float4* __restrict__ head_z, int n, AzHeadParams hp, float* __restrict__ value)
{
    __shared__ float s_v[HB][42], s_red[HB][6][8];
    const int b0 = blockIdx.x * HB, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nb = n - b0 < HB ? n - b0 : HB;
    const float scv = hp.bn_v[0] * rsqrtf(hp.bn_v[3] + AZ_NN_BN_EPS);
    for (int i = threadIdx.x; i < nb * 42; i += 256) {
        const int bl = i / 42, p = i - bl * 42;
        s_v[bl][p] = fmaxf((__ldg(head_z + (size_t)(b0 + bl) * 42 + p).z - hp.bn_v[2]) * scv + hp.bn_v[1], 0.0f);
    }
    __syncthreads();
    float acc[HB];
#pragma unroll
    for (int bl = 0; bl < HB; ++bl) acc[bl] = hp.dense1_b[threadIdx.x];
    for (int k = 0; k < 42; ++k) {
        const float w = hp.dense1_w[k * 256 + threadIdx.x];
#pragma unroll
        for (int bl = 0; bl < HB; ++bl) acc[bl] = fmaf(s_v[bl][k], w, acc[bl]);
    }
#pragma unroll
    for (int c = 0; c < 6; ++c) {
        const float w2 = hp.dense2_w[threadIdx.x * 6 + c];
#pragma unroll
        for (int bl = 0; bl < HB; ++bl) {
            const float part = warp_sum_tc(fmaxf(acc[bl], 0.0f) * w2);
            if (lane == 0) s_red[bl][c][warp] = part;
        }
    }
    __syncthreads();
    if (threadIdx.x < nb * 6) {
        const int bl = threadIdx.x / 6, c = threadIdx.x - bl * 6;
        float sum = hp.dense2_b[c];
        for (int i = 0; i < 8; ++i) sum += s_red[bl][c][i];
        value[(size_t)b0 * 6 + threadIdx.x] = tanhf(sum);
    }
}

// the bf16 forward of a six-output network: d_value holds [n][6]
int az_nn_tc_forward_value6(az_nn* nn, const float* d_x, int n, float* d_policy, float* d_value, cudaStream_t s)
{
    int rc = az_nn_tc_forward(nn, d_x, nullptr, n, d_policy, d_value, s);
    if (rc) return rc;
    k_nn_value6_tail<<<(n + HB - 1) / HB, 256, 0, s>>>(nn->tc->scratch[0].d_head_z, n, az_nn_head_params(nn), d_value);
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}
