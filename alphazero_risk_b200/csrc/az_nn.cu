// az_nn.cu — policy/value network of the reference (python/src/build_graph.py:54-90), weights,
// the fp32 validation forward and the az_nn_* C ABI.  The bf16 tcgen05 tower lives in az_nn_tc.cu.
//
// Network (N2 in SURVEY.md §8a): input [n,7,6,13] NHWC -> conv3x3 13->256 (no bias) -> BN over the
// BOARD-ROW axis (7 parameters: build_graph.py:68 passes axis=1 on an NHWC tensor) -> ReLU ->
// BLOCKS x {conv3x3, BN(256), ReLU, conv3x3, BN(256), +skip, ReLU} -> policy head conv1x1->2, BN,
// ReLU, flatten(84, NHWC order), dense 43 + bias, softmax ; value head conv1x1->1, BN, ReLU,
// flatten(42), dense 256 + bias, ReLU, dense 1 + bias, tanh (dense value_outputs = 6 for the six-seat value vector of
// SIXPLAYER.md §2, each output through tanh; 16 input planes instead of 13 for its seat planes, az_nn_create_planes).  Inference BN:
// y = (x - moving_mean) * (gamma * rsqrt(moving_variance + 0.001)) + beta.
// Replaces the TensorFlow session->Run of neural_network/alphazero_nn.cpp:247-248, :339-340.
#include <cmath>
#include <cstring>
#include <map>
#include <string>
#include <vector>
#include <new>

#include "az_common.cuh"
#include "az_nn.cuh"

// ---------------------------------------------------------------- variable inventory
static std::string block_letter(int i) { return std::string(1, (char)('a' + i)); }

static void add_var(az_nn* nn, const std::string& name, std::vector<int> shape, float init_limit, float init_const)
{
    AzVar v; v.name = name; v.shape = shape; v.count = 1; for (int d : shape) v.count *= (size_t)d;
    v.offset = nn->blob.size(); v.glorot_limit = init_limit; v.init_const = init_const;
    nn->blob.resize(nn->blob.size() + v.count, init_const);
    nn->index[name] = (int)nn->vars.size();
    nn->vars.push_back(v);
}
static void add_bn(az_nn* nn, const std::string& prefix, int c)
{
    add_var(nn, prefix + "/gamma", { c }, 0.0f, 1.0f);
    add_var(nn, prefix + "/beta", { c }, 0.0f, 0.0f);
    add_var(nn, prefix + "/moving_mean", { c }, 0.0f, 0.0f);
    add_var(nn, prefix + "/moving_variance", { c }, 0.0f, 1.0f);
}
static float glorot(int fan_in, int fan_out) { return sqrtf(6.0f / (float)(fan_in + fan_out)); }

// variable names / shapes of the shipped GraphDef (python/model/model_txt_V2_5.pb); Glorot-uniform
// limits reproduce the initializers recorded there (stem 0.049783, tower 0.036084, pi 0.152499, ...)
static void build_inventory(az_nn* nn)
{
    add_var(nn, "conv/kernel", { 3, 3, nn->input_planes, AZ_NN_CH }, glorot(9 * nn->input_planes, 9 * AZ_NN_CH), 0.0f);
    add_bn(nn, "conv_bn", 7);
    for (int i = 0; i < nn->blocks; ++i) {
        std::string s = std::to_string(i) + block_letter(i);
        add_var(nn, "res" + s + "_branch2a/kernel", { 3, 3, AZ_NN_CH, AZ_NN_CH }, glorot(9 * AZ_NN_CH, 9 * AZ_NN_CH), 0.0f);
        add_bn(nn, "bn" + s + "_branch2a", AZ_NN_CH);
        add_var(nn, "res" + s + "_branch2b/kernel", { 3, 3, AZ_NN_CH, AZ_NN_CH }, glorot(9 * AZ_NN_CH, 9 * AZ_NN_CH), 0.0f);
        add_bn(nn, "bn" + s + "_branch2b", AZ_NN_CH);
    }
    add_var(nn, "pi/kernel", { 1, 1, AZ_NN_CH, 2 }, glorot(AZ_NN_CH, 2), 0.0f);
    add_bn(nn, "bn_pi", 2);
    add_var(nn, "dense/kernel", { 84, 43 }, glorot(84, 43), 0.0f);
    add_var(nn, "dense/bias", { 43 }, 0.0f, 0.0f);
    add_var(nn, "v/kernel", { 1, 1, AZ_NN_CH, 1 }, glorot(AZ_NN_CH, 1), 0.0f);
    add_bn(nn, "bn_v", 1);
    add_var(nn, "dense_1/kernel", { 42, 256 }, glorot(42, 256), 0.0f);
    add_var(nn, "dense_1/bias", { 256 }, 0.0f, 0.0f);
    add_var(nn, "dense_2/kernel", { 256, nn->value_outputs }, glorot(256, nn->value_outputs), 0.0f);
    add_var(nn, "dense_2/bias", { nn->value_outputs }, 0.0f, 0.0f);
}

const float* az_nn_host_var(const az_nn* nn, const std::string& name)
{
    auto it = nn->index.find(name);
    return it == nn->index.end() ? nullptr : nn->blob.data() + nn->vars[it->second].offset;
}

// ---------------------------------------------------------------- fp32 kernels
// neighbour of board cell p for tap t (ky*3+kx), -1 outside the 7x6 board (padding SAME)
__constant__ int8_t c_nb[42 * 9];

// stem: conv3x3 P->256 + row-indexed BN + ReLU.  One block per board, thread = output channel.  P = input planes: 13 (the reference
// graph), 16 (the six-player seat planes)
template <int P>
__global__ void __launch_bounds__(256) k_nn_stem_fp32(const float* __restrict__ x, int n, const float* __restrict__ w /*[9][P][256]*/,
                                                       const float* __restrict__ bn /*[4][7]: gamma,beta,mean,var*/,
                                                       float* __restrict__ out /*[n][42][256]*/)
{
    __shared__ float s_in[43 * P];
    int b = blockIdx.x, co = threadIdx.x;
    for (int i = threadIdx.x; i < 42 * P; i += 256) s_in[i] = x[(size_t)b * 42 * P + i];
    if (threadIdx.x < P) s_in[42 * P + threadIdx.x] = 0.0f;
    __syncthreads();
    float wr[9 * P];
#pragma unroll
    for (int i = 0; i < 9 * P; ++i) wr[i] = w[i * AZ_NN_CH + co];
    for (int p = 0; p < 42; ++p) {
        float acc = 0.0f;
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            int q = c_nb[p * 9 + t]; q = q < 0 ? 42 : q;
#pragma unroll
            for (int ci = 0; ci < P; ++ci) acc = fmaf(s_in[q * P + ci], wr[t * P + ci], acc);
        }
        int y = p / 6;
        float sc = bn[y] * rsqrtf(bn[21 + y] + AZ_NN_BN_EPS);
        float v = (acc - bn[14 + y]) * sc + bn[7 + y];
        out[((size_t)b * 42 + p) * AZ_NN_CH + co] = v > 0.0f ? v : 0.0f;
    }
}

// tower conv3x3 256->256 (+BN, optional skip, ReLU), fp32 on CUDA cores.  Block = 4 boards x 64
// output channels, 128 threads, each thread 21 rows x 4 channels; input channels in chunks of 32.
#define F32_BOARDS 4
#define F32_ROWS (F32_BOARDS * 42)
#define F32_CO 64
#define F32_CI 32
#define F32_SMEM_FLOATS ((F32_ROWS + 1) * F32_CI + 9 * F32_CI * F32_CO)

__global__ void __launch_bounds__(128) k_nn_conv_fp32(const float* __restrict__ in /*[n][42][256]*/, int n,
                                                       const float* __restrict__ w /*[9][256][256]*/,
                                                       const float* __restrict__ bn /*[4][256]*/, const float* __restrict__ skip,
                                                       float* __restrict__ out)
{
    extern __shared__ float sm[];
    float* s_in = sm;                               // [F32_ROWS + 1][F32_CI], last row = zeros
    float* s_w = sm + (F32_ROWS + 1) * F32_CI;      // [9][F32_CI][F32_CO]
    const int b0 = blockIdx.x * F32_BOARDS, co0 = blockIdx.y * F32_CO;
    const int cg = threadIdx.x & 15, rg = threadIdx.x >> 4;
    const int rows_valid = min(F32_BOARDS, n - b0) * 42;
    float acc[21][4];
#pragma unroll
    for (int j = 0; j < 21; ++j) { acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.0f; }
    if (threadIdx.x < F32_CI) s_in[F32_ROWS * F32_CI + threadIdx.x] = 0.0f;
    for (int c0 = 0; c0 < AZ_NN_CH; c0 += F32_CI) {
        __syncthreads();
        for (int i = threadIdx.x; i < F32_ROWS * F32_CI; i += 128) {
            int r = i / F32_CI, ci = i - r * F32_CI;
            s_in[i] = r < rows_valid ? in[((size_t)b0 * 42 + r) * AZ_NN_CH + c0 + ci] : 0.0f;
        }
        for (int i = threadIdx.x; i < 9 * F32_CI * F32_CO; i += 128) {
            int t = i / (F32_CI * F32_CO), rem = i - t * (F32_CI * F32_CO), ci = rem / F32_CO, co = rem - ci * F32_CO;
            s_w[i] = w[((size_t)t * AZ_NN_CH + c0 + ci) * AZ_NN_CH + co0 + co];
        }
        __syncthreads();
        for (int t = 0; t < 9; ++t) {
            int src[21];
#pragma unroll
            for (int j = 0; j < 21; ++j) {
                int r = rg * 21 + j, bi = r / 42, p = r - bi * 42;
                int q = c_nb[p * 9 + t];
                src[j] = (q < 0 ? F32_ROWS : bi * 42 + q) * F32_CI;
            }
            const float* wt = s_w + t * F32_CI * F32_CO + cg * 4;
#pragma unroll 4
            for (int ci = 0; ci < F32_CI; ++ci) {
                float4 w4 = *reinterpret_cast<const float4*>(wt + ci * F32_CO);
#pragma unroll
                for (int j = 0; j < 21; ++j) {
                    float a = s_in[src[j] + ci];
                    acc[j][0] = fmaf(a, w4.x, acc[j][0]); acc[j][1] = fmaf(a, w4.y, acc[j][1]);
                    acc[j][2] = fmaf(a, w4.z, acc[j][2]); acc[j][3] = fmaf(a, w4.w, acc[j][3]);
                }
            }
        }
    }
    float sc[4], sh[4], mu[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        int co = co0 + cg * 4 + k;
        sc[k] = bn[co] * rsqrtf(bn[3 * AZ_NN_CH + co] + AZ_NN_BN_EPS); sh[k] = bn[AZ_NN_CH + co]; mu[k] = bn[2 * AZ_NN_CH + co];
    }
#pragma unroll
    for (int j = 0; j < 21; ++j) {
        int r = rg * 21 + j;
        if (r < rows_valid) {
            size_t o = ((size_t)b0 * 42 + r) * AZ_NN_CH + co0 + cg * 4;
            float4 v;
            v.x = (acc[j][0] - mu[0]) * sc[0] + sh[0]; v.y = (acc[j][1] - mu[1]) * sc[1] + sh[1];
            v.z = (acc[j][2] - mu[2]) * sc[2] + sh[2]; v.w = (acc[j][3] - mu[3]) * sc[3] + sh[3];
            if (skip) { float4 s = *reinterpret_cast<const float4*>(skip + o); v.x += s.x; v.y += s.y; v.z += s.z; v.w += s.w; }
            v.x = fmaxf(v.x, 0.0f); v.y = fmaxf(v.y, 0.0f); v.z = fmaxf(v.z, 0.0f); v.w = fmaxf(v.w, 0.0f);
            *reinterpret_cast<float4*>(out + o) = v;
        }
    }
}

// heads.  One block (256 threads) per board; works on fp32 activations [n][42][256].
__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// VO = value outputs (AzHeadParams::vo); with VO = 1 the arithmetic is the one-output graph's, operation for operation
template <int VO>
__global__ void __launch_bounds__(256) k_nn_heads_fp32(const float* __restrict__ act, int n, AzHeadParams hp,
                                                        float* __restrict__ policy /*[n][43]*/, float* __restrict__ value /*[n][VO]*/)
{
    __shared__ float s_pi[84], s_v[42], s_h[256], s_logit[43], s_red[VO][8];
    const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // 1x1 convs: every warp takes cells warp, warp+8, ...
    for (int p = warp; p < 42; p += 8) {
        const float* a = act + ((size_t)b * 42 + p) * AZ_NN_CH;
        float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f;
        for (int c = lane; c < AZ_NN_CH; c += 32) {
            float x = a[c];
            s0 = fmaf(x, hp.pi_w[c * 2 + 0], s0); s1 = fmaf(x, hp.pi_w[c * 2 + 1], s1); s2 = fmaf(x, hp.v_w[c], s2);
        }
        s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2);
        if (lane == 0) {
            float y0 = (s0 - hp.bn_pi[4]) * (hp.bn_pi[0] * rsqrtf(hp.bn_pi[6] + AZ_NN_BN_EPS)) + hp.bn_pi[2];
            float y1 = (s1 - hp.bn_pi[5]) * (hp.bn_pi[1] * rsqrtf(hp.bn_pi[7] + AZ_NN_BN_EPS)) + hp.bn_pi[3];
            float yv = (s2 - hp.bn_v[2]) * (hp.bn_v[0] * rsqrtf(hp.bn_v[3] + AZ_NN_BN_EPS)) + hp.bn_v[1];
            s_pi[p * 2 + 0] = fmaxf(y0, 0.0f); s_pi[p * 2 + 1] = fmaxf(y1, 0.0f); s_v[p] = fmaxf(yv, 0.0f);
        }
    }
    __syncthreads();
    // dense 84 -> 43 (+bias)
    if (threadIdx.x < 43) {
        float s = hp.dense_b[threadIdx.x];
        for (int k = 0; k < 84; ++k) s = fmaf(s_pi[k], hp.dense_w[k * 43 + threadIdx.x], s);
        s_logit[threadIdx.x] = s;
    }
    // dense 42 -> 256 (+bias, ReLU)
    {
        float s = hp.dense1_b[threadIdx.x];
        for (int k = 0; k < 42; ++k) s = fmaf(s_v[k], hp.dense1_w[k * 256 + threadIdx.x], s);
        s_h[threadIdx.x] = fmaxf(s, 0.0f);
    }
    __syncthreads();
    // dense 256 -> VO (+bias, tanh)
#pragma unroll
    for (int k = 0; k < VO; ++k) {
        const float part = warp_sum(s_h[threadIdx.x] * hp.dense2_w[threadIdx.x * VO + k]);
        if (lane == 0) s_red[k][warp] = part;
    }
    __syncthreads();
    if (threadIdx.x < VO) {
        float s = hp.dense2_b[threadIdx.x];
        for (int i = 0; i < 8; ++i) s += s_red[threadIdx.x][i];
        value[(size_t)b * VO + threadIdx.x] = tanhf(s);
    }
    // softmax over 43 logits
    if (warp == 0) {
        float l0 = s_logit[lane], l1 = lane < 11 ? s_logit[32 + lane] : -INFINITY;
        float m = fmaxf(l0, l1);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        float e0 = expf(l0 - m), e1 = lane < 11 ? expf(l1 - m) : 0.0f;
        float sum = warp_sum(e0 + e1);
        policy[(size_t)b * 43 + lane] = e0 / sum;
        if (lane < 11) policy[(size_t)b * 43 + 32 + lane] = e1 / sum;
    }
}

// ---------------------------------------------------------------- host: handle
static int upload(float** d, const float* h, size_t count)
{
    if (!*d) AZ_CUDA(cudaMalloc(d, sizeof(float) * count));
    AZ_CUDA(cudaMemcpy(*d, h, sizeof(float) * count, cudaMemcpyHostToDevice));
    return AZ_OK;
}

extern "C" int az_nn_create_planes(int blocks, int value_outputs, int input_planes, int device, az_nn** out)
{
    AZ_REQUIRE(out != nullptr, "out is NULL");
    AZ_REQUIRE(blocks >= 1 && blocks <= 26, "blocks must be in [1, 26]");
    AZ_REQUIRE(value_outputs == 1 || value_outputs == 6, "value_outputs must be 1 or 6");
    AZ_REQUIRE(input_planes == AZ_NN_IN_CH || input_planes == AZ_NN_IN_CH6, "input_planes must be 13 or 16");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); az_set_error("no CUDA device: libaz_b200 has no CPU fallback"); return AZ_ERR_NO_DEVICE; }
    AZ_REQUIRE(device >= 0 && device < ndev, "device index out of range");
    AzDeviceGuard guard(device);
    az_nn* nn = new (std::nothrow) az_nn();
    AZ_REQUIRE(nn != nullptr, "out of host memory");
    nn->blocks = blocks; nn->device = device; nn->value_outputs = value_outputs; nn->input_planes = input_planes;
    build_inventory(nn);
    int8_t nb[42 * 9];
    for (int p = 0; p < 42; ++p)
        for (int t = 0; t < 9; ++t) {
            int y = p / 6 + t / 3 - 1, x = p % 6 + t % 3 - 1;
            nb[p * 9 + t] = (y < 0 || y >= 7 || x < 0 || x >= 6) ? (int8_t)-1 : (int8_t)(y * 6 + x);
        }
    cudaError_t ce = cudaMemcpyToSymbol(c_nb, nb, sizeof nb);
    if (ce == cudaSuccess) ce = cudaFuncSetAttribute(k_nn_conv_fp32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(F32_SMEM_FLOATS * sizeof(float)));
    if (ce != cudaSuccess) { az_set_error("az_nn_create: %s", cudaGetErrorString(ce)); cudaGetLastError(); delete nn; return AZ_ERR_CUDA; }
    *out = nn;
    return AZ_OK;
}

extern "C" int az_nn_create_value(int blocks, int value_outputs, int device, az_nn** out)
{
    return az_nn_create_planes(blocks, value_outputs, AZ_NN_IN_CH, device, out);
}
extern "C" int az_nn_create(int blocks, int device, az_nn** out) { return az_nn_create_value(blocks, 1, device, out); }

extern "C" int az_nn_destroy(az_nn* nn)
{
    if (!nn) return AZ_OK;
    AzDeviceGuard guard(nn->device);
    cudaFree(nn->d_blob); cudaFree(nn->d_act[0]); cudaFree(nn->d_act[1]); cudaFree(nn->d_act[2]);
    cudaFree(nn->d_x); cudaFree(nn->d_policy); cudaFree(nn->d_value);
    az_nn_tc_release(nn);
    az_nn_train_release(nn);
    delete nn;
    return AZ_OK;
}

extern "C" int az_nn_num_vars(const az_nn* nn) { return nn ? (int)nn->vars.size() : 0; }
extern "C" size_t az_nn_num_params(const az_nn* nn) { return nn ? nn->blob.size() : 0; }
extern "C" int az_nn_blocks(const az_nn* nn) { return nn ? nn->blocks : 0; }
extern "C" int az_nn_value_outputs(const az_nn* nn) { return nn ? nn->value_outputs : 0; }
extern "C" int az_nn_input_planes(const az_nn* nn) { return nn ? nn->input_planes : 0; }

extern "C" int az_nn_var_info(const az_nn* nn, int i, const char** name, size_t* count, int* rank, int* shape4)
{
    AZ_REQUIRE(nn && i >= 0 && i < (int)nn->vars.size(), "variable index out of range");
    const AzVar& v = nn->vars[i];
    if (name) *name = v.name.c_str();
    if (count) *count = v.count;
    if (rank) *rank = (int)v.shape.size();
    if (shape4) for (int k = 0; k < 4; ++k) shape4[k] = k < (int)v.shape.size() ? v.shape[k] : 1;
    return AZ_OK;
}

extern "C" int az_nn_load_weights(az_nn* nn, const char* name, const float* h_ptr, size_t count)
{
    AZ_REQUIRE(nn && name && h_ptr, "NULL argument");
    auto it = nn->index.find(name);
    if (it == nn->index.end()) { az_set_error("unknown variable '%s'", name); return AZ_ERR_INVALID_ARG; }
    const AzVar& v = nn->vars[it->second];
    if (v.count != count) { az_set_error("variable '%s' has %zu elements, got %zu", name, v.count, count); return AZ_ERR_INVALID_ARG; }
    { AzDeviceGuard guard(nn->device); int rc = az_nn_sync_host(nn); if (rc) return rc; }
    memcpy(nn->blob.data() + v.offset, h_ptr, sizeof(float) * count);
    nn->finalized = false;
    return AZ_OK;
}

extern "C" int az_nn_get_weights(const az_nn* nn, const char* name, float* h_ptr, size_t count)
{
    AZ_REQUIRE(nn && name && h_ptr, "NULL argument");
    { AzDeviceGuard guard(nn->device); int rc = az_nn_sync_host(const_cast<az_nn*>(nn)); if (rc) return rc; }
    auto it = nn->index.find(name);
    if (it == nn->index.end()) { az_set_error("unknown variable '%s'", name); return AZ_ERR_INVALID_ARG; }
    const AzVar& v = nn->vars[it->second];
    AZ_REQUIRE(v.count == count, "element count mismatch");
    memcpy(h_ptr, nn->blob.data() + v.offset, sizeof(float) * count);
    return AZ_OK;
}

extern "C" int az_nn_export_blob(const az_nn* nn, float* h_out, size_t count)
{
    AZ_REQUIRE(nn && h_out && count == nn->blob.size(), "blob size mismatch");
    { AzDeviceGuard guard(nn->device); int rc = az_nn_sync_host(const_cast<az_nn*>(nn)); if (rc) return rc; }
    memcpy(h_out, nn->blob.data(), sizeof(float) * count);
    return AZ_OK;
}
extern "C" int az_nn_import_blob(az_nn* nn, const float* h_in, size_t count)
{
    AZ_REQUIRE(nn && h_in && count == nn->blob.size(), "blob size mismatch");
    memcpy(nn->blob.data(), h_in, sizeof(float) * count);
    nn->finalized = false; nn->host_stale = false;
    return AZ_OK;
}

// random init = what the graph's "init" op does (alphazero_nn.cpp:185): Glorot-uniform kernels,
// zero biases, gamma = 1, beta = 0, moving_mean = 0, moving_variance = 1.  splitmix64 stream.
extern "C" int az_nn_init_random(az_nn* nn, uint64_t seed)
{
    AZ_REQUIRE(nn != nullptr, "nn is NULL");
    nn->host_stale = false;
    uint64_t s = seed;
    for (const AzVar& v : nn->vars) {
        float* p = nn->blob.data() + v.offset;
        if (v.glorot_limit > 0.0f) {
            for (size_t i = 0; i < v.count; ++i) {
                s += 0x9E3779B97F4A7C15ull;
                uint64_t z = s; z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; z ^= z >> 31;
                float u = (float)(z >> 40) * (1.0f / 16777216.0f);
                p[i] = (2.0f * u - 1.0f) * v.glorot_limit;
            }
        } else for (size_t i = 0; i < v.count; ++i) p[i] = v.init_const;
    }
    nn->finalized = false;
    return AZ_OK;
}

// weights a training step has moved on the device -> nn->blob (the packed bf16 tiles are then rebuilt by the next finalize)
int az_nn_sync_host(az_nn* nn)
{
    if (!nn->host_stale) return AZ_OK;
    AZ_CUDA(cudaMemcpy(nn->blob.data(), nn->d_blob, sizeof(float) * nn->blob.size(), cudaMemcpyDeviceToHost));
    nn->host_stale = false; nn->finalized = false;
    return AZ_OK;
}

static int finalize(az_nn* nn)
{
    if (nn->host_stale) { int rc = az_nn_sync_host(nn); if (rc) return rc; }
    if (nn->finalized) return AZ_OK;
    int rc = upload(&nn->d_blob, nn->blob.data(), nn->blob.size());
    if (rc) return rc;
    rc = az_nn_tc_prepare(nn);
    if (rc) return rc;
    nn->finalized = true;
    return AZ_OK;
}
extern "C" int az_nn_finalize(az_nn* nn)
{
    AZ_REQUIRE(nn != nullptr, "nn is NULL");
    AzDeviceGuard guard(nn->device);
    return finalize(nn);
}

const float* az_nn_dev_var(const az_nn* nn, const std::string& name)
{
    auto it = nn->index.find(name);
    return it == nn->index.end() ? nullptr : nn->d_blob + nn->vars[it->second].offset;
}

int az_nn_reserve(az_nn* nn, int n)
{
    if (n <= nn->cap) return AZ_OK;
    for (int i = 0; i < 3; ++i) { cudaFree(nn->d_act[i]); nn->d_act[i] = nullptr; }
    cudaFree(nn->d_x); cudaFree(nn->d_policy); cudaFree(nn->d_value);
    nn->d_x = nullptr; nn->d_policy = nullptr; nn->d_value = nullptr;
    for (int i = 0; i < 3; ++i) AZ_CUDA(cudaMalloc(&nn->d_act[i], sizeof(float) * (size_t)n * 42 * AZ_NN_CH));
    AZ_CUDA(cudaMalloc(&nn->d_x, sizeof(float) * (size_t)n * 42 * nn->input_planes));
    AZ_CUDA(cudaMalloc(&nn->d_policy, sizeof(float) * (size_t)n * 43));
    AZ_CUDA(cudaMalloc(&nn->d_value, sizeof(float) * (size_t)n * nn->value_outputs));
    nn->cap = n;
    return AZ_OK;
}

AzHeadParams az_nn_head_params(const az_nn* nn)
{
    AzHeadParams hp;
    hp.pi_w = az_nn_dev_var(nn, "pi/kernel"); hp.bn_pi = az_nn_dev_var(nn, "bn_pi/gamma");
    hp.dense_w = az_nn_dev_var(nn, "dense/kernel"); hp.dense_b = az_nn_dev_var(nn, "dense/bias");
    hp.v_w = az_nn_dev_var(nn, "v/kernel"); hp.bn_v = az_nn_dev_var(nn, "bn_v/gamma");
    hp.dense1_w = az_nn_dev_var(nn, "dense_1/kernel"); hp.dense1_b = az_nn_dev_var(nn, "dense_1/bias");
    hp.dense2_w = az_nn_dev_var(nn, "dense_2/kernel"); hp.dense2_b = az_nn_dev_var(nn, "dense_2/bias");
    hp.vo = nn->value_outputs;
    return hp;
}

static int forward_fp32(az_nn* nn, const float* d_x, int n, float* d_policy, float* d_value, cudaStream_t s)
{
    float* buf[3] = { nn->d_act[0], nn->d_act[1], nn->d_act[2] };
    int cur = 0, tmp = 1, nxt = 2;
    if (nn->input_planes == AZ_NN_IN_CH6)
        k_nn_stem_fp32<AZ_NN_IN_CH6><<<n, 256, 0, s>>>(d_x, n, az_nn_dev_var(nn, "conv/kernel"), az_nn_dev_var(nn, "conv_bn/gamma"), buf[cur]);
    else k_nn_stem_fp32<AZ_NN_IN_CH><<<n, 256, 0, s>>>(d_x, n, az_nn_dev_var(nn, "conv/kernel"), az_nn_dev_var(nn, "conv_bn/gamma"), buf[cur]);
    AZ_CUDA(cudaGetLastError());
    dim3 grid((n + F32_BOARDS - 1) / F32_BOARDS, AZ_NN_CH / F32_CO);
    size_t smem = F32_SMEM_FLOATS * sizeof(float);
    for (int i = 0; i < nn->blocks; ++i) {
        std::string sfx = std::to_string(i) + block_letter(i);
        k_nn_conv_fp32<<<grid, 128, smem, s>>>(buf[cur], n, az_nn_dev_var(nn, "res" + sfx + "_branch2a/kernel"),
                                               az_nn_dev_var(nn, "bn" + sfx + "_branch2a/gamma"), nullptr, buf[tmp]);
        AZ_CUDA(cudaGetLastError());
        k_nn_conv_fp32<<<grid, 128, smem, s>>>(buf[tmp], n, az_nn_dev_var(nn, "res" + sfx + "_branch2b/kernel"),
                                               az_nn_dev_var(nn, "bn" + sfx + "_branch2b/gamma"), buf[cur], buf[nxt]);
        AZ_CUDA(cudaGetLastError());
        int o = cur; cur = nxt; nxt = o;
    }
    float* a = buf[cur];
    if (nn->value_outputs == 6) k_nn_heads_fp32<6><<<n, 256, 0, s>>>(a, n, az_nn_head_params(nn), d_policy, d_value);
    else k_nn_heads_fp32<1><<<n, 256, 0, s>>>(a, n, az_nn_head_params(nn), d_policy, d_value);
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

extern "C" int az_nn_forward_dev(az_nn* nn, const float* d_x, int n, float* d_policy, float* d_value, int precision, void* stream)
{
    AZ_REQUIRE(nn && d_x && d_policy && d_value, "NULL argument");
    AZ_REQUIRE(n > 0, "n must be positive");
    AZ_REQUIRE(precision == AZ_NN_FP32 || precision == AZ_NN_BF16, "precision must be AZ_NN_FP32 or AZ_NN_BF16");
    AzDeviceGuard guard(nn->device);
    int rc = finalize(nn); if (rc) return rc;
    rc = az_nn_reserve(nn, n); if (rc) return rc;
    if (precision == AZ_NN_BF16 && nn->input_planes == AZ_NN_IN_CH6) return az_nn_tc_forward_planes16(nn, d_x, n, d_policy, d_value, (cudaStream_t)stream);
    if (precision == AZ_NN_BF16 && nn->value_outputs == 6) return az_nn_tc_forward_value6(nn, d_x, n, d_policy, d_value, (cudaStream_t)stream);
    if (precision == AZ_NN_BF16) return az_nn_tc_forward(nn, d_x, nullptr, n, d_policy, d_value, (cudaStream_t)stream);
    return forward_fp32(nn, d_x, n, d_policy, d_value, (cudaStream_t)stream);
}

extern "C" int az_nn_forward(az_nn* nn, const float* h_x, int n, float* h_policy, float* h_value, int precision, void* stream)
{
    AZ_REQUIRE(nn && h_x && h_policy && h_value, "NULL argument");
    AZ_REQUIRE(n > 0, "n must be positive");
    AzDeviceGuard guard(nn->device);
    cudaStream_t s = (cudaStream_t)stream;
    int rc = finalize(nn); if (rc) return rc;
    rc = az_nn_reserve(nn, n); if (rc) return rc;
    AZ_CUDA(cudaMemcpyAsync(nn->d_x, h_x, sizeof(float) * (size_t)n * 42 * nn->input_planes, cudaMemcpyHostToDevice, s));
    rc = az_nn_forward_dev(nn, nn->d_x, n, nn->d_policy, nn->d_value, precision, stream);
    if (rc) return rc;
    AZ_CUDA(cudaMemcpyAsync(h_policy, nn->d_policy, sizeof(float) * (size_t)n * 43, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaMemcpyAsync(h_value, nn->d_value, sizeof(float) * (size_t)n * nn->value_outputs, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    return AZ_OK;
}
