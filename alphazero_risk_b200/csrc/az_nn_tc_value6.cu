// az_nn_tc_value6.cu — the translation unit of the bf16 tensor-core forward: az_nn_tc.cu itself (included byte for byte: the ncu capture
// of its tower kernel in profiles/traffic.json is keyed by that file's hash) plus the value tail of a network with six value outputs
// (SIXPLAYER.md §2, az_nn_create_value) and the input side of a network with 16 input planes (the seat planes, az_nn_create_planes),
// and the test entries that read the forward's work buffers (AzTcState and AzTcScratch are defined only in az_nn_tc.cu).
//
// A six-output network shares everything with the one-output graph up to dense_1: the same tower, the same 1x1 head convolutions (whose
// per-cell sums the last tower layer's epilogue writes to d_head_z) and the same policy head.  So its forward is az_nn_tc_forward
// unchanged — policy bit for bit what a one-output network with the same shared weights gives — followed by k_nn_value6_tail, which
// reads d_head_z again and writes value [n][6] over the scalar the one-output tail left in the first n entries.
#define az_nn_tc_prepare az_nn_tc_prepare_13
#include "az_nn_tc.cu"
#undef az_nn_tc_prepare
#include "az_tc_gemm.cuh"

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

// ---------------------------------------------------------------- 16 input planes (SIXPLAYER.md §2, "seat planes")
// The stem's bf16 operand has two chunks of 8 channels whatever the plane count: 13 planes leave channels 13..15 zero, 16 planes fill
// them.  So a 16-plane network runs the same stem kernel (k_nn_conv_tc<2, true, 3>), tower and heads; only its weight stages and its
// input packing differ.

// finalize's bf16 preparation: az_nn_tc.cu packs the stem as [3][3][13][256] (channels 13..15 zero); a 16-plane network's stem stages
// are packed again from all 16 channels before anything reads them
int az_nn_tc_prepare(az_nn* nn)
{
    int rc = az_nn_tc_prepare_13(nn);
    if (rc || nn->input_planes == AZ_NN_IN_CH) return rc;
    std::vector<uint8_t> packed((size_t)TC_STEM_BYTES);
    pack_conv(az_nn_host_var(nn, "conv/kernel"), AZ_NN_IN_CH6, 2, reinterpret_cast<__nv_bfloat16*>(packed.data()));
    AZ_CUDA(cudaMemcpy(nn->tc->d_wpacked, packed.data(), packed.size(), cudaMemcpyHostToDevice));
    return AZ_OK;
}

// fp32 [n][42][16] -> bf16 [2 chunks][r_alloc][8], every channel data (no zero padding); thread = board cell.  The three copies
// var_stride elements apart (plain, x = 5 cells zeroed, x = 0 cells zeroed) as k_nn_pack_input_tc writes them
__global__ void __launch_bounds__(256) k_nn_pack_input16_tc(const float* __restrict__ x, int n, __nv_bfloat16* __restrict__ out, int r_alloc,
                                                             size_t var_stride)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n * 42) return;
    const int b = i / 42, p = i - b * 42;
    const float* src = x + (size_t)i * AZ_NN_IN_CH6;
    const int row = b * TC_RPB + p;
    const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        uint4 o;
        __nv_bfloat162* o2 = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
        for (int e = 0; e < 4; ++e) o2[e] = __floats2bfloat162_rn(src[c * 8 + 2 * e], src[c * 8 + 2 * e + 1]);
        const size_t at = ((size_t)c * r_alloc + TC_HALO + row) * 8;
        *reinterpret_cast<uint4*>(out + at) = o;
        *reinterpret_cast<uint4*>(out + var_stride + at) = (p % 6) == 5 ? zero : o;
        *reinterpret_cast<uint4*>(out + 2 * var_stride + at) = (p % 6) == 0 ? zero : o;
    }
}

// the bf16 forward of a 16-plane network (one or six value outputs): k_nn_pack_input16_tc, then the stem, the tower and the heads tail
// launched exactly as az_nn_tc_forward launches them, then k_nn_value6_tail for six outputs.  The layer loop repeats
// az_nn_tc_forward's because that function packs its input itself and az_nn_tc.cu cannot change (its hash keys the ncu captures).
int az_nn_tc_forward_planes16(az_nn* nn, const float* d_x, int n, float* d_policy, float* d_value, cudaStream_t s)
{
    AzTcState* st = nn->tc;
    if (!st || !st->d_wpacked) { az_set_error("network not finalized"); return AZ_ERR_NOT_READY; }
    AzTcScratch* tc = &st->scratch[0];
    int rc = tc_reserve(tc, n); if (rc) return rc;
    const int tiles = (n * TC_RPB + TC_TILE_ROWS - 1) / TC_TILE_ROWS;
    const int grid = tiles < st->n_sm ? tiles : st->n_sm;
    const int layers = 2 * nn->blocks;
    int cur = 0, tmp = 1, nxt = 2;
    k_nn_pack_input16_tc<<<(n * 42 + 255) / 256, 256, 0, s>>>(d_x, n, tc->d_in, tc->r_alloc, tc->in_var_stride);
    AZ_CUDA(cudaGetLastError());
    AZ_CUDA((launch_conv<2, true, 3>(grid, s, tc->d_in, st->d_wpacked, st->d_scale + layers * 256, st->d_shift + layers * 256, nullptr, tc->d_act[cur], n,
                                     tc->r_alloc, tiles, tc->in_var_stride * 2)));
    const int pitems = (tiles + 1) / 2;
    const int pgrid = 2 * (pitems < st->max_pairs ? pitems : st->max_pairs);
    for (int i = 0; i < nn->blocks; ++i) {
        for (int h = 0; h < 2; ++h) {                        // branch2a: cur -> tmp; branch2b: tmp (+ cur as the residual) -> nxt
            const int L = 2 * i + h;
            const __nv_bfloat16* src = h ? tc->d_act[tmp] : tc->d_act[cur];
            const __nv_bfloat16* res = h ? tc->d_act[cur] : nullptr;
            __nv_bfloat16* dst = h ? tc->d_act[nxt] : tc->d_act[tmp];
            const bool last = L == layers - 1;              // the last layer feeds the heads directly: no activation store
            AZ_CUDA(launch_conv_pair3(pgrid, s, src, st->d_wpacked3 + (size_t)L * TC_LAYER_BYTES, st->d_scale + L * 256, st->d_shift + L * 256, res, dst, n,
                                      tc->r_alloc, tiles, last ? st->d_head_w : nullptr, last ? tc->d_head_z : nullptr));
        }
        int o = cur; cur = nxt; nxt = o;
    }
    k_nn_heads_tail<<<(n + HB - 1) / HB, 256, 0, s>>>(tc->d_head_z, n, az_nn_head_params(nn), d_policy, d_value);
    AZ_CUDA(cudaGetLastError());
    if (nn->value_outputs == 6) {
        k_nn_value6_tail<<<(n + HB - 1) / HB, 256, 0, s>>>(tc->d_head_z, n, az_nn_head_params(nn), d_value);
        AZ_CUDA(cudaGetLastError());
    }
    return AZ_OK;
}

// ---------------------------------------------------------------- test introspection (tests/test_tc_operands_gpu.py)
// The work buffers of the bf16 forward and the training step's tensor-core contractions, for tests that check every contraction on the
// operands it actually read against an fp64 reference.  Neither entry changes what a production call computes.

// one buffer of scratch set `s` as of the last bf16 forward that used it: which = 0 the stem operand d_in (bf16 bits, [3 copies][2 chunks]
// [r_alloc][8]), 1..3 d_act[0..2] (bf16 bits, [32][r_alloc][8], halos and padding rows included), 4 d_head_z (float4 [n][42]).
// h_out == NULL with bytes == 0 only reports r_alloc (0 before the first forward).
extern "C" int az_nn_tc_probe(az_nn* nn, int s, int which, int n, void* h_out, size_t bytes, int* r_alloc)
{
    AZ_REQUIRE(nn && nn->tc, "no bf16 forward state on this network");
    AZ_REQUIRE(s >= 0 && s < AZ_TC_SCRATCH_SETS, "scratch set out of range");
    AZ_REQUIRE(which >= 0 && which <= 4, "which must be 0 (input), 1..3 (activation buffers) or 4 (head sums)");
    const AzTcScratch& tc = nn->tc->scratch[s];
    if (r_alloc) *r_alloc = tc.r_alloc;
    if (!h_out && bytes == 0) return AZ_OK;
    AZ_REQUIRE(h_out != nullptr, "h_out is NULL");
    AZ_REQUIRE(tc.cap_boards > 0, "no bf16 forward has run on this scratch set");
    AZ_REQUIRE(n >= 1 && n <= tc.cap_boards, "n out of range");
    const void* src = which == 0 ? (const void*)tc.d_in : which == 4 ? (const void*)tc.d_head_z : (const void*)tc.d_act[which - 1];
    const size_t want = which == 0 ? (size_t)3 * 2 * tc.r_alloc * 16 : which == 4 ? sizeof(float4) * (size_t)n * 42 : (size_t)TC_CHUNKS * tc.r_alloc * 16;
    AZ_REQUIRE(bytes == want, "byte count does not match the buffer");
    AzDeviceGuard guard(nn->device);
    AZ_CUDA(cudaDeviceSynchronize());
    AZ_CUDA(cudaMemcpy(h_out, src, bytes, cudaMemcpyDeviceToHost));
    return AZ_OK;
}

// The training step's tensor-core contractions through their production functions on fp32 host arrays (rounded to bf16 on the device):
//   mode 0: out[n * 42][256] = conv(a[n * 42][256], w = b[9][256][256] HWIO)          az_tc_conv_raw, flip = 0
//   mode 1: out[n * 42][256] = data gradient of dz = a through w = b                   az_tc_dz_prepare + az_tc_dgrad_prepared
//   mode 2: out[9][256][256] = weight gradient of activation a with dz = b [n * 42][256]  az_tc_dz_prepare + az_tc_wgrad_prepared
//           (at most max_splits K splits) + az_tg_reduce
// n_warm > n first runs the same mode at n_warm boards with other data on the same scratch, so the measured call reuses buffers a larger
// batch left dirty (and mode 1 / 2 take the n < dz_boards clearing path).
extern "C" int az_tc_conv_test(int mode, const float* h_a, const float* h_b, int n, int n_warm, int max_splits, float* h_out)
{
    AZ_REQUIRE(h_a && h_b && h_out, "NULL argument");
    AZ_REQUIRE(mode >= 0 && mode <= 2, "mode must be 0 (forward), 1 (data gradient) or 2 (weight gradient)");
    AZ_REQUIRE(n >= 1 && n_warm >= 0 && max_splits >= 1 && max_splits <= 64, "bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); az_set_error("no CUDA device: libaz_b200 has no CPU fallback"); return AZ_ERR_NO_DEVICE; }
    const int n_max = n_warm > n ? n_warm : n;
    const size_t rows_max = (size_t)n_max * 42 * 256, wsz = (size_t)9 * 256 * 256;
    const size_t b_elems = mode == 2 ? rows_max : wsz, out_elems = mode == 2 ? wsz : rows_max;
    AzTcConvScratch sc;
    float *d_a = nullptr, *d_b = nullptr, *d_out = nullptr, *d_part = nullptr;
    int rc = AZ_OK;
    cudaError_t ce = cudaMalloc(&d_a, rows_max * sizeof(float));
    if (ce == cudaSuccess) ce = cudaMalloc(&d_b, b_elems * sizeof(float));
    if (ce == cudaSuccess) ce = cudaMalloc(&d_out, out_elems * sizeof(float));
    if (ce == cudaSuccess && mode == 2) ce = cudaMalloc(&d_part, (size_t)max_splits * wsz * sizeof(float));
    auto run = [&](int nb) -> int {
        if (mode == 0) return az_tc_conv_raw(&sc, d_a, nb, d_b, 0, d_out, 0);
        int r = az_tc_dz_prepare(&sc, mode == 1 ? d_a : d_b, nb, 0); if (r) return r;
        if (mode == 1) return az_tc_dgrad_prepared(&sc, nb, d_b, d_out, 0);
        int splits = 0;
        r = az_tc_wgrad_prepared(&sc, d_a, nb, d_part, max_splits, &splits, 0); if (r) return r;
        return az_tg_reduce(d_part, splits, 9 * 256, 9 * 256, d_out, 0);
    };
    if (ce == cudaSuccess && n_warm > n) {
        // other data, exact in bf16: small multiples of 1/64 from a multiplicative hash of the index
        std::vector<float> wa(rows_max), wb(b_elems);
        for (size_t i = 0; i < wa.size(); ++i) wa[i] = (float)((uint32_t)(i * 2654435761u) >> 26) / 64.0f - 0.5f;
        for (size_t i = 0; i < wb.size(); ++i) wb[i] = mode == 2 ? (float)((uint32_t)(i * 2246822519u) >> 26) / 64.0f - 0.5f : h_b[i];
        ce = cudaMemcpy(d_a, wa.data(), wa.size() * sizeof(float), cudaMemcpyHostToDevice);
        if (ce == cudaSuccess) ce = cudaMemcpy(d_b, wb.data(), wb.size() * sizeof(float), cudaMemcpyHostToDevice);
        if (ce == cudaSuccess) rc = run(n_warm);
        if (ce == cudaSuccess && rc == AZ_OK) ce = cudaDeviceSynchronize();
    }
    const size_t a_elems = (size_t)n * 42 * 256;
    if (ce == cudaSuccess && rc == AZ_OK) ce = cudaMemcpy(d_a, h_a, a_elems * sizeof(float), cudaMemcpyHostToDevice);
    if (ce == cudaSuccess && rc == AZ_OK) ce = cudaMemcpy(d_b, h_b, (mode == 2 ? a_elems : wsz) * sizeof(float), cudaMemcpyHostToDevice);
    if (ce == cudaSuccess && rc == AZ_OK) rc = run(n);
    if (ce == cudaSuccess && rc == AZ_OK) ce = cudaDeviceSynchronize();
    if (ce == cudaSuccess && rc == AZ_OK) ce = cudaMemcpy(h_out, d_out, (mode == 2 ? wsz : a_elems) * sizeof(float), cudaMemcpyDeviceToHost);
    az_tc_conv_raw_release(&sc);
    cudaFree(d_a); cudaFree(d_b); cudaFree(d_out); cudaFree(d_part);
    if (ce != cudaSuccess) { az_set_error("az_tc_conv_test: %s", cudaGetErrorString(ce)); cudaGetLastError(); return AZ_ERR_CUDA; }
    return rc;
}
