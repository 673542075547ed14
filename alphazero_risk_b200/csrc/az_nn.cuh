// az_nn.cuh — internal declarations shared by az_nn.cu (weights, fp32 forward, ABI),
// az_nn_tc.cu (bf16 tcgen05 tower) and az_mcts.cu (leaf evaluation).
#pragma once

#include <map>
#include <string>
#include <vector>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "az_b200.h"

#define AZ_NN_CH 256          // FILTERS, python/src/build_graph.py:32
#define AZ_NN_IN_CH 13        // FEATURES (INPUT_VECTOR_TYPE_2), build_graph.py:18
#define AZ_NN_IN_CH6 16       // the six-player seat planes (SIXPLAYER.md §2, az_nn_create_planes)
#define AZ_NN_BN_EPS 0.001f   // tf.layers.batch_normalization default epsilon (GraphDef: 0.0010000000474974513)

struct AzVar {
    std::string name;
    std::vector<int> shape;
    size_t count = 0, offset = 0;
    float glorot_limit = 0.0f, init_const = 0.0f;
};

struct AzHeadParams {
    const float *pi_w, *bn_pi, *dense_w, *dense_b, *v_w, *bn_v, *dense1_w, *dense1_b, *dense2_w, *dense2_b;
    int vo;                           // value outputs: 1, or 6 (seat (cur + k) % 6); dense2_w is [256][vo]
};

struct AzTcState;   // az_nn_tc.cu
struct AzTrainState; // az_nn_train.cu

struct az_nn {
    int blocks = 5, device = 0;
    int value_outputs = 1;            // 1 = the reference graph; 6 = the six-seat value vector (SIXPLAYER.md §2)
    int input_planes = AZ_NN_IN_CH;   // 13 = the reference graph; 16 = the six-player seat planes (SIXPLAYER.md §2)
    std::vector<AzVar> vars;
    std::map<std::string, int> index;
    std::vector<float> blob;          // every variable, fp32, TF layouts (HWIO kernels), inventory order
    bool finalized = false;           // d_blob == blob and the packed bf16 tiles are current
    bool host_stale = false;          // training has moved d_blob ahead of blob (synced back by az_nn_sync_host)
    float* d_blob = nullptr;          // device copy of blob
    int cap = 0;                      // positions the work buffers are sized for
    float* d_act[3] = { nullptr, nullptr, nullptr };   // fp32 activations [cap][42][256]
    float* d_x = nullptr; float* d_policy = nullptr; float* d_value = nullptr;   // staging for host-buffer calls (d_x: [cap][42][input_planes])
    AzTcState* tc = nullptr;
    AzTrainState* train = nullptr;    // optimizer state + training work buffers, created on first use
};

const float* az_nn_host_var(const az_nn* nn, const std::string& name);
const float* az_nn_dev_var(const az_nn* nn, const std::string& name);
AzHeadParams az_nn_head_params(const az_nn* nn);
int az_nn_reserve(az_nn* nn, int n);
int az_nn_sync_host(az_nn* nn);            // copies trained weights back into nn->blob when they are ahead
void az_nn_train_release(az_nn* nn);        // az_nn_train.cu

// bf16 tensor-core path (az_nn_tc.cu)
int az_nn_tc_prepare(az_nn* nn);            // fold BN, pack bf16 weight tiles; called by finalize
void az_nn_tc_release(az_nn* nn);
// x: fp32 [n][7][6][13] (or NULL when env_state is given: encode fused into the stem; env_state = SoA words with stride
// state_stride >= n between words, 0 = n)
// scratch_set: which of the two sets of work buffers to use (two forwards of one network may be in flight on two streams);
// shared_device: another forward shares the device right now (no programmatic dependent launch between the layers, see az_nn_tc.cu)
int az_nn_tc_forward(az_nn* nn, const float* d_x, const uint32_t* d_env_state, int n, float* d_policy, float* d_value, cudaStream_t s,
                     int state_stride = 0, int scratch_set = 0, bool shared_device = false);
// the same forward for a network with six value outputs: value [n][6] (az_nn_tc_value6.cu)
int az_nn_tc_forward_value6(az_nn* nn, const float* d_x, int n, float* d_policy, float* d_value, cudaStream_t s);
// the forward of a network with 16 input planes, x fp32 [n][7][6][16], one or six value outputs (az_nn_tc_value6.cu)
int az_nn_tc_forward_planes16(az_nn* nn, const float* d_x, int n, float* d_policy, float* d_value, cudaStream_t s);

// raw 3x3 convolution of the training step on the tower kernel (az_nn_tc.cu): fp32 [n * 42][256] in, fp32 HWIO device weights
// [9][256][256] (flip = 1: the data gradient's kernel), fp32 [n * 42][256] out; bf16 operands, fp32 accumulation
// The chunked bf16 board layout of the tensor-core kernels: [channel chunk of 8][row][8 channels], AZ_TC_RPB rows per board —
// cell (y, x) at row y*6 + x, then six zero rows.  Six is the minimum: a vertical tap reaches 6 rows up or down, and the seventh row a
// diagonal tap would reach (the previous board's cell (6,5), the next board's cell (0,0)) is exactly a cell the x-masked operand
// copy of that tap zeroes (az_nn_tc.cu).  42 of 48 rows carry data (the first version had 49 rows; 56 before the masked copies).
#define AZ_TC_RPB 48
#define AZ_TC_HALO 8                   // zero rows in front of the first board (az_nn_tc.cu: TC_HALO)
struct AzTcConvScratch {
    int cap_boards = 0, r_alloc = 0, max_pairs = 0, n_sm = 148, dz_boards = 0;
    std::vector<__nv_bfloat16*> a_rpb;    // per tower layer: the layer's activation in the chunked layout (written by the fused BN kernel)
    __nv_bfloat16* d_in = nullptr;      // [32][r_alloc][8], AZ_TC_RPB rows per board: the tensor being convolved / the weight gradient's activation
    __nv_bfloat16* d_in3 = nullptr;     // [3][32][r_alloc][8]: a layer's dz — plain, x = 0 cells zeroed, x = 5 cells zeroed
    uint8_t* d_w = nullptr;             // one layer's packed stages
};
int az_tc_conv_raw_reserve(AzTcConvScratch* sc, int n);
int az_tc_conv_raw(AzTcConvScratch* sc, const float* d_src, int n, const float* d_w, int flip, float* d_out, cudaStream_t s);
// backward of one 256 -> 256 layer: convert dz once, then the weight gradient (k_tc_wgrad, MN-major operands straight from the chunked
// buffers) and the data gradient (tower kernel on the flipped + transposed weights) read it
int az_tc_dz_prepare(AzTcConvScratch* sc, const float* d_dz, int n, cudaStream_t s);
int az_tc_wgrad_prepared(AzTcConvScratch* sc, const float* d_a, int n, float* d_part, int max_splits, int* splits_out, cudaStream_t s);
int az_tc_dgrad_prepared(AzTcConvScratch* sc, int n, const float* d_w, float* d_out, cudaStream_t s);
// the fused BatchNorm kernels of az_nn_train.cu write the chunked copies themselves: per-layer activation buffers, the dz target
int az_tc_layers_reserve(AzTcConvScratch* sc, int n, int layers);
int az_tc_dz_target(AzTcConvScratch* sc, int n, cudaStream_t s, __nv_bfloat16** d_dz3, size_t* var_stride_u4);
int az_tc_conv_raw_rpb(AzTcConvScratch* sc, const __nv_bfloat16* in_rpb, int n, const float* d_w, int flip, float* d_out, cudaStream_t s);
int az_tc_wgrad_rpb(AzTcConvScratch* sc, const __nv_bfloat16* a_rpb, int n, float* d_part, int max_splits, int* splits_out, cudaStream_t s);
void az_tc_conv_raw_release(AzTcConvScratch* sc);
