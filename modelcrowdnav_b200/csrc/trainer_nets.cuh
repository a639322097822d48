// trainer_nets.cuh -- what trainer.cu (the cn_trainer_* entry points, SGD / reduce kernels) and trainer_nets.cu (the forward
// + backward kernel of CADRL and LSTM-RL) share: one parameter layer of the flat block and the network description.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

// One weight matrix of the flat master block (torch state-dict order).  w_off / b_off: its weight [out][in] and bias in the
// block; t_off: its block in the transposed copy Wt -- [in][out] followed by the bias, both padded to 4 floats, 16-byte
// aligned (one cp.async target); a_off: its block in the aligned copy Wa of the ORIGINAL [out][in] layout (what the
// backward-data products read).  LSTM-RL's nn.LSTM is two such layers, weight_ih / bias_ih and weight_hh / bias_hh.
struct TLayer { int in, out; int w_off, b_off, t_off, a_off; };

constexpr int kNetMaxLayers = 10;     // LSTM-RL ValueNetwork2: mlp1 (4) + mlp (4) + weight_ih + weight_hh
constexpr int kNetMaxOps = 2 * kNetMaxLayers;

// CADRL (net = CN_NET_CADRL): L[0..3] = value_network.{0,2,4,6}, one row per sample.
// LSTM-RL (CN_NET_LSTM_RL): [L[0..3] = mlp1.{0,2,4,6} (ValueNetwork2)], then mlp.{0,2,4,6}, weight_ih, weight_hh.
// ops: the weight blocks in the order the kernel stages them, op_layer[k] = layer, op_bwd[k] = 1 for a backward-data
// product (block from Wa, no bias) and 0 for a forward layer (block from Wt, bias behind the weights).
struct NetDims {
    int net, n_layers;
    TLayer L[kNetMaxLayers];
    int n_params, t_size, a_size;
    int in, self_dim;
    int vn2;                   // LSTM-RL with the per-row mlp1 in front of the LSTM
    int lstm_h, lstm_in;
    int mlp0;                  // first layer of the value mlp (0 for CADRL and ValueNetwork1, 4 for ValueNetwork2)
    int ih, hh;                // layers of weight_ih / weight_hh
    int n_ops;
    int8_t op_layer[kNetMaxOps], op_bwd[kNetMaxOps];
    int wbuf_floats;           // size of one staging buffer = the largest block
};

// Samples per CTA of the network (several CADRL rows share one CTA; one LSTM sequence per CTA).
int trainer_nets_spc(const NetDims &d);
// Shared memory of one CTA: activations for `H` humans and nbuf staging buffers (bytes).
size_t trainer_nets_smem(const NetDims &d, int H, int nbuf);
// The kernel's shared-memory limit (call after cudaSetDevice).
cudaError_t trainer_nets_configure();
// Forward + backward of `batch` samples -> per-CTA partial gradients gpart[cta][n_params] and squared errors loss_part[cta];
// *nparts = CTAs launched.  Same arguments as trainer_fwd_bwd_kernel.
int trainer_nets_launch(const NetDims &d, const float *Wt, const float *Wa, const float *X, const float *target,
                        const int64_t *index, int batch, int H, float *gpart, float *loss_part, int *nparts, cudaStream_t s);
