// trainer_nets.cuh -- what trainer.cu (the cn_trainer_* entry points, SGD / reduce kernels) and trainer_nets.cu (the forward
// + backward kernels of every value network) share: one parameter layer of the flat block, the network description and the
// host interface of the forward + backward step.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

// One weight matrix of the flat master block (torch state-dict order).  w_off / b_off: its weight [out][in] and bias in the
// block; t_off: its block in the transposed copy Wt -- [in][out] followed by the bias, both padded to 4 floats, 16-byte
// aligned (one cp.async target); a_off: its block in the aligned copy Wa of the ORIGINAL [out][in] layout (what the
// backward-data products read).  LSTM-RL's nn.LSTM is two such layers, weight_ih / bias_ih and weight_hh / bias_hh.
struct TLayer { int in, out; int w_off, b_off, t_off, a_off; };

constexpr int kNetMaxLayers = 11;     // SARL: mlp1 (2) + mlp2 (2) + attention (3) + mlp3 (4)
constexpr int kNetMaxOps = 2 * kNetMaxLayers;

// SARL / OM-SARL (net = CN_NET_SARL): L[0..10] = mlp1.{0,2}, mlp2.{0,2}, attention.{0,2,4}, mlp3.{0,2,4,6}.
// CADRL (CN_NET_CADRL): L[0..3] = value_network.{0,2,4,6}, one row per sample.
// LSTM-RL (CN_NET_LSTM_RL): [L[0..3] = mlp1.{0,2,4,6} (ValueNetwork2)], then mlp.{0,2,4,6}, weight_ih, weight_hh.
// ops: the weight blocks in the order the kernel stages them, op_layer[k] = layer, op_bwd[k] = 1 for a backward-data
// product (block from Wa, no bias) and 0 for a forward layer (block from Wt, bias behind the weights).
struct NetDims {
    int net, n_layers;
    TLayer L[kNetMaxLayers];
    int n_params, t_size, a_size;
    int in, self_dim;
    int no_gs;                 // SARL without the global state: attention.0's input is e (L[4].in = L[1].out), not [e | mean]
    int vn2;                   // LSTM-RL with the per-row mlp1 in front of the LSTM
    int lstm_h, lstm_in;
    int mlp0;                  // first layer of the value mlp (0 for CADRL and ValueNetwork1, 4 for ValueNetwork2)
    int ih, hh;                // layers of weight_ih / weight_hh
    int n_ops;
    int8_t op_layer[kNetMaxOps], op_bwd[kNetMaxOps];
    int wbuf_floats;           // size of one staging buffer = the largest block
};

// The learned human-motion models (world_trainer.cu), next to the value networks' CN_NET_* kinds:
// AttentionWorld: L[0..10] = mlp1.{0,2}, mlp2.{0,2}, attention.{0,2,4}, mlp3.{0,2,4,6} -- SARL's layers, in = 4, mlp3 on
//   every human row with 2 outputs; one sample (H rows) per CTA.
// MlpWorld: L[0..3] = mlp.{0,3,6,8} (4H -> 128 -> 64 -> 12 -> 2H, tanh at the end); several samples per CTA.
constexpr int kNetWorldAttention = 16;
constexpr int kNetWorldMlp = 17;

// What a world-model step adds to a value-network step: inverted dropout after the ReLUs of MlpWorld's layers 0 and 1
// (p = 0: none), and the forward-only form (validation: squared errors only, no gradient).
struct WorldStep {
    float p;                   // drop probability
    uint64_t seed;
    uint32_t step;             // the mask of (sample position, layer, unit) is a Philox draw keyed by (seed, step)
    uint8_t *mask;             // optional [batch][L[0].out + L[1].out]: 1 = unit kept
    int fwd_only;
};

// 227 kB: the opt-in dynamic shared memory of one CTA on sm_100
constexpr size_t kTrainerMaxSmem = 232448;

// Samples per CTA of the network (one SARL, LSTM-RL or AttentionWorld sample per CTA, several CADRL / MlpWorld rows).
int trainer_spc(const NetDims &d);
// Shared memory of one CTA: activations for `H` humans and nbuf staging buffers (bytes).
size_t trainer_smem(const NetDims &d, int H, int nbuf);
// The network's kernel may use kTrainerMaxSmem (call after cudaSetDevice).
cudaError_t trainer_configure(const NetDims &d);
// Forward + backward of `batch` samples (item index[s] of X / target, or sample s itself when index is NULL) -> per-CTA
// partial gradients gpart[cta][n_params] and squared errors loss_part[cta]; *nparts = CTAs launched.  The world models
// need `w` (their targets are batch x H x 2 velocities); with w->fwd_only the op list of d must end after the forward.
int trainer_launch(const NetDims &d, const float *Wt, const float *Wa, const float *X, const float *target,
                   const int64_t *index, int batch, int H, float *gpart, float *loss_part, int *nparts, cudaStream_t s,
                   const WorldStep *w = nullptr);

// The transposed / aligned weight copies of d.L (t_off, a_off, t_size, a_size, wbuf_floats; trainer.cu) and the maps from
// the flat block into them (flat index -> Wt index, -> Wa index).
void trainer_layout(NetDims &d);
void trainer_maps(const NetDims &d, int32_t *tmap, int32_t *amap);
// Wt / Wa <- the flat block W (trainer.cu)
int trainer_refresh(int n_params, const float *W, float *Wt, float *Wa, const int32_t *tmap, const int32_t *amap, cudaStream_t s);
