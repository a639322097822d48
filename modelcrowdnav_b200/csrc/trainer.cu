// trainer.cu -- one optimisation step of a value network on the device (FP32):
//   MSE( ValueNetwork(states), targets ) -> backward -> [gradient all-reduce by the caller] -> SGD with momentum.
// Replaces the ~150 kernel launches (+ one host sync) of the torch autograd step the reference runs per batch
// (crowd_nav/utils/trainer.py:61-82: zero_grad, model(inputs), MSELoss, backward, SGD(momentum 0.9).step, loss.item())
// with TWO kernels:
//   forward + backward       the network's kernel in trainer_nets.cu (trainer_launch): the whole forward and backward of a
//                            few samples per CTA with every activation in shared memory and the weight blocks staged in
//                            the order of the op list built here -> per-CTA partial weight gradients gpart[cta][n_params]
//   trainer_reduce_kernel    fixed-order sum of the partials (deterministic) -> gradient; with grad_out == NULL it also
//                            applies SGD momentum in place and refreshes the transposed weight copy the forward reads
//   trainer_apply_kernel     the SGD half alone, for the data-parallel form (gradient -> NCCL all-reduce -> apply)
//
// Parameter layout = the torch state-dict order of the value network, the same flat block cn_policy_load_weights takes,
// derived from the same layer list (cn_layers), so the torch model's parameters can be VIEWS of the block this trainer
// updates.  SARL: mlp1.0, mlp1.2, mlp2.0, mlp2.2, attention.0, .2, .4, mlp3.0, .2, .4, .6 (weight [out][in] then bias);
// with occupancy maps mlp1.0 reads 13 + cell_num^2 * om_channel_size columns.  CADRL: value_network.{0,2,4,6}.  LSTM-RL:
// [mlp1.*] mlp.* lstm.weight_ih_l0, weight_hh_l0, bias_ih_l0, bias_hh_l0.
#include "cn_common.cuh"
#include "dense_f32.cuh"
#include "trainer_nets.cuh"

#include <string.h>

#include <vector>

namespace {

using dense_f32::pad4;
constexpr int kMaxH = 16;         // humans per sample supported by the shared-memory plans

// gradient = fixed-order sum of the per-CTA partials; loss = sum of the partial squared errors / B.
// grad_out != NULL: write the gradient (the caller all-reduces it, then trainer_apply_kernel).
// grad_out == NULL: apply SGD with momentum in place (torch.optim.SGD: buf = mu * buf + g; w -= lr * buf) and refresh Wt.
__global__ void trainer_reduce_kernel(int n_params, int nparts, const float *__restrict__ gpart, const float *__restrict__ loss_part,
                                      int B, float *__restrict__ grad_out, float *__restrict__ W, float *__restrict__ Wt,
                                      float *__restrict__ Wa, float *__restrict__ mom, const int32_t *__restrict__ tmap,
                                      const int32_t *__restrict__ amap, float lr, float mu, float *__restrict__ loss_out,
                                      int loss_accumulate)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0 && loss_out) {
        float s = 0.0f;
        for (int c = 0; c < nparts; ++c) s += loss_part[c];
        *loss_out = (loss_accumulate ? *loss_out : 0.0f) + s / (float)B;
    }
    if (i >= n_params) return;
    float g = 0.0f;
    for (int c = 0; c < nparts; ++c) g += gpart[(size_t)c * n_params + i];
    if (grad_out) { grad_out[i] = g; return; }
    const float b = mu * mom[i] + g;
    mom[i] = b;
    const float w = W[i] - lr * b;
    W[i] = w;
    Wt[tmap[i]] = w;
    if (amap[i] >= 0) Wa[amap[i]] = w;
}

__global__ void trainer_apply_kernel(int n_params, const float *__restrict__ grad, float scale, float *__restrict__ W,
                                     float *__restrict__ Wt, float *__restrict__ Wa, float *__restrict__ mom,
                                     const int32_t *__restrict__ tmap, const int32_t *__restrict__ amap, float lr, float mu)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_params) return;
    const float b = mu * mom[i] + grad[i] * scale;
    mom[i] = b;
    const float w = W[i] - lr * b;
    W[i] = w;
    Wt[tmap[i]] = w;
    if (amap[i] >= 0) Wa[amap[i]] = w;
}

__global__ void trainer_transpose_kernel(int n_params, const float *__restrict__ W, float *__restrict__ Wt, float *__restrict__ Wa,
                                         const int32_t *__restrict__ tmap, const int32_t *__restrict__ amap)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_params) return;
    Wt[tmap[i]] = W[i];
    if (amap[i] >= 0) Wa[amap[i]] = W[i];
}

}  // namespace

struct cn_trainer {
    int device;
    NetDims d;
    int max_batch, max_humans;
    float *Wt, *Wa, *mom, *gpart, *loss_part;     // transposed / aligned weight copies, momentum, per-CTA partials
    int32_t *tmap, *amap;                         // flat parameter index -> index in Wt / Wa (-1: not in Wa)
    int nparts_cap;
};

void trainer_layout(NetDims &d)
{
    int toff = 0, aoff = 0;
    d.wbuf_floats = 0;
    for (int i = 0; i < d.n_layers; ++i) {
        TLayer &l = d.L[i];
        l.t_off = toff; toff += pad4(l.in * l.out) + pad4(l.out);      // [in][out] | bias, 16-byte aligned blocks
        l.a_off = aoff; aoff += pad4(l.in * l.out);                    // [out][in]
        const int blk = pad4(l.in * l.out) + pad4(l.out);
        if (blk > d.wbuf_floats) d.wbuf_floats = blk;
    }
    d.t_size = toff; d.a_size = aoff;
}

void trainer_maps(const NetDims &d, int32_t *tmap, int32_t *amap)
{
    for (int i = 0; i < d.n_params; ++i) amap[i] = -1;
    for (int i = 0; i < d.n_layers; ++i) {
        const TLayer &l = d.L[i];
        for (int o = 0; o < l.out; ++o)
            for (int k = 0; k < l.in; ++k) {
                tmap[l.w_off + o * l.in + k] = l.t_off + k * l.out + o;
                amap[l.w_off + o * l.in + k] = l.a_off + o * l.in + k;
            }
        for (int o = 0; o < l.out; ++o) tmap[l.b_off + o] = l.t_off + pad4(l.in * l.out) + o;
    }
}

int trainer_refresh(int n_params, const float *W, float *Wt, float *Wa, const int32_t *tmap, const int32_t *amap, cudaStream_t s)
{
    trainer_transpose_kernel<<<(n_params + 255) / 256, 256, 0, s>>>(n_params, W, Wt, Wa, tmap, amap);
    CN_LAUNCH_CHECK();
    return CN_OK;
}

// The weight matrices of the flat block in state-dict order, from the layer list the lookahead loads (cn_layers): a Linear
// is one TLayer, the LSTM block two (weight_ih with bias_ih, weight_hh with bias_hh).  Fills d.L / n_layers (w_off / b_off),
// the parameter count, and through trainer_layout the Wt / Wa blocks and wbuf_floats = the largest staged block.
static void trainer_layers(const cn_sarl_cfg *cfg, NetDims &d)
{
    SarlWeightsDev w;        // only the destinations of the layer list, never written here
    int off = 0, n = 0;
    for (const LayerSpec &l : cn_layers(cn_dims_of(cfg, 0), w)) {
        if (!l.dst_hh) {
            d.L[n++] = {l.in, l.out, off, off + l.in * l.out, 0, 0};
        } else {                                          // weight_ih_l0, weight_hh_l0, bias_ih_l0, bias_hh_l0
            const int hid = l.out / 4, whh = off + l.out * l.in, bih = whh + l.out * hid;
            d.L[n++] = {l.in, l.out, off, bih, 0, 0};
            d.L[n++] = {hid, l.out, whh, bih + l.out, 0, 0};
        }
        off += (int)cn_layer_floats(l);
    }
    d.n_layers = n;
    d.n_params = off;
    trainer_layout(d);
}

// The rest of the network description (after trainer_layers) and the order in which its kernel stages the weight blocks
static void trainer_net_dims(const cn_sarl_cfg *cfg, NetDims &d)
{
    d.net = cfg->network;
    d.in = cfg->input_dim; d.self_dim = cfg->self_state_dim;
    d.no_gs = cfg->network == CN_NET_SARL && cfg->without_global_state ? 1 : 0;
    const bool lstm = cfg->network == CN_NET_LSTM_RL;
    d.vn2 = lstm && cfg->lstm_mlp1_dims[0] > 0;
    d.lstm_h = lstm ? cfg->lstm_hidden : 0;
    d.lstm_in = d.vn2 ? cfg->lstm_mlp1_dims[3] : cfg->input_dim;
    d.mlp0 = d.vn2 ? 4 : 0;
    d.ih = d.mlp0 + 4; d.hh = d.mlp0 + 5;
    int n = 0;
    auto push = [&](int layer, int bwd) { d.op_layer[n] = (int8_t)layer; d.op_bwd[n] = (int8_t)bwd; ++n; };
    if (cfg->network == CN_NET_SARL) {
        for (int i = 0; i < 11; ++i) push(i, 0);                               // forward, then the backward-data products
        for (int i : {10, 9, 8, 7, 3, 6, 5, 4, 2, 1}) push(i, 1);              // (mlp3, mlp2.2, attention, mlp2.0 into de, mlp1.2)
        d.n_ops = n;
        return;
    }
    if (lstm) {
        if (d.vn2) for (int i = 0; i < 4; ++i) push(i, 0);                    // mlp1
        push(d.ih, 0); push(d.hh, 0);                                          // x W_ih^T, then W_hh^T for the recurrence
    }
    for (int i = 0; i < 4; ++i) push(d.mlp0 + i, 0);                           // the value mlp
    for (int i = 3; i >= (lstm ? 0 : 1); --i) push(d.mlp0 + i, 1);             // its backward-data products (LSTM-RL: down to h_H)
    if (lstm) {
        push(d.hh, 1);                                                         // BPTT
        if (d.vn2) { push(d.ih, 1); for (int i = 3; i >= 1; --i) push(i, 1); }   // dx_t, then mlp1
    }
    d.n_ops = n;
}

extern "C" {

int cn_trainer_create(const cn_sarl_cfg *cfg, int device, int32_t max_batch, int32_t max_humans, cn_trainer **out)
{
    if (!cfg || !out) { cn_set_error("null argument"); return CN_EINVAL; }
    int rc = cn_check_net_cfg(cfg);
    if (rc) return rc;
    const int net = cfg->network;
    if (cfg->with_om) {
        const int om_in = 13 + cfg->cell_num * cfg->cell_num * cfg->om_channel_size;
        if (cfg->input_dim != om_in) {
            cn_set_error("with_om: input_dim %d must be 13 + cell_num^2 * om_channel_size = %d", cfg->input_dim, om_in); return CN_EINVAL;
        }
    }
    if (max_batch < 1 || max_humans < 1 || (net == CN_NET_SARL && max_humans > kMaxH)) {
        cn_set_error("1 <= max_humans <= %d, max_batch >= 1", kMaxH); return CN_EINVAL;
    }
    if (net == CN_NET_CADRL && max_humans != 1) {
        cn_set_error("CADRL trains on single-human states (cadrl.py:209): max_humans must be 1"); return CN_EINVAL;
    }
    if (max_humans > kMaxH) {
        cn_set_error("fused trainer: at most %d humans per sample (max_humans %d)", kMaxH, max_humans); return CN_EUNSUPPORTED;
    }
    if (net == CN_NET_LSTM_RL && cfg->lstm_hidden < 1) { cn_set_error("lstm_hidden >= 1 required"); return CN_EINVAL; }
    if (net == CN_NET_LSTM_RL && (cfg->self_state_dim < 1 || cfg->self_state_dim > cfg->input_dim)) {
        cn_set_error("1 <= self_state_dim <= input_dim required (the self state is the first columns of row 0)"); return CN_EINVAL;
    }
    NetDims d;
    memset(&d, 0, sizeof(d));
    trainer_layers(cfg, d);
    for (int i = 0; i < d.n_layers; ++i)
        if (d.L[i].in < 1 || d.L[i].out < 1) { cn_set_error("layer widths must be >= 1"); return CN_EINVAL; }
    if (net == CN_NET_SARL && (cfg->attn_dims[2] != 1 || cfg->mlp3_dims[3] != 1)) {
        cn_set_error("attention and mlp3 must end in 1 unit"); return CN_EINVAL;
    }
    if (net != CN_NET_SARL && cfg->mlp3_dims[3] != 1) { cn_set_error("the value mlp must end in 1 unit"); return CN_EINVAL; }
    trainer_net_dims(cfg, d);
    if ((rc = use_device(device))) return rc;
    if (trainer_smem(d, max_humans, 1) > kTrainerMaxSmem) {
        cn_set_error("fused trainer: %d humans per sample%s do not fit the shared-memory plan", max_humans,
                     net == CN_NET_LSTM_RL ? " at this lstm_hidden / layer widths" : "");
        return CN_EUNSUPPORTED;
    }
    const int n_params = d.n_params;
    std::vector<int32_t> tmap(n_params), amap(n_params);
    trainer_maps(d, tmap.data(), amap.data());
    cn_trainer *t = new cn_trainer();
    memset(t, 0, sizeof(*t));
    t->device = device; t->d = d; t->max_batch = max_batch; t->max_humans = max_humans;
    const int spc = trainer_spc(d);
    t->nparts_cap = (max_batch + spc - 1) / spc;
    if (cudaMalloc((void **)&t->Wt, sizeof(float) * d.t_size) != cudaSuccess ||
        cudaMalloc((void **)&t->Wa, sizeof(float) * d.a_size) != cudaSuccess ||
        cudaMalloc((void **)&t->mom, sizeof(float) * n_params) != cudaSuccess ||
        cudaMalloc((void **)&t->gpart, sizeof(float) * (size_t)n_params * t->nparts_cap) != cudaSuccess ||
        cudaMalloc((void **)&t->loss_part, sizeof(float) * t->nparts_cap) != cudaSuccess ||
        cudaMalloc((void **)&t->tmap, sizeof(int32_t) * n_params) != cudaSuccess ||
        cudaMalloc((void **)&t->amap, sizeof(int32_t) * n_params) != cudaSuccess) {
        cn_set_error("cudaMalloc failed in cn_trainer_create");
        cn_trainer_destroy(t);
        return CN_ENOMEM;
    }
    // (the padding floats of the blocks are read by cp.async, hence the memsets)
    cudaError_t ce = cudaMemset(t->Wt, 0, sizeof(float) * d.t_size);
    if (ce == cudaSuccess) ce = cudaMemset(t->Wa, 0, sizeof(float) * d.a_size);
    if (ce == cudaSuccess) ce = cudaMemset(t->mom, 0, sizeof(float) * n_params);
    if (ce == cudaSuccess) ce = cudaMemcpy(t->tmap, tmap.data(), sizeof(int32_t) * n_params, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess) ce = cudaMemcpy(t->amap, amap.data(), sizeof(int32_t) * n_params, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess) ce = trainer_configure(d);
    if (ce != cudaSuccess) {
        cn_set_error("cn_trainer_create: %s", cudaGetErrorString(ce));
        cn_trainer_destroy(t);
        return CN_ECUDA;
    }
    *out = t;
    return CN_OK;
}

int cn_trainer_destroy(cn_trainer *t)
{
    if (!t) return CN_OK;
    cudaSetDevice(t->device);
    void *ptrs[] = {t->Wt, t->Wa, t->mom, t->gpart, t->loss_part, t->tmap, t->amap};
    for (void *q : ptrs) if (q) cudaFree(q);
    delete t;
    return CN_OK;
}

int64_t cn_trainer_param_count(const cn_trainer *t) { return t ? t->d.n_params : 0; }

int cn_trainer_sync_weights(cn_trainer *t, const float *w_dev, int zero_momentum, void *stream)
{
    if (!t || !w_dev) { cn_set_error("null argument"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(t->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int n = t->d.n_params;
    const int rc = trainer_refresh(n, w_dev, t->Wt, t->Wa, t->tmap, t->amap, s);
    if (rc) return rc;
    if (zero_momentum) CN_CUDA_CHECK(cudaMemsetAsync(t->mom, 0, sizeof(float) * n, s));
    return CN_OK;
}

static int trainer_step_impl(cn_trainer *t, float *w_dev, const float *states_dev, const float *targets_dev,
                             const int64_t *index_dev, int32_t batch, int32_t human_num, float lr, float momentum,
                             float *grad_out_dev, float *loss_dev, int loss_accumulate, void *stream)
{
    if (!t || !w_dev || !states_dev || !targets_dev) { cn_set_error("null argument"); return CN_EINVAL; }
    if (t->d.net == CN_NET_CADRL && human_num != 1) {
        cn_set_error("CADRL trains on single-human states (cadrl.py:209): human_num must be 1, got %d", human_num); return CN_EINVAL;
    }
    if (batch < 1 || batch > t->max_batch || human_num < 1 || human_num > t->max_humans) {
        cn_set_error("batch %d / human_num %d outside the trainer's capacity (%d, %d)", batch, human_num, t->max_batch, t->max_humans);
        return CN_EINVAL;
    }
    CN_CUDA_CHECK(cudaSetDevice(t->device));
    cudaStream_t s = (cudaStream_t)stream;
    int nparts = 0;
    const int rc = trainer_launch(t->d, t->Wt, t->Wa, states_dev, targets_dev, index_dev, batch, human_num, t->gpart, t->loss_part,
                                  &nparts, s);
    if (rc != CN_OK) return rc;
    const int n = t->d.n_params;
    trainer_reduce_kernel<<<(n + 255) / 256, 256, 0, s>>>(n, nparts, t->gpart, t->loss_part, batch, grad_out_dev, w_dev, t->Wt, t->Wa,
                                                         t->mom, t->tmap, t->amap, lr, momentum, loss_dev, loss_accumulate);
    CN_LAUNCH_CHECK();
    return CN_OK;
}

int cn_trainer_step(cn_trainer *t, float *w_dev, const float *states_dev, const float *targets_dev, int32_t batch,
                    int32_t human_num, float lr, float momentum, float *grad_out_dev, float *loss_dev, void *stream)
{
    return trainer_step_impl(t, w_dev, states_dev, targets_dev, nullptr, batch, human_num, lr, momentum, grad_out_dev, loss_dev, 0,
                             stream);
}

int cn_trainer_step_indexed(cn_trainer *t, float *w_dev, const float *memory_states_dev, const float *memory_values_dev,
                            const int64_t *index_dev, int32_t batch, int32_t human_num, float lr, float momentum,
                            float *grad_out_dev, float *loss_sum_dev, void *stream)
{
    if (!index_dev) { cn_set_error("index_dev is null"); return CN_EINVAL; }
    return trainer_step_impl(t, w_dev, memory_states_dev, memory_values_dev, index_dev, batch, human_num, lr, momentum, grad_out_dev,
                             loss_sum_dev, 1, stream);
}

int cn_trainer_apply(cn_trainer *t, float *w_dev, const float *grad_dev, float grad_scale, float lr, float momentum, void *stream)
{
    if (!t || !w_dev || !grad_dev) { cn_set_error("null argument"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(t->device));
    const int n = t->d.n_params;
    trainer_apply_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(n, grad_dev, grad_scale, w_dev, t->Wt, t->Wa, t->mom, t->tmap,
                                                                          t->amap, lr, momentum);
    CN_LAUNCH_CHECK();
    return CN_OK;
}

}  // extern "C"
