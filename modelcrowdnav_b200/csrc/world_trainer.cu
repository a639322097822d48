// world_trainer.cu -- one optimisation step of a learned human-motion model on the device (FP32):
//   MSELoss( AttentionWorld / MlpWorld (human states), next velocities ) -> backward -> [all-reduce by the caller] -> Adam.
// The model-based half of the fork trains its world model with torch autograd and torch.optim.Adam; here a step is TWO
// kernels, the pattern of the value-network trainer (trainer.cu):
//   forward + backward       world_attention_fwd_bwd_kernel / world_mlp_fwd_bwd_kernel (trainer_nets.cu, through
//                            trainer_launch): per-CTA partial gradients and squared errors
//   world_adam_reduce_kernel fixed-order sum of the partials (deterministic) -> gradient; with grad_out == NULL also Adam in
//                            place and the refresh of the transposed weight copies the forward reads
//   world_adam_apply_kernel  the Adam half alone, for the data-parallel form (gradient -> all-reduce -> apply)
// Parameter layout = the reference module's state-dict order (the block cn_world_load_weights takes): AttentionWorld mlp1.0,
// mlp1.2, mlp2.0, mlp2.2, attention.0, .2, .4, mlp3.0, .2, .4, .6; MlpWorld mlp.0, .3, .6, .8 (weight [out][in], then bias).
#include "cn_common.cuh"
#include "dense_f32.cuh"
#include "trainer_nets.cuh"

#include <math.h>
#include <string.h>

#include <vector>

namespace {

// torch.optim.Adam's per-parameter arithmetic (no weight decay, no amsgrad); the bias corrections come from the host
struct AdamArgs { float b1, omb1, b2, omb2, step_size, bc2_sqrt, eps; };

__device__ __forceinline__ float adam_update(float w, float g, float &m, float &v, const AdamArgs &a)
{
    m = a.b1 * m + a.omb1 * g;
    v = a.b2 * v + a.omb2 * g * g;
    const float denom = sqrtf(v) / a.bc2_sqrt + a.eps;
    return w - a.step_size * (m / denom);
}

// gradient = fixed-order sum of the per-CTA partials; *loss_out += sum of the partial squared errors / loss_div.
// grad_out != NULL: write the gradient.  grad_out == NULL: Adam in place, then refresh Wt / Wa.
__global__ void world_adam_reduce_kernel(int n_params, int nparts, const float *__restrict__ gpart, const float *__restrict__ loss_part,
                                         float loss_div, float *__restrict__ loss_out, float *__restrict__ grad_out,
                                         float *__restrict__ W, float *__restrict__ Wt, float *__restrict__ Wa, float *__restrict__ m,
                                         float *__restrict__ v, const int32_t *__restrict__ tmap, const int32_t *__restrict__ amap,
                                         AdamArgs a)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0 && loss_out) {
        float s = 0.0f;
        for (int c = 0; c < nparts; ++c) s += loss_part[c];
        *loss_out += s / loss_div;
    }
    if (i >= n_params || !gpart) return;
    float g = 0.0f;
    for (int c = 0; c < nparts; ++c) g += gpart[(size_t)c * n_params + i];
    if (grad_out) { grad_out[i] = g; return; }
    float mi = m[i], vi = v[i];
    const float w = adam_update(W[i], g, mi, vi, a);
    m[i] = mi; v[i] = vi;
    W[i] = w;
    Wt[tmap[i]] = w;
    if (amap[i] >= 0) Wa[amap[i]] = w;
}

__global__ void world_adam_apply_kernel(int n_params, const float *__restrict__ grad, float scale, float *__restrict__ W,
                                        float *__restrict__ Wt, float *__restrict__ Wa, float *__restrict__ m, float *__restrict__ v,
                                        const int32_t *__restrict__ tmap, const int32_t *__restrict__ amap, AdamArgs a)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_params) return;
    float mi = m[i], vi = v[i];
    const float w = adam_update(W[i], grad[i] * scale, mi, vi, a);
    m[i] = mi; v[i] = vi;
    W[i] = w;
    Wt[tmap[i]] = w;
    if (amap[i] >= 0) Wa[amap[i]] = w;
}

}  // namespace

struct cn_world_trainer {
    int device, kind, H, max_batch;
    float drop;
    NetDims d, d_fwd;                 // d_fwd: the same network with the op list cut after the forward (validation)
    float *Wt, *Wa, *m, *v, *gpart, *loss_part;
    int32_t *tmap, *amap;
    int nparts_cap;
    int synced;
    int64_t adam_t;                   // Adam steps taken (the bias corrections' t)
    uint32_t draws;                   // steps since the last optimizer reset: the dropout masks' Philox key
};

extern "C" {

int cn_world_trainer_create(int32_t kind, int32_t human_num, int device, int32_t max_batch, float drop_rate,
                            cn_world_trainer **out)
{
    if (!out) { cn_set_error("null argument"); return CN_EINVAL; }
    if (kind != CN_WORLD_ATTENTION && kind != CN_WORLD_MLP) { cn_set_error("unknown world model kind %d", kind); return CN_EINVAL; }
    if (human_num < 1 || human_num > CN_MAX_HUMANS || max_batch < 1) {
        cn_set_error("1 <= human_num <= %d and max_batch >= 1 required", CN_MAX_HUMANS); return CN_EINVAL;
    }
    if (!(drop_rate >= 0.0f && drop_rate < 1.0f)) { cn_set_error("drop_rate %g outside [0, 1)", (double)drop_rate); return CN_EINVAL; }
    if (kind == CN_WORLD_ATTENTION && drop_rate != 0.0f) { cn_set_error("AttentionWorld has no dropout: drop_rate must be 0"); return CN_EINVAL; }
    NetDims d;
    memset(&d, 0, sizeof(d));
    int ins[kNetMaxLayers], outs[kNetMaxLayers];
    d.n_layers = world_layer_dims(kind, human_num, ins, outs);
    int off = 0;
    for (int i = 0; i < d.n_layers; ++i) {
        d.L[i] = {ins[i], outs[i], off, off + ins[i] * outs[i], 0, 0};
        off += ins[i] * outs[i] + outs[i];
    }
    d.n_params = off;
    trainer_layout(d);
    d.in = ins[0];
    int n = 0;
    auto push = [&](int layer, int bwd) { d.op_layer[n] = (int8_t)layer; d.op_bwd[n] = (int8_t)bwd; ++n; };
    if (kind == CN_WORLD_ATTENTION) {
        d.net = kNetWorldAttention;
        d.self_dim = ins[0];
        for (int i = 0; i < 11; ++i) push(i, 0);                               // SARL's op list
        for (int i : {10, 9, 8, 7, 3, 6, 5, 4, 2, 1}) push(i, 1);
    } else {
        d.net = kNetWorldMlp;
        for (int i = 0; i < 4; ++i) push(i, 0);
        for (int i = 3; i >= 1; --i) push(i, 1);
    }
    d.n_ops = n;
    NetDims d_fwd = d;
    d_fwd.n_ops = d.n_layers;
    int rc = use_device(device);
    if (rc) return rc;
    // AttentionWorld: human_num is the most humans a sample may have; MlpWorld is built for exactly human_num
    if (trainer_smem(d, human_num, 1) > kTrainerMaxSmem) {
        cn_set_error("world trainer: %d humans per sample do not fit the shared-memory plan", human_num);
        return CN_EUNSUPPORTED;
    }
    cn_world_trainer *t = new cn_world_trainer();
    memset(t, 0, sizeof(*t));
    t->device = device; t->kind = kind; t->H = human_num; t->max_batch = max_batch; t->drop = drop_rate;
    t->d = d; t->d_fwd = d_fwd;
    const int spc = trainer_spc(d);
    t->nparts_cap = (max_batch + spc - 1) / spc;
    const int np = d.n_params;
    if (cudaMalloc((void **)&t->Wt, sizeof(float) * d.t_size) != cudaSuccess ||
        cudaMalloc((void **)&t->Wa, sizeof(float) * d.a_size) != cudaSuccess ||
        cudaMalloc((void **)&t->m, sizeof(float) * np) != cudaSuccess ||
        cudaMalloc((void **)&t->v, sizeof(float) * np) != cudaSuccess ||
        cudaMalloc((void **)&t->gpart, sizeof(float) * (size_t)np * t->nparts_cap) != cudaSuccess ||
        cudaMalloc((void **)&t->loss_part, sizeof(float) * t->nparts_cap) != cudaSuccess ||
        cudaMalloc((void **)&t->tmap, sizeof(int32_t) * np) != cudaSuccess ||
        cudaMalloc((void **)&t->amap, sizeof(int32_t) * np) != cudaSuccess) {
        cn_set_error("cudaMalloc failed in cn_world_trainer_create");
        cn_world_trainer_destroy(t);
        return CN_ENOMEM;
    }
    std::vector<int32_t> tmap(np), amap(np);
    trainer_maps(d, tmap.data(), amap.data());
    // (the padding floats of the blocks are read by cp.async, hence the memsets)
    cudaError_t ce = cudaMemset(t->Wt, 0, sizeof(float) * d.t_size);
    if (ce == cudaSuccess) ce = cudaMemset(t->Wa, 0, sizeof(float) * d.a_size);
    if (ce == cudaSuccess) ce = cudaMemset(t->m, 0, sizeof(float) * np);
    if (ce == cudaSuccess) ce = cudaMemset(t->v, 0, sizeof(float) * np);
    if (ce == cudaSuccess) ce = cudaMemcpy(t->tmap, tmap.data(), sizeof(int32_t) * np, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess) ce = cudaMemcpy(t->amap, amap.data(), sizeof(int32_t) * np, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess) ce = trainer_configure(d);
    if (ce != cudaSuccess) {
        cn_set_error("cn_world_trainer_create: %s", cudaGetErrorString(ce));
        cn_world_trainer_destroy(t);
        return CN_ECUDA;
    }
    *out = t;
    return CN_OK;
}

int cn_world_trainer_destroy(cn_world_trainer *t)
{
    if (!t) return CN_OK;
    cudaSetDevice(t->device);
    void *ptrs[] = {t->Wt, t->Wa, t->m, t->v, t->gpart, t->loss_part, t->tmap, t->amap};
    for (void *q : ptrs) if (q) cudaFree(q);
    delete t;
    return CN_OK;
}

int64_t cn_world_trainer_param_count(const cn_world_trainer *t) { return t ? t->d.n_params : 0; }

int cn_world_trainer_sync_weights(cn_world_trainer *t, const float *w_dev, int reset_optimizer, void *stream)
{
    if (!t || !w_dev) { cn_set_error("null argument"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(t->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int n = t->d.n_params;
    const int rc = trainer_refresh(n, w_dev, t->Wt, t->Wa, t->tmap, t->amap, s);
    if (rc) return rc;
    if (reset_optimizer) {
        CN_CUDA_CHECK(cudaMemsetAsync(t->m, 0, sizeof(float) * n, s));
        CN_CUDA_CHECK(cudaMemsetAsync(t->v, 0, sizeof(float) * n, s));
        t->adam_t = 0;
        t->draws = 0;
    }
    t->synced = 1;
    return CN_OK;
}

// The checks of a step or an evaluation on `batch` samples of `human_num` humans
static int world_check(const cn_world_trainer *t, const float *x_dev, const float *y_dev, int32_t human_num)
{
    if (!t || !x_dev || !y_dev) { cn_set_error("null argument"); return CN_EINVAL; }
    if (!t->synced) { cn_set_error("cn_world_trainer_sync_weights has not been called"); return CN_EINVAL; }
    if (t->kind == CN_WORLD_MLP && human_num != t->H) {
        cn_set_error("MlpWorld was built for %d humans, the data has %d", t->H, human_num); return CN_EINVAL;
    }
    if (human_num < 1 || human_num > t->H) {
        cn_set_error("human_num %d outside the trainer's capacity (1..%d)", human_num, t->H); return CN_EINVAL;
    }
    return CN_OK;
}

static AdamArgs adam_args(int64_t step, float lr, float beta1, float beta2, float eps)
{
    AdamArgs a;
    a.b1 = beta1; a.omb1 = (float)(1.0 - (double)beta1);
    a.b2 = beta2; a.omb2 = (float)(1.0 - (double)beta2);
    a.step_size = (float)((double)lr / (1.0 - pow((double)beta1, (double)step)));
    a.bc2_sqrt = (float)sqrt(1.0 - pow((double)beta2, (double)step));
    a.eps = eps;
    return a;
}

int cn_world_trainer_step(cn_world_trainer *t, float *w_dev, const float *x_dev, const float *y_dev, const int64_t *index_dev,
                          int32_t batch, int32_t human_num, float lr, float beta1, float beta2, float eps, uint64_t seed,
                          float *grad_out_dev, float *loss_sum_dev, uint8_t *mask_dev, void *stream)
{
    int rc = world_check(t, x_dev, y_dev, human_num);
    if (rc) return rc;
    if (!w_dev) { cn_set_error("null argument"); return CN_EINVAL; }
    if (batch < 1 || batch > t->max_batch) { cn_set_error("batch %d outside 1..max_batch (%d)", batch, t->max_batch); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(t->device));
    cudaStream_t s = (cudaStream_t)stream;
    const WorldStep ws = {t->drop, seed, t->draws, mask_dev, 0};
    int nparts = 0;
    if ((rc = trainer_launch(t->d, t->Wt, t->Wa, x_dev, y_dev, index_dev, batch, human_num, t->gpart, t->loss_part, &nparts, s, &ws)))
        return rc;
    ++t->draws;
    if (!grad_out_dev) ++t->adam_t;
    const AdamArgs a = adam_args(grad_out_dev ? 1 : t->adam_t, lr, beta1, beta2, eps);
    const int n = t->d.n_params;
    world_adam_reduce_kernel<<<(n + 255) / 256, 256, 0, s>>>(n, nparts, t->gpart, t->loss_part, (float)((int64_t)batch * human_num * 2),
                                                            loss_sum_dev, grad_out_dev, w_dev, t->Wt, t->Wa, t->m, t->v, t->tmap,
                                                            t->amap, a);
    CN_LAUNCH_CHECK();
    return CN_OK;
}

int cn_world_trainer_apply(cn_world_trainer *t, float *w_dev, const float *grad_dev, float grad_scale, float lr, float beta1,
                           float beta2, float eps, void *stream)
{
    if (!t || !w_dev || !grad_dev) { cn_set_error("null argument"); return CN_EINVAL; }
    if (!t->synced) { cn_set_error("cn_world_trainer_sync_weights has not been called"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(t->device));
    ++t->adam_t;
    const int n = t->d.n_params;
    world_adam_apply_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(n, grad_dev, grad_scale, w_dev, t->Wt, t->Wa, t->m, t->v,
                                                                             t->tmap, t->amap,
                                                                             adam_args(t->adam_t, lr, beta1, beta2, eps));
    CN_LAUNCH_CHECK();
    return CN_OK;
}

int cn_world_trainer_eval(cn_world_trainer *t, const float *x_dev, const float *y_dev, const int64_t *index_dev, int32_t n,
                          int32_t human_num, float *loss_sum_dev, void *stream)
{
    int rc = world_check(t, x_dev, y_dev, human_num);
    if (rc) return rc;
    if (n < 1 || !loss_sum_dev) { cn_set_error("n >= 1 and loss_sum_dev required"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(t->device));
    cudaStream_t s = (cudaStream_t)stream;
    const WorldStep ws = {0.0f, 0, 0, nullptr, 1};
    const float div = (float)((int64_t)n * human_num * 2);
    for (int32_t off = 0; off < n; off += t->max_batch) {           // max_batch samples per launch: the loss_part capacity
        const int32_t b = n - off < t->max_batch ? n - off : t->max_batch;
        const size_t rows = index_dev ? 0 : (size_t)off * human_num;     // humans before this chunk's first sample
        int nparts = 0;
        if ((rc = trainer_launch(t->d_fwd, t->Wt, t->Wa, x_dev + rows * 4, y_dev + rows * 2, index_dev ? index_dev + off : nullptr,
                                 b, human_num, nullptr, t->loss_part, &nparts, s, &ws)))
            return rc;
        world_adam_reduce_kernel<<<1, 32, 0, s>>>(0, nparts, nullptr, t->loss_part, div, loss_sum_dev, nullptr, nullptr, nullptr,
                                                  nullptr, nullptr, nullptr, nullptr, nullptr, AdamArgs{});
        CN_LAUNCH_CHECK();
    }
    return CN_OK;
}

}  // extern "C"
