// world_model.cu -- the fork's learned human-motion models on the device (crowd_nav/policy/world_model.py:20-106):
//   AttentionWorld  the SARL block structure on (px, py, vx, vy) rows: mlp1 (4 -> 150 -> 100), mlp2 (100 -> 100 -> 50),
//                   attention ([e_i | mean e] 200 -> 100 -> 100 -> 1), masked softmax, mlp3 on [state_i | weighted feature]
//                   (54 -> 150 -> 100 -> 100 -> 2) = one (vx, vy) per human                       (world_model.py:53-106)
//   MlpWorld        (H * 4 -> 128 -> 64 -> 12 -> H * 2), ReLU between, tanh at the end (Dropout is the identity in eval)
//                                                                                                  (world_model.py:20-50)
// ModelCrowdSim.step asks the model for every human's next velocity instead of solving ORCA (model_crowd_sim.py:397-425).
// cn_world_predict reads the humans' (px, py, vx, vy) from the env's SoA state -- cast to fp32 like torch.Tensor([...]) --
// and writes the prediction where cn_env_orca would have put the ORCA velocities, so cn_env_step / the query_env lookahead
// consume it without a host round trip.  FP32 on CUDA cores (0.5 MMAC per env: < 1 % of a lookahead), arithmetic twin of the
// torch module to ~1e-6.
#include "cn_common.cuh"
#include "dense_f32.cuh"

#include <math.h>
#include <string.h>

#include <vector>

namespace {

using namespace dense_f32;

constexpr int kMaxLayers = 11;
struct WLayer { int in, out, w_off, b_off; };      // offsets into the transposed device block ([in][out], then bias)
struct WDims {
    int kind;                  // 0 = AttentionWorld, 1 = MlpWorld
    int n_layers;
    WLayer L[kMaxLayers];
    int H;                     // MlpWorld: humans the model was built for
};

struct WPlan { int ld[12]; int off[12]; int sc, wt, total; };

// AttentionWorld buffers: 0 x(4) 1 a1 2 e 3 f1 4 f 5 u 6 t1 7 t2 8 j(54) 9 g1 10 g2 11 g3
__host__ __device__ inline WPlan attn_plan(const WDims &d, int R)
{
    WPlan p;
    const int w[12] = {d.L[0].in, d.L[0].out, d.L[1].out, d.L[2].out, d.L[3].out, d.L[4].in, d.L[4].out, d.L[5].out,
                       d.L[7].in, d.L[7].out, d.L[8].out, d.L[9].out};
    int o = 0;
    for (int i = 0; i < 12; ++i) { p.ld[i] = pad4(w[i]); p.off[i] = o; o += R * p.ld[i]; }
    p.sc = o; o += pad4(R);
    p.wt = o; o += pad4(R);
    p.total = o;
    return p;
}

__global__ void __launch_bounds__(kThreads, 1)
attention_world_kernel(WDims d, EnvDims ed, const float *__restrict__ W, const double *__restrict__ st,
                       const uint8_t *__restrict__ frozen, int envs_per_cta, double *__restrict__ human_v)
{
    extern __shared__ __align__(16) float sm[];
    const int H = ed.H, tid = threadIdx.x;
    const int e0 = blockIdx.x * envs_per_cta;
    const int ne = min(envs_per_cta, ed.E - e0);
    const int R = ne * H;
    const WPlan p = attn_plan(d, envs_per_cta * H);
    float *x = sm + p.off[0], *a1 = sm + p.off[1], *e = sm + p.off[2], *f1 = sm + p.off[3], *f = sm + p.off[4], *u = sm + p.off[5],
          *t1 = sm + p.off[6], *t2 = sm + p.off[7], *j = sm + p.off[8], *g1 = sm + p.off[9], *g2 = sm + p.off[10],
          *g3 = sm + p.off[11], *sc = sm + p.sc, *wt = sm + p.wt;
    const WLayer *L = d.L;
    const int E1 = L[1].out, F = L[3].out, IN = L[0].in;
#define WT(i) (W + L[i].w_off)
#define BS(i) (W + L[i].b_off)
    // state rows: (px, py, vx, vy) of human h of env e0 + r / H, fp32 like torch.Tensor (model_crowd_sim.py:399-401)
    for (int idx = tid; idx < R * p.ld[0]; idx += kThreads) {
        const int r = idx / p.ld[0], k = idx - r * p.ld[0];
        const int env = e0 + r / H, h = r % H;
        const int field = k == 0 ? F_PX : (k == 1 ? F_PY : (k == 2 ? F_VX : F_VY));
        x[idx] = k < IN ? (float)st[st_idx(ed, field, h + 1, env)] : 0.0f;
    }
    __syncthreads();
    dense(x, p.ld[0], R, L[0].in, WT(0), BS(0), L[0].out, a1, p.ld[1], true, false);
    __syncthreads();
    dense(a1, p.ld[1], R, L[1].in, WT(1), BS(1), L[1].out, e, p.ld[2], true, false);
    __syncthreads();
    dense(e, p.ld[2], R, L[2].in, WT(2), BS(2), L[2].out, f1, p.ld[3], true, false);
    for (int idx = tid; idx < ne * E1; idx += kThreads) {                      // u = [e_i | mean over the env's humans]
        const int s = idx / E1, k = idx - s * E1;
        float m = 0.0f;
        for (int h = 0; h < H; ++h) m += e[(size_t)(s * H + h) * p.ld[2] + k];
        m /= (float)H;
        for (int h = 0; h < H; ++h) {
            u[(size_t)(s * H + h) * p.ld[5] + k] = e[(size_t)(s * H + h) * p.ld[2] + k];
            u[(size_t)(s * H + h) * p.ld[5] + E1 + k] = m;
        }
    }
    __syncthreads();
    dense(f1, p.ld[3], R, L[3].in, WT(3), BS(3), L[3].out, f, p.ld[4], false, false);
    dense(u, p.ld[5], R, L[4].in, WT(4), BS(4), L[4].out, t1, p.ld[6], true, false);
    __syncthreads();
    dense(t1, p.ld[6], R, L[5].in, WT(5), BS(5), L[5].out, t2, p.ld[7], true, false);
    __syncthreads();
    dense(t2, p.ld[7], R, L[6].in, WT(6), BS(6), 1, sc, 1, false, false);
    __syncthreads();
    if (tid < ne) {                                                            // masked softmax (world_model.py:85-86)
        float z = 0.0f;
        for (int h = 0; h < H; ++h) {
            const float s = sc[tid * H + h];
            const float ex = expf(s) * (s != 0.0f ? 1.0f : 0.0f);
            wt[tid * H + h] = ex; z += ex;
        }
        for (int h = 0; h < H; ++h) wt[tid * H + h] /= z;
    }
    __syncthreads();
    for (int idx = tid; idx < R * p.ld[8]; idx += kThreads) {                  // joint_i = [state_i | weighted feature of the env]
        const int r = idx / p.ld[8], k = idx - r * p.ld[8];
        const int s = r / H;
        float val = 0.0f;
        if (k < IN) val = x[(size_t)r * p.ld[0] + k];
        else if (k < IN + F) {
            const int kk = k - IN;
            for (int h = 0; h < H; ++h) val = fmaf(wt[s * H + h], f[(size_t)(s * H + h) * p.ld[4] + kk], val);
        }
        j[idx] = val;
    }
    __syncthreads();
    dense(j, p.ld[8], R, L[7].in, WT(7), BS(7), L[7].out, g1, p.ld[9], true, false);
    __syncthreads();
    dense(g1, p.ld[9], R, L[8].in, WT(8), BS(8), L[8].out, g2, p.ld[10], true, false);
    __syncthreads();
    dense(g2, p.ld[10], R, L[9].in, WT(9), BS(9), L[9].out, g3, p.ld[11], true, false);
    __syncthreads();
    float *out = t1;                                                           // [R][2] (t1 is dead)
    dense(g3, p.ld[11], R, L[10].in, WT(10), BS(10), 2, out, 2, false, false);
    __syncthreads();
    for (int idx = tid; idx < R * 2; idx += kThreads) {
        const int r = idx >> 1, c = idx & 1;
        const int env = e0 + r / H, h = r % H;
        if (!frozen[env]) human_v[(size_t)(c * H + h) * ed.E + env] = (double)out[idx];
    }
#undef WT
#undef BS
}

// MlpWorld: one env = one row of H * 4 inputs; a CTA serves envs_per_cta envs
__global__ void __launch_bounds__(kThreads, 1)
mlp_world_kernel(WDims d, EnvDims ed, const float *__restrict__ W, const double *__restrict__ st,
                 const uint8_t *__restrict__ frozen, int envs_per_cta, double *__restrict__ human_v)
{
    extern __shared__ __align__(16) float sm[];
    const int H = ed.H, tid = threadIdx.x;
    const int e0 = blockIdx.x * envs_per_cta;
    const int R = min(envs_per_cta, ed.E - e0);
    const WLayer *L = d.L;
    int ld[5], off[5];
    const int w[5] = {L[0].in, L[0].out, L[1].out, L[2].out, L[3].out};
    int o = 0;
    for (int i = 0; i < 5; ++i) { ld[i] = pad4(w[i]); off[i] = o; o += envs_per_cta * ld[i]; }
    float *x = sm + off[0];
    for (int idx = tid; idx < R * ld[0]; idx += kThreads) {
        const int r = idx / ld[0], k = idx - r * ld[0];
        const int h = k >> 2, c = k & 3;
        const int field = c == 0 ? F_PX : (c == 1 ? F_PY : (c == 2 ? F_VX : F_VY));
        x[idx] = k < L[0].in ? (float)st[st_idx(ed, field, h + 1, e0 + r)] : 0.0f;
    }
    __syncthreads();
    for (int i = 0; i < 4; ++i) {
        dense(sm + off[i], ld[i], R, L[i].in, W + L[i].w_off, W + L[i].b_off, L[i].out, sm + off[i + 1], ld[i + 1], i < 3, false);
        __syncthreads();
    }
    const float *out = sm + off[4];
    for (int idx = tid; idx < R * 2 * H; idx += kThreads) {
        const int r = idx / (2 * H), k = idx - r * 2 * H;
        const int h = k >> 1, c = k & 1;
        if (!frozen[e0 + r]) human_v[(size_t)(c * H + h) * ed.E + e0 + r] = (double)tanhf(out[(size_t)r * ld[4] + k]);
    }
}

// cn_world_load_weights_device: the flat state-dict block (weight [out][in], bias per layer) -> W ([in][out], bias)
__global__ void world_load_kernel(WDims d, int n, const float *__restrict__ flat, float *__restrict__ W)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int base = 0;
    for (int l = 0; l < d.n_layers; ++l) {
        const WLayer &L = d.L[l];
        const int nw = L.in * L.out;
        if (i < base + nw) {
            const int o = (i - base) / L.in, k = (i - base) - o * L.in;
            W[L.w_off + k * L.out + o] = flat[i];
            return;
        }
        if (i < base + nw + L.out) { W[L.b_off + i - base - nw] = flat[i]; return; }
        base += nw + L.out;
    }
}

}  // namespace

int world_layer_dims(int kind, int human_num, int *ins, int *outs)
{
    if (kind == CN_WORLD_ATTENTION) {          // world_model.py:56-69
        const int in_[11] = {4, 150, 100, 100, 200, 100, 100, 54, 150, 100, 100};
        const int out_[11] = {150, 100, 100, 50, 100, 100, 1, 150, 100, 100, 2};
        for (int i = 0; i < 11; ++i) { ins[i] = in_[i]; outs[i] = out_[i]; }
        return 11;
    }
    const int in_[4] = {human_num * 4, 128, 64, 12};   // world_model.py:25-37
    const int out_[4] = {128, 64, 12, human_num * 2};
    for (int i = 0; i < 4; ++i) { ins[i] = in_[i]; outs[i] = out_[i]; }
    return 4;
}

struct cn_world {
    int device;
    WDims d;
    int64_t n_params;
    float *W;          // transposed blocks + biases
    int loaded;
};

extern "C" {

int cn_world_create(int32_t kind, int32_t human_num, int device, cn_world **out)
{
    if (!out) { cn_set_error("null argument"); return CN_EINVAL; }
    if (kind != CN_WORLD_ATTENTION && kind != CN_WORLD_MLP) { cn_set_error("unknown world model kind %d", kind); return CN_EINVAL; }
    if (kind == CN_WORLD_MLP && (human_num < 1 || human_num > CN_MAX_HUMANS)) { cn_set_error("MlpWorld needs its human count"); return CN_EINVAL; }
    const int rc = use_device(device);
    if (rc) return rc;
    cn_world *w = new cn_world();
    memset(w, 0, sizeof(*w));
    w->device = device;
    WDims &d = w->d;
    d.kind = kind; d.H = human_num;
    int ins[kMaxLayers], outs[kMaxLayers];
    d.n_layers = world_layer_dims(kind, human_num, ins, outs);
    for (int i = 0; i < d.n_layers; ++i) { d.L[i].in = ins[i]; d.L[i].out = outs[i]; }
    int off = 0;
    for (int i = 0; i < d.n_layers; ++i) {
        d.L[i].w_off = off; off += d.L[i].in * d.L[i].out;
        d.L[i].b_off = off; off += d.L[i].out;
    }
    w->n_params = off;
    if (cudaMalloc((void **)&w->W, sizeof(float) * off) != cudaSuccess) { delete w; cn_set_error("cudaMalloc failed in cn_world_create"); return CN_ENOMEM; }
    cudaError_t ce = cudaFuncSetAttribute(attention_world_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    if (ce == cudaSuccess) ce = cudaFuncSetAttribute(mlp_world_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    if (ce != cudaSuccess) {
        cn_set_error("cn_world_create: %s", cudaGetErrorString(ce));
        cn_world_destroy(w);
        return CN_ECUDA;
    }
    *out = w;
    return CN_OK;
}

int cn_world_destroy(cn_world *w)
{
    if (!w) return CN_OK;
    cudaSetDevice(w->device);
    if (w->W) cudaFree(w->W);
    delete w;
    return CN_OK;
}

int64_t cn_world_param_count(const cn_world *w) { return w ? w->n_params : 0; }

int cn_world_load_weights(cn_world *w, const float *flat_host, int64_t n, void *stream)
{
    if (!w || !flat_host) { cn_set_error("null argument"); return CN_EINVAL; }
    if (n != w->n_params) { cn_set_error("expected %lld parameters, got %lld", (long long)w->n_params, (long long)n); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(w->device));
    cudaStream_t s = (cudaStream_t)stream;
    std::vector<float> t((size_t)n);
    const float *src = flat_host;
    for (int i = 0; i < w->d.n_layers; ++i) {                 // state-dict order: weight [out][in], bias
        const WLayer &L = w->d.L[i];
        for (int o = 0; o < L.out; ++o)
            for (int k = 0; k < L.in; ++k) t[(size_t)L.w_off + (size_t)k * L.out + o] = src[(size_t)o * L.in + k];
        src += (size_t)L.in * L.out;
        for (int o = 0; o < L.out; ++o) t[(size_t)L.b_off + o] = src[o];
        src += L.out;
    }
    CN_CUDA_CHECK(cudaMemcpyAsync(w->W, t.data(), sizeof(float) * n, cudaMemcpyHostToDevice, s));
    CN_CUDA_CHECK(cudaStreamSynchronize(s));
    w->loaded = 1;
    return CN_OK;
}

int cn_world_load_weights_device(cn_world *w, const float *flat_dev, int64_t n, void *stream)
{
    if (!w || !flat_dev) { cn_set_error("null argument"); return CN_EINVAL; }
    if (n != w->n_params) { cn_set_error("expected %lld parameters, got %lld", (long long)w->n_params, (long long)n); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(w->device));
    world_load_kernel<<<(int)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(w->d, (int)n, flat_dev, w->W);
    CN_LAUNCH_CHECK();
    w->loaded = 1;
    return CN_OK;
}

int cn_world_predict(cn_world *w, cn_env *env, void *stream)
{
    if (!w || !env) { cn_set_error("null handle"); return CN_EINVAL; }
    if (!w->loaded) { cn_set_error("cn_world_load_weights has not been called"); return CN_EINVAL; }
    if (w->device != env->device) { cn_set_error("world model and env live on different devices"); return CN_EINVAL; }
    const EnvDims ed = env->p.d;
    if (w->d.kind == CN_WORLD_MLP && w->d.H != ed.H) { cn_set_error("MlpWorld was built for %d humans, the env has %d", w->d.H, ed.H); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(w->device));
    cudaStream_t s = (cudaStream_t)stream;
    if (w->d.kind == CN_WORLD_ATTENTION) {
        if (ed.H > 32) { cn_set_error("AttentionWorld kernel supports human_num <= 32"); return CN_EUNSUPPORTED; }
        const int epc = 32 / ed.H > 0 ? 32 / ed.H : 1;
        const WPlan pl = attn_plan(w->d, epc * ed.H);
        attention_world_kernel<<<(ed.E + epc - 1) / epc, kThreads, sizeof(float) * (size_t)pl.total, s>>>(
            w->d, ed, w->W, env->state, env->frozen, epc, env->human_v);
    } else {
        const int epc = 16;
        size_t fl = 0;
        for (int i = 0; i < 4; ++i) fl += (size_t)epc * pad4(w->d.L[i].in);
        fl += (size_t)epc * pad4(w->d.L[3].out);
        mlp_world_kernel<<<(ed.E + epc - 1) / epc, kThreads, sizeof(float) * fl, s>>>(w->d, ed, w->W, env->state, env->frozen, epc,
                                                                                   env->human_v);
    }
    CN_LAUNCH_CHECK();
    env->orca_valid = 1;        // the prediction takes the place of the cached ORCA result for step / onestep_lookahead
    return CN_OK;
}

}  // extern "C"
