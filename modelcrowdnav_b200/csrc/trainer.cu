// trainer.cu -- one optimisation step of a value network on the device (FP32):
//   MSE( ValueNetwork(states), targets ) -> backward -> [gradient all-reduce by the caller] -> SGD with momentum.
// Replaces the ~150 kernel launches (+ one host sync) of the torch autograd step the reference runs per batch
// (crowd_nav/utils/trainer.py:61-82: zero_grad, model(inputs), MSELoss, backward, SGD(momentum 0.9).step, loss.item())
// with TWO kernels:
//   trainer_fwd_bwd_kernel   SARL / OM-SARL (CN_NET_SARL): one CTA per kSPC samples of the batch: the whole forward
//                            (sarl.py:28-65) and backward of those samples with every activation in shared memory.  The 21
//                            weight blocks a step walks through (11 forward layers, 10 backward-data products) are STAGED:
//                            while layer i computes from one shared-memory buffer, cp.async brings layer i + 1's block
//                            (<= 80 kB, L2-resident) into the other -- streamed straight from L2 the dependent loads of a
//                            256-thread CTA were all latency (226 us per step in the ncu launch list,
//                            profiles/r02l_train_launches_summary.txt); per-CTA partial weight gradients -> gpart[cta][n_params]
//   trainer_nets_fwd_bwd_kernel   the same for CADRL and LSTM-RL (ValueNetwork1 / 2, with or without maps): trainer_nets.cu
//   trainer_reduce_kernel    fixed-order sum of the partials (deterministic) -> gradient; with grad_out == NULL it also
//                            applies SGD momentum in place and refreshes the transposed weight copy the forward reads
//   trainer_apply_kernel     the SGD half alone, for the data-parallel form (gradient -> NCCL all-reduce -> apply)
// SARL is FP32 FMA bound: ~3 x 62 k MAC per (sample, human) row; 100 x 5 rows = 0.1 GFLOP per step.
//
// Parameter layout = the torch state-dict order of the value network, the same flat block cn_policy_load_weights takes,
// derived from the same layer list (cn_layers), so the torch model's parameters can be VIEWS of the block this trainer
// updates.  SARL: mlp1.0, mlp1.2, mlp2.0, mlp2.2, attention.0, .2, .4, mlp3.0, .2, .4, .6 (weight [out][in] then bias);
// with occupancy maps mlp1.0 reads 13 + cell_num^2 * om_channel_size columns.  Without the global state ([sarl]
// with_global_state = false, sarl.py:40-47) attention.0 reads e_i itself: no [e | mean] input is built and its gradient has
// no mean term.  CADRL: value_network.{0,2,4,6}.  LSTM-RL: [mlp1.*] mlp.* lstm.weight_ih_l0, weight_hh_l0, bias_ih_l0,
// bias_hh_l0.
#include "cn_common.cuh"
#include "dense_f32.cuh"
#include "trainer_nets.cuh"

#include <math.h>
#include <string.h>

#include <vector>

namespace {

using namespace dense_f32;      // kThreads, pad4, dense_t, weight_grad
constexpr int kSPC = 1;           // samples per CTA: 100 CTAs for the reference batch of 100; H <= 8 rows = one weight pass per layer
constexpr int kMaxH = 16;         // humans per sample supported by the shared-memory plan
constexpr int kLayers = 11;

struct TDims {
    TLayer L[kLayers];
    int n_params, t_size, a_size;
    int in, self_dim;
    int no_gs;                 // without the global state: attention.0's input is e (L[4].in = E1), not [e | mean]
    int wbuf_floats;           // size of one staging buffer = the largest block
};

// shared-memory plan (floats); every row stride is a multiple of 4 floats
struct Plan {
    int R, ns;
    int ld_x, ld_a1, ld_e, ld_f1, ld_f, ld_u, ld_t, ld_j, ld_g1, ld_g;
    int x, a1, e, f1, f, u, t1, t2, sc, wt, c, j, g1, g2, g3, v, d0, d1, total;
};

__host__ __device__ inline Plan make_plan(const TDims &d, int H, int ns)
{
    Plan p;
    p.ns = ns; p.R = ns * H;
    const int R = p.R;
    p.ld_x = pad4(d.in); p.ld_a1 = pad4(d.L[0].out); p.ld_e = pad4(d.L[1].out); p.ld_f1 = pad4(d.L[2].out);
    p.ld_f = pad4(d.L[3].out); p.ld_u = pad4(d.L[4].in);
    int wt_ = d.L[4].out > d.L[5].out ? d.L[4].out : d.L[5].out;          // t1 / t2 rows also host de (mlp1's output gradient)
    if (d.L[1].out > wt_) wt_ = d.L[1].out;
    p.ld_t = pad4(wt_);
    p.ld_j = pad4(d.L[7].in); p.ld_g1 = pad4(d.L[7].out); p.ld_g = pad4(d.L[8].out > d.L[9].out ? d.L[8].out : d.L[9].out);
    int o = 0;
    p.x = o; o += R * p.ld_x;
    p.a1 = o; o += R * p.ld_a1;
    p.e = o; o += R * p.ld_e;
    p.f1 = o; o += R * p.ld_f1;
    p.f = o; o += R * p.ld_f;
    p.u = o; o += R * p.ld_u;             // attention input [e_i | mean] (unused without the global state)
    p.t1 = o; o += R * p.ld_t;
    p.t2 = o; o += R * p.ld_t;
    p.sc = o; o += pad4(R);
    p.wt = o; o += pad4(R);
    p.c = o; o += ns * p.ld_f;
    p.j = o; o += ns * p.ld_j;
    p.g1 = o; o += ns * p.ld_g1;
    p.g2 = o; o += ns * p.ld_g;
    p.g3 = o; o += ns * p.ld_g;
    p.v = o; o += 4;
    // two gradient scratch buffers, each as wide as the widest activation row
    int wide = p.ld_u;
    if (p.ld_a1 > wide) wide = p.ld_a1;
    if (p.ld_g1 > wide) wide = p.ld_g1;
    p.d0 = o; o += R * wide;
    p.d1 = o; o += R * wide;
    p.total = o;
    return p;
}

// The step walks 21 weighted ops and 11 weight-gradient passes once, front to back: inlined, that is 32 k SASS instructions
// (0.5 MB) that every CTA fetches exactly once, and the instruction fetch becomes the largest stall (ncu: stall_no_inst 31 %).
// One out-of-line copy of each routine keeps the whole kernel inside the instruction cache.
__device__ __noinline__ void dense_staged(const float *X, int ldx, int R, int K, const float *Wt, const float *b, int O, float *Y,
                                          int ldy, bool relu, bool accumulate, const float *gate, int ldg)
{
    dense_t<true>(X, ldx, R, K, Wt, b, O, Y, ldy, relu, accumulate, gate, ldg);
}
__device__ __noinline__ void weight_grad_call(const float *dY, int ldy, const float *Xin, int ldx, int R, int O, int K, float *gW,
                                              float *gb)
{
    weight_grad(dY, ldy, Xin, ldx, R, O, K, gW, gb);
}
__device__ __noinline__ void stage_block(float *dst, const float *src, int n) { stage_async(dst, src, n); }

__global__ void __launch_bounds__(kThreads, 1)
trainer_fwd_bwd_kernel(TDims d, const float *__restrict__ Wt, const float *__restrict__ Wa, const float *__restrict__ X,
                       const float *__restrict__ target, const int64_t *__restrict__ index, int B, int H, int nbuf,
                       float *__restrict__ gpart, float *__restrict__ loss_part)
{
    extern __shared__ __align__(16) float sm[];
    const int s0 = blockIdx.x * kSPC;
    const int ns = min(kSPC, B - s0);
    const Plan p = make_plan(d, H, ns);
    const Plan pmax = make_plan(d, H, kSPC);            // the staging buffers sit behind the largest activation plan
    const int R = p.R, tid = threadIdx.x;
    float *xs = sm + p.x, *a1 = sm + p.a1, *e = sm + p.e, *f1 = sm + p.f1, *f = sm + p.f, *u = sm + p.u, *t1 = sm + p.t1,
          *t2 = sm + p.t2, *sc = sm + p.sc, *wt = sm + p.wt, *c = sm + p.c, *j = sm + p.j, *g1 = sm + p.g1, *g2 = sm + p.g2,
          *g3 = sm + p.g3, *v = sm + p.v, *d0 = sm + p.d0, *d1 = sm + p.d1;
    float *wbuf[2] = {sm + pad4(pmax.total), sm + pad4(pmax.total) + (nbuf == 2 ? d.wbuf_floats : 0)};
    float *G = gpart + (size_t)blockIdx.x * d.n_params;
    const TLayer *L = d.L;
    const int E1 = L[1].out, F = L[3].out;

    // ---- the 21 weight blocks in the order the step uses them: forward layers 0..10 (transposed copy, bias behind the
    //      weights), then the backward-data products (original [out][in] layout) ----
    constexpr int kOps = 21;
    const int bwd_layer[10] = {10, 9, 8, 7, 3, 6, 5, 4, 2, 1};
    auto op_src = [&](int k) -> const float * { return k < kLayers ? Wt + L[k].t_off : Wa + L[bwd_layer[k - kLayers]].a_off; };
    auto op_floats = [&](int k) -> int {
        const TLayer &l = k < kLayers ? L[k] : L[bwd_layer[k - kLayers]];
        return pad4(l.in * l.out) + (k < kLayers ? pad4(l.out) : 0);
    };
    auto fetch = [&](int k, float *dst) {
        const float *src = op_src(k);
        const int n = op_floats(k);
        stage_block(dst, src, n);
    };
    int op = 0;
    // start of weighted op `op`: with two buffers the NEXT block's copy is started (its buffer was released by the barrier that
    // ended op - 1) and this op's block, fetched one op ago, is waited for; with one buffer the block is fetched here
    auto begin_op = [&]() -> const float * {
        if (nbuf == 2) {
            if (op + 1 < kOps) { fetch(op + 1, wbuf[(op + 1) & 1]); cp_async_wait<1>(); }
            else cp_async_wait<0>();
        } else {
            fetch(op, wbuf[0]);
            cp_async_wait<0>();
        }
        __syncthreads();
        return wbuf[nbuf == 2 ? (op & 1) : 0];
    };
    auto end_op = [&]() { __syncthreads(); ++op; };
    if (nbuf == 2) fetch(0, wbuf[0]);
#define FWD(i, Xp, ldx_, Rr, Yp, ldy_, relu_)                                                                       \
    do {                                                                                                            \
        const float *wb = begin_op();                                                                               \
        dense_staged(Xp, ldx_, Rr, L[i].in, wb, wb + pad4(L[i].in * L[i].out), L[i].out, Yp, ldy_, relu_, false, nullptr, 0);  \
    } while (0)
    // dX[r][k] = sum_o dY[r][o] W[o][k]: the same routine with X = dY, "K" = out, "O" = in, no bias
#define BWD(i, dYp, ldy_, Rr, dXp, ldx_, acc_, gate_, ldg_)                                                                      \
    do {                                                                                                            \
        const float *wb = begin_op();                                                                               \
        dense_staged(dYp, ldy_, Rr, L[i].out, wb, nullptr, L[i].in, dXp, ldx_, false, acc_, gate_, ldg_);                       \
    } while (0)

    // ---------------- forward (sarl.py:28-65) ----------------
    // sample s of the batch = item index[s0 + s] of the replay tensors (index == NULL: the batch is X / target itself)
    for (int idx = tid; idx < R * p.ld_x; idx += kThreads) {
        const int r = idx / p.ld_x, k = idx - r * p.ld_x;
        const size_t item = index ? (size_t)index[s0 + r / H] : (size_t)(s0 + r / H);
        xs[idx] = k < d.in ? X[(item * H + r % H) * d.in + k] : 0.0f;
    }
    FWD(0, xs, p.ld_x, R, a1, p.ld_a1, true); end_op();                        // mlp1.0 + ReLU
    FWD(1, a1, p.ld_a1, R, e, p.ld_e, true); end_op();                         // mlp1.2 + ReLU (last_relu)
    FWD(2, e, p.ld_e, R, f1, p.ld_f1, true);                                   // mlp2.0 + ReLU
    // attention input u = [e_i | mean over the sample's humans]; without the global state attention.0 reads e itself
    const float *att_in = d.no_gs ? e : u;
    const int ld_att = d.no_gs ? p.ld_e : p.ld_u;
    if (!d.no_gs)
        for (int idx = tid; idx < ns * E1; idx += kThreads) {
            const int s = idx / E1, k = idx - s * E1;
            float m = 0.0f;
            for (int h = 0; h < H; ++h) m += e[(size_t)(s * H + h) * p.ld_e + k];
            m /= (float)H;
            for (int h = 0; h < H; ++h) {
                u[(size_t)(s * H + h) * p.ld_u + k] = e[(size_t)(s * H + h) * p.ld_e + k];
                u[(size_t)(s * H + h) * p.ld_u + E1 + k] = m;
            }
        }
    end_op();
    FWD(3, f1, p.ld_f1, R, f, p.ld_f, false); end_op();                        // mlp2.2
    FWD(4, att_in, ld_att, R, t1, p.ld_t, true); end_op();                     // attention.0 + ReLU
    FWD(5, t1, p.ld_t, R, t2, p.ld_t, true); end_op();                         // attention.2 + ReLU
    FWD(6, t2, p.ld_t, R, sc, 1, false); end_op();                             // attention.4 -> score
    if (tid < ns) {                                                            // masked softmax (sarl.py:52-53)
        float z = 0.0f;
        for (int h = 0; h < H; ++h) {
            const float s = sc[tid * H + h];
            const float ex = expf(s) * (s != 0.0f ? 1.0f : 0.0f);
            wt[tid * H + h] = ex; z += ex;
        }
        for (int h = 0; h < H; ++h) wt[tid * H + h] /= z;
    }
    __syncthreads();
    for (int idx = tid; idx < ns * p.ld_j; idx += kThreads) {                  // joint = [self | weighted feature]
        const int s = idx / p.ld_j, k = idx - s * p.ld_j;
        float val = 0.0f;
        if (k < d.self_dim) val = xs[(size_t)(s * H) * p.ld_x + k];
        else if (k < d.self_dim + F) {
            const int kk = k - d.self_dim;
            for (int h = 0; h < H; ++h) val = fmaf(wt[s * H + h], f[(size_t)(s * H + h) * p.ld_f + kk], val);
            c[(size_t)s * p.ld_f + kk] = val;
        }
        j[idx] = val;
    }
    FWD(7, j, p.ld_j, ns, g1, p.ld_g1, true); end_op();                        // mlp3.0   (begin_op's barrier publishes j)
    FWD(8, g1, p.ld_g1, ns, g2, p.ld_g, true); end_op();                       // mlp3.2
    FWD(9, g2, p.ld_g, ns, g3, p.ld_g, true); end_op();                        // mlp3.4
    FWD(10, g3, p.ld_g, ns, v, 1, false); end_op();                            // mlp3.6 -> value

    // ---------------- loss and backward ----------------
    // MSELoss(mean): dL/dv_b = 2 (v_b - y_b) / B
    if (tid == 0) {
        float ls = 0.0f;
        for (int s = 0; s < ns; ++s) { const float df = v[s] - target[index ? index[s0 + s] : s0 + s]; ls += df * df; }
        loss_part[blockIdx.x] = ls;
    }
    float *dv = d0;                                                 // [ns][1]
    if (tid < ns) dv[tid] = 2.0f * (v[tid] - target[index ? index[s0 + tid] : s0 + tid]) / (float)B;
    __syncthreads();
    // mlp3.6
    weight_grad_call(dv, 1, g3, p.ld_g, ns, 1, L[10].in, G + L[10].w_off, G + L[10].b_off);
    float *dg3 = d1;                                                // [ns][ld_g]
    BWD(10, dv, 1, ns, dg3, p.ld_g, false, g3, p.ld_g); end_op();
    // mlp3.4
    weight_grad_call(dg3, p.ld_g, g2, p.ld_g, ns, L[9].out, L[9].in, G + L[9].w_off, G + L[9].b_off);
    float *dg2 = d0;                                                // dv is dead
    BWD(9, dg3, p.ld_g, ns, dg2, p.ld_g, false, g2, p.ld_g); end_op();
    // mlp3.2
    weight_grad_call(dg2, p.ld_g, g1, p.ld_g1, ns, L[8].out, L[8].in, G + L[8].w_off, G + L[8].b_off);
    float *dg1 = d1;                                                // dg3 is dead
    BWD(8, dg2, p.ld_g, ns, dg1, p.ld_g1, false, g1, p.ld_g1); end_op();
    // mlp3.0
    weight_grad_call(dg1, p.ld_g1, j, p.ld_j, ns, L[7].out, L[7].in, G + L[7].w_off, G + L[7].b_off);
    float *dj = d0;                                                 // [ns][ld_j]; the self-state part has no parameters upstream
    BWD(7, dg1, p.ld_g1, ns, dj, p.ld_j, false, nullptr, 0); end_op();
    // weighted feature c = sum_i w_i f_i :  df_i = w_i dc,  dw_i = dc . f_i ;  softmax: ds_i = w_i (dw_i - sum_k w_k dw_k)
    float *df = d1;                                                 // [R][ld_f]  (dg1 is dead)
    float *dsc = sm + p.sc;                                         // scores are dead after the softmax: reuse for ds
    if (tid < R) {
        const int s = tid / H;
        float dw = 0.0f;
        for (int k = 0; k < F; ++k) dw = fmaf(dj[(size_t)s * p.ld_j + d.self_dim + k], f[(size_t)tid * p.ld_f + k], dw);
        dsc[tid] = dw;                                              // dw_i for now
    }
    for (int idx = tid; idx < R * F; idx += kThreads) {
        const int r = idx / F, k = idx - r * F;
        df[(size_t)r * p.ld_f + k] = wt[r] * dj[(size_t)(r / H) * p.ld_j + d.self_dim + k];
    }
    __syncthreads();
    if (tid < ns) {
        float dot = 0.0f;
        for (int h = 0; h < H; ++h) dot = fmaf(wt[tid * H + h], dsc[tid * H + h], dot);
        for (int h = 0; h < H; ++h) dsc[tid * H + h] = wt[tid * H + h] * (dsc[tid * H + h] - dot);
    }
    __syncthreads();
    // mlp2.2 (no ReLU after it) and attention.4
    weight_grad_call(df, p.ld_f, f1, p.ld_f1, R, L[3].out, L[3].in, G + L[3].w_off, G + L[3].b_off);
    weight_grad_call(dsc, 1, t2, p.ld_t, R, 1, L[6].in, G + L[6].w_off, G + L[6].b_off);
    float *df1 = d0;                                                // [R][ld_f1]  (dj is dead)
    BWD(3, df, p.ld_f, R, df1, p.ld_f1, false, f1, p.ld_f1); end_op();
    // mlp2.0's weights now; its data path joins de below
    weight_grad_call(df1, p.ld_f1, e, p.ld_e, R, L[2].out, L[2].in, G + L[2].w_off, G + L[2].b_off);
    float *dt2 = d1;                                                // [R][ld_t]  (df is dead)
    BWD(6, dsc, 1, R, dt2, p.ld_t, false, t2, p.ld_t); end_op();                // dt2 = ds * W_att4[0][:]
    // attention.2
    weight_grad_call(dt2, p.ld_t, t1, p.ld_t, R, L[5].out, L[5].in, G + L[5].w_off, G + L[5].b_off);
    float *dt1 = t2;                                                // t2 is dead once its mask and attention.4's gradient are taken
    BWD(5, dt2, p.ld_t, R, dt1, p.ld_t, false, t1, p.ld_t); end_op();
    // attention.0 on u = [e | mean] (or on e)
    weight_grad_call(dt1, p.ld_t, att_in, ld_att, R, L[4].out, L[4].in, G + L[4].w_off, G + L[4].b_off);
    float *de = t1;                                                 // t1 is dead; rows of ld_t floats
    if (d.no_gs) {
        BWD(4, dt1, p.ld_t, R, de, p.ld_t, false, nullptr, 0); end_op();      // de_i = du_i
    } else {
        float *du = d1;                                             // [R][ld_u]  (dt2 is dead)
        BWD(4, dt1, p.ld_t, R, du, p.ld_u, false, nullptr, 0); end_op();
        // de_i = du_i[:E1] + (1/H) sum_k du_k[E1:]
        for (int idx = tid; idx < ns * E1; idx += kThreads) {
            const int s = idx / E1, k = idx - s * E1;
            float m = 0.0f;
            for (int h = 0; h < H; ++h) m += du[(size_t)(s * H + h) * p.ld_u + E1 + k];
            m /= (float)H;
            for (int h = 0; h < H; ++h) de[(size_t)(s * H + h) * p.ld_t + k] = du[(size_t)(s * H + h) * p.ld_u + k] + m;
        }
    }
    // + mlp2.0's path (df1 W_20)
    BWD(2, df1, p.ld_f1, R, de, p.ld_t, true, e, p.ld_e); end_op();            // += df1 * W_mlp2.0   (begin_op's barrier publishes de)
    // mlp1.2
    weight_grad_call(de, p.ld_t, a1, p.ld_a1, R, L[1].out, L[1].in, G + L[1].w_off, G + L[1].b_off);
    float *da1 = d1;                                                // [R][ld_a1]  (du is dead)
    BWD(1, de, p.ld_t, R, da1, p.ld_a1, false, a1, p.ld_a1); end_op();
    // mlp1.0 (no gradient w.r.t. the input)
    weight_grad_call(da1, p.ld_a1, xs, p.ld_x, R, L[0].out, L[0].in, G + L[0].w_off, G + L[0].b_off);
#undef FWD
#undef BWD
}

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
    int net;                                      // CN_NET_*: SARL runs trainer_fwd_bwd_kernel on d, the others trainer_nets.cu on nd
    TDims d;
    NetDims nd;
    int n_params;
    int max_batch, max_humans;
    float *Wt, *Wa, *mom, *gpart, *loss_part;     // transposed / aligned weight copies, momentum, per-CTA partials
    int32_t *tmap, *amap;                         // flat parameter index -> index in Wt / Wa (-1: not in Wa)
    int nparts_cap;
};

// The weight matrices of the flat block in state-dict order, from the layer list the lookahead loads (cn_layers): a Linear
// is one TLayer, the LSTM block two (weight_ih with bias_ih, weight_hh with bias_hh).  Fills w_off / b_off / t_off / a_off;
// returns the parameter count, *wbuf = the largest staged block.
static int trainer_layers(const cn_sarl_cfg *cfg, std::vector<TLayer> &L, int *t_size, int *a_size, int *wbuf)
{
    SarlWeightsDev w;        // only the destinations of the layer list, never written here
    int off = 0;
    for (const LayerSpec &l : cn_layers(cn_dims_of(cfg, 0), w)) {
        if (!l.dst_hh) {
            L.push_back({l.in, l.out, off, off + l.in * l.out, 0, 0});
        } else {                                          // weight_ih_l0, weight_hh_l0, bias_ih_l0, bias_hh_l0
            const int hid = l.out / 4, whh = off + l.out * l.in, bih = whh + l.out * hid;
            L.push_back({l.in, l.out, off, bih, 0, 0});
            L.push_back({hid, l.out, whh, bih + l.out, 0, 0});
        }
        off += (int)cn_layer_floats(l);
    }
    int toff = 0, aoff = 0;
    *wbuf = 0;
    for (TLayer &l : L) {
        l.t_off = toff; toff += pad4(l.in * l.out) + pad4(l.out);      // [in][out] | bias, 16-byte aligned blocks
        l.a_off = aoff; aoff += pad4(l.in * l.out);                    // [out][in]
        const int blk = pad4(l.in * l.out) + pad4(l.out);
        if (blk > *wbuf) *wbuf = blk;
    }
    *t_size = toff; *a_size = aoff;
    return off;
}

// CADRL / LSTM-RL: the layers and the order in which trainer_nets_fwd_bwd_kernel stages their blocks
static void trainer_net_dims(const cn_sarl_cfg *cfg, const std::vector<TLayer> &L, NetDims &nd)
{
    nd.net = cfg->network;
    nd.n_layers = (int)L.size();
    for (int i = 0; i < nd.n_layers; ++i) nd.L[i] = L[i];
    nd.in = cfg->input_dim; nd.self_dim = cfg->self_state_dim;
    const bool lstm = cfg->network == CN_NET_LSTM_RL;
    nd.vn2 = lstm && cfg->lstm_mlp1_dims[0] > 0;
    nd.lstm_h = lstm ? cfg->lstm_hidden : 0;
    nd.lstm_in = nd.vn2 ? cfg->lstm_mlp1_dims[3] : cfg->input_dim;
    nd.mlp0 = nd.vn2 ? 4 : 0;
    nd.ih = nd.mlp0 + 4; nd.hh = nd.mlp0 + 5;
    int n = 0;
    auto push = [&](int layer, int bwd) { nd.op_layer[n] = (int8_t)layer; nd.op_bwd[n] = (int8_t)bwd; ++n; };
    if (lstm) {
        if (nd.vn2) for (int i = 0; i < 4; ++i) push(i, 0);                 // mlp1
        push(nd.ih, 0); push(nd.hh, 0);                                        // x W_ih^T, then W_hh^T for the recurrence
    }
    for (int i = 0; i < 4; ++i) push(nd.mlp0 + i, 0);                          // the value mlp
    for (int i = 3; i >= (lstm ? 0 : 1); --i) push(nd.mlp0 + i, 1);            // its backward-data products (LSTM-RL: down to h_H)
    if (lstm) {
        push(nd.hh, 1);                                                        // BPTT
        if (nd.vn2) { push(nd.ih, 1); for (int i = 3; i >= 1; --i) push(i, 1); }   // dx_t, then mlp1
    }
    nd.n_ops = n;
}

extern "C" {

int cn_trainer_create(const cn_sarl_cfg *cfg, int device, int32_t max_batch, int32_t max_humans, cn_trainer **out)
{
    if (!cfg || !out) { cn_set_error("null argument"); return CN_EINVAL; }
    const int net = cfg->network;
    if (net != CN_NET_SARL && net != CN_NET_CADRL && net != CN_NET_LSTM_RL) { cn_set_error("unknown value network %d", net); return CN_EINVAL; }
    if (cfg->without_global_state && net != CN_NET_SARL) {
        cn_set_error("without_global_state is a [sarl] option; CADRL and LSTM-RL have no global state"); return CN_EINVAL;
    }
    if (cfg->with_om) {
        if (net == CN_NET_CADRL) { cn_set_error("CADRL has no occupancy maps (cadrl.py:60-62)"); return CN_EINVAL; }
        if (cfg->cell_num < 1 || cfg->cell_num > 8 || cfg->om_channel_size < 1 || cfg->om_channel_size > 3) {
            cn_set_error("with_om needs 1 <= cell_num <= 8 and om_channel_size in {1, 2, 3}"); return CN_EINVAL;
        }
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
    std::vector<TLayer> L;
    int t_size = 0, a_size = 0, wbuf = 0;
    const int n_params = trainer_layers(cfg, L, &t_size, &a_size, &wbuf);
    for (const TLayer &l : L)
        if (l.in < 1 || l.out < 1) { cn_set_error("layer widths must be >= 1"); return CN_EINVAL; }
    NetDims nd;
    memset(&nd, 0, sizeof(nd));
    size_t smem = 0;
    int spc = kSPC;
    if (net == CN_NET_SARL) {
        if (cfg->attn_dims[2] != 1 || cfg->mlp3_dims[3] != 1) { cn_set_error("attention and mlp3 must end in 1 unit"); return CN_EINVAL; }
    } else {
        if (cfg->mlp3_dims[3] != 1) { cn_set_error("the value mlp must end in 1 unit"); return CN_EINVAL; }
        trainer_net_dims(cfg, L, nd);
        nd.n_params = n_params; nd.t_size = t_size; nd.a_size = a_size; nd.wbuf_floats = wbuf;
        smem = trainer_nets_smem(nd, max_humans, 1);
        spc = trainer_nets_spc(nd);
    }
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); cn_set_error("no CUDA device available; no CPU fallback"); return CN_ECUDA; }
    if (device < 0 || device >= n) { cn_set_error("device %d out of range", device); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(device));
    cn_trainer *t = new cn_trainer();
    memset(t, 0, sizeof(*t));
    t->device = device; t->net = net; t->max_batch = max_batch; t->max_humans = max_humans;
    t->n_params = n_params;
    t->nd = nd;
    TDims &d = t->d;
    if (net == CN_NET_SARL) {
        for (int i = 0; i < kLayers; ++i) d.L[i] = L[i];
        d.n_params = n_params; d.t_size = t_size; d.a_size = a_size; d.wbuf_floats = wbuf;
        d.in = cfg->input_dim; d.self_dim = cfg->self_state_dim; d.no_gs = cfg->without_global_state ? 1 : 0;
        smem = sizeof(float) * ((size_t)pad4(make_plan(d, max_humans, kSPC).total) + wbuf);
    }
    std::vector<int32_t> tmap(n_params), amap(n_params, -1);
    for (const TLayer &l : L) {
        for (int o = 0; o < l.out; ++o)
            for (int k = 0; k < l.in; ++k) {
                tmap[l.w_off + o * l.in + k] = l.t_off + k * l.out + o;
                amap[l.w_off + o * l.in + k] = l.a_off + o * l.in + k;
            }
        for (int o = 0; o < l.out; ++o) tmap[l.b_off + o] = l.t_off + pad4(l.in * l.out) + o;
    }
    t->nparts_cap = (max_batch + spc - 1) / spc;
    if (smem > 232448) {
        delete t;
        cn_set_error("fused trainer: %d humans per sample%s do not fit the shared-memory plan", max_humans,
                     net == CN_NET_LSTM_RL ? " at this lstm_hidden / layer widths" : "");
        return CN_EUNSUPPORTED;
    }
    if (cudaMalloc((void **)&t->Wt, sizeof(float) * t_size) != cudaSuccess ||
        cudaMalloc((void **)&t->Wa, sizeof(float) * a_size) != cudaSuccess ||
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
    cudaError_t ce = cudaMemset(t->Wt, 0, sizeof(float) * t_size);
    if (ce == cudaSuccess) ce = cudaMemset(t->Wa, 0, sizeof(float) * a_size);
    if (ce == cudaSuccess) ce = cudaMemset(t->mom, 0, sizeof(float) * n_params);
    if (ce == cudaSuccess) ce = cudaMemcpy(t->tmap, tmap.data(), sizeof(int32_t) * n_params, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess) ce = cudaMemcpy(t->amap, amap.data(), sizeof(int32_t) * n_params, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess)
        ce = net == CN_NET_SARL ? cudaFuncSetAttribute(trainer_fwd_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448)
                                : trainer_nets_configure();
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

int64_t cn_trainer_param_count(const cn_trainer *t) { return t ? t->n_params : 0; }

int cn_trainer_sync_weights(cn_trainer *t, const float *w_dev, int zero_momentum, void *stream)
{
    if (!t || !w_dev) { cn_set_error("null argument"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(t->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int n = t->n_params;
    trainer_transpose_kernel<<<(n + 255) / 256, 256, 0, s>>>(n, w_dev, t->Wt, t->Wa, t->tmap, t->amap);
    CN_LAUNCH_CHECK();
    if (zero_momentum) CN_CUDA_CHECK(cudaMemsetAsync(t->mom, 0, sizeof(float) * n, s));
    return CN_OK;
}

static int trainer_step_impl(cn_trainer *t, float *w_dev, const float *states_dev, const float *targets_dev,
                             const int64_t *index_dev, int32_t batch, int32_t human_num, float lr, float momentum,
                             float *grad_out_dev, float *loss_dev, int loss_accumulate, void *stream)
{
    if (!t || !w_dev || !states_dev || !targets_dev) { cn_set_error("null argument"); return CN_EINVAL; }
    if (t->net == CN_NET_CADRL && human_num != 1) {
        cn_set_error("CADRL trains on single-human states (cadrl.py:209): human_num must be 1, got %d", human_num); return CN_EINVAL;
    }
    if (batch < 1 || batch > t->max_batch || human_num < 1 || human_num > t->max_humans) {
        cn_set_error("batch %d / human_num %d outside the trainer's capacity (%d, %d)", batch, human_num, t->max_batch, t->max_humans);
        return CN_EINVAL;
    }
    CN_CUDA_CHECK(cudaSetDevice(t->device));
    cudaStream_t s = (cudaStream_t)stream;
    int nparts = (batch + kSPC - 1) / kSPC;
    if (t->net == CN_NET_SARL) {
        const Plan pl = make_plan(t->d, human_num, kSPC);
        // two staging buffers (the next weight block is copied while the current layer computes) when they fit, else one
        const size_t act = (size_t)pad4(pl.total);
        const int nbuf = sizeof(float) * (act + 2 * (size_t)t->d.wbuf_floats) <= 232448 ? 2 : 1;
        const size_t smem = sizeof(float) * (act + (size_t)nbuf * t->d.wbuf_floats);
        trainer_fwd_bwd_kernel<<<nparts, kThreads, smem, s>>>(t->d, t->Wt, t->Wa, states_dev, targets_dev, index_dev, batch,
                                                             human_num, nbuf, t->gpart, t->loss_part);
        CN_LAUNCH_CHECK();
    } else {
        const int rc = trainer_nets_launch(t->nd, t->Wt, t->Wa, states_dev, targets_dev, index_dev, batch, human_num, t->gpart,
                                           t->loss_part, &nparts, s);
        if (rc != CN_OK) return rc;
    }
    const int n = t->n_params;
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
    const int n = t->n_params;
    trainer_apply_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(n, grad_dev, grad_scale, w_dev, t->Wt, t->Wa, t->mom, t->tmap,
                                                                          t->amap, lr, momentum);
    CN_LAUNCH_CHECK();
    return CN_OK;
}

}  // extern "C"
