// trainer_nets.cu -- the forward + hand-written backward of CADRL and LSTM-RL for the fused trainer (trainer.cu owns the
// cn_trainer_* entry points, the reduce / SGD kernels and the parameter layout; this file only produces the per-CTA partial
// gradients and squared errors, exactly like trainer_fwd_bwd_kernel does for SARL).
//
//   CADRL      value_network = mlp(13 -> a, b, c, 1) on single-human rows (cadrl.py:22-30,209): kCadrlSPC samples per CTA.
//   LSTM-RL    (lstm_rl.py:9-66) one sample per CTA: [ValueNetwork2: mlp1 on every row, no ReLU after its last layer]
//              -> nn.LSTM over the H rows in the given order (gates i, f, g, o) -> mlp on [state[0, :self_dim] | h_H].
//              Backward = BPTT over the gates, c_t and h_t the forward left in shared memory; W_hh stays staged in shared
//              memory for the whole recurrence (forward: transposed, backward: original layout); the weight gradients are
//              one weight_grad pass over all H rows after the loop: dW_ih = dgates^T X, dW_hh = dgates^T [h_0 .. h_{H-1}]
//              with h_0 = 0, and bias_ih and bias_hh both receive sum_t dgates_t.
//
// Every weight block a step uses is staged into shared memory with cp.async, the next block while the current one computes
// (the ops list of NetDims, built by the host in trainer.cu), as in trainer_fwd_bwd_kernel.
#include "cn_common.cuh"
#include "dense_f32.cuh"
#include "trainer_nets.cuh"

#include <assert.h>
#include <math.h>

namespace {

using namespace dense_f32;      // kThreads, pad4, dense_t, weight_grad, stage_async
// CADRL samples per CTA: one row each, so a CTA of 8 samples runs every layer as ONE pass over its weight block (dense_t
// computes 8 rows per weight load) and the reduce sums 13 partial gradients instead of 100 for the reference batch of 100.
// (Chosen from that reasoning, not from a measured sweep.)
constexpr int kCadrlSPC = 8;

// shared-memory plan (floats); every row stride is a multiple of 4 floats
struct NPlan {
    int ld_x, ld_a[3], ld_m[4], ld_g4, ld_h, ld_j, wide;
    int x, a[3], v, m[4], gt, dg, c, hs, dh, dc, j, d0, d1, total;
};

__host__ __device__ inline NPlan make_nplan(const NetDims &d, int H, int ns)
{
    NPlan p = {};
    const bool lstm = d.net == CN_NET_LSTM_RL;
    const int R = lstm ? H : ns;                     // rows of the input: the sample's humans, or one row per CADRL sample
    int o = 0, wide = 0;
    auto grow = [&](int w) { if (w > wide) wide = w; };
    p.ld_x = pad4(d.in); p.x = o; o += R * p.ld_x; grow(p.ld_x);
    for (int i = 0; i < 3; ++i) {                    // value mlp: one row per sample
        p.ld_a[i] = pad4(d.L[d.mlp0 + i].out); p.a[i] = o; o += ns * p.ld_a[i]; grow(p.ld_a[i]);
    }
    p.v = o; o += pad4(ns);
    if (lstm) {
        if (d.vn2)
            for (int i = 0; i < 4; ++i) { p.ld_m[i] = pad4(d.L[i].out); p.m[i] = o; o += H * p.ld_m[i]; grow(p.ld_m[i]); }
        p.ld_g4 = pad4(4 * d.lstm_h); p.ld_h = pad4(d.lstm_h);
        p.gt = o; o += H * p.ld_g4;                  // gates of every step (pre-activation, then i, f, g, o in place)
        p.dg = o; o += H * p.ld_g4;                  // their pre-activation gradients
        p.c = o; o += H * p.ld_h;                    // c_t
        p.hs = o; o += (H + 1) * p.ld_h;             // h_0 = 0, h_1 .. h_H
        p.dh = o; o += p.ld_h;
        p.dc = o; o += p.ld_h;
        p.ld_j = pad4(d.self_dim + d.lstm_h); p.j = o; o += p.ld_j; grow(p.ld_j);
    }
    p.wide = wide;
    p.d0 = o; o += R * wide;                         // two gradient scratch buffers, each as wide as the widest activation
    p.d1 = o; o += R * wide;
    p.total = o;
    return p;
}

// out-of-line copies keep the step inside the instruction cache (see trainer.cu)
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

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

__global__ void __launch_bounds__(kThreads, 1)
trainer_nets_fwd_bwd_kernel(NetDims d, const float *__restrict__ Wt, const float *__restrict__ Wa, const float *__restrict__ X,
                            const float *__restrict__ target, const int64_t *__restrict__ index, int B, int H, int spc, int nbuf,
                            float *__restrict__ gpart, float *__restrict__ loss_part)
{
    extern __shared__ __align__(16) float sm[];
    const int s0 = blockIdx.x * spc;
    const int ns = min(spc, B - s0);
    const NPlan p = make_nplan(d, H, ns);
    const NPlan pmax = make_nplan(d, H, spc);           // the staging buffers sit behind the largest activation plan
    const bool lstm = d.net == CN_NET_LSTM_RL;
    const int R = lstm ? H : ns, tid = threadIdx.x;
    const int nh = d.lstm_h, g4 = 4 * d.lstm_h;
    float *xs = sm + p.x, *v = sm + p.v, *d0 = sm + p.d0, *d1 = sm + p.d1;
    float *a[3] = {sm + p.a[0], sm + p.a[1], sm + p.a[2]};
    float *wbuf[2] = {sm + pad4(pmax.total), sm + pad4(pmax.total) + (nbuf == 2 ? d.wbuf_floats : 0)};
    float *G = gpart + (size_t)blockIdx.x * d.n_params;
    const TLayer *L = d.L;

    auto fetch = [&](int k, float *dst) {
        const TLayer &l = L[d.op_layer[k]];
        const bool bwd = d.op_bwd[k];
        stage_block(dst, bwd ? Wa + l.a_off : Wt + l.t_off, pad4(l.in * l.out) + (bwd ? 0 : pad4(l.out)));
    };
    int op = 0;
    // start of weighted op `op`: with two buffers the NEXT block's copy is started (its buffer was released by the barrier that
    // ended op - 1) and this op's block, fetched one op ago, is waited for; with one buffer the block is fetched here.
    // (layer, bwd) = the block the caller computes with: it must be the one the host's op list staged for this op.
    auto begin_op = [&](int layer, int bwd) -> const float * {
        assert(op < d.n_ops && d.op_layer[op] == layer && d.op_bwd[op] == bwd);
        if (nbuf == 2) {
            if (op + 1 < d.n_ops) { fetch(op + 1, wbuf[(op + 1) & 1]); cp_async_wait<1>(); }
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
    // Y = act(X W_i^T + b_i) over Rr rows
    auto fwd = [&](int i, const float *Xp, int ldx, int Rr, float *Yp, int ldy, bool relu) {
        const float *wb = begin_op(i, 0);
        dense_staged(Xp, ldx, Rr, L[i].in, wb, wb + pad4(L[i].in * L[i].out), L[i].out, Yp, ldy, relu, false, nullptr, 0);
        end_op();
    };
    // dX[r][k] = sum_o dY[r][o] W_i[o][k], times the ReLU mask of `gate` (the layer's input activation) when given
    auto bwd = [&](int i, const float *dYp, int ldy, int Rr, float *dXp, int ldx, const float *gate, int ldg) {
        const float *wb = begin_op(i, 1);
        dense_staged(dYp, ldy, Rr, L[i].out, wb, nullptr, L[i].in, dXp, ldx, false, false, gate, ldg);
        end_op();
    };
    auto wgrad = [&](int i, const float *dYp, int ldy, const float *Xin, int ldx, int Rr) {
        weight_grad_call(dYp, ldy, Xin, ldx, Rr, L[i].out, L[i].in, G + L[i].w_off, G + L[i].b_off);
    };

    // ---------------- forward ----------------
    // row r = human r % H of item index[s0 + r / H] of the replay tensors (index == NULL: the batch is X / target itself)
    for (int idx = tid; idx < R * p.ld_x; idx += kThreads) {
        const int r = idx / p.ld_x, k = idx - r * p.ld_x;
        const size_t item = index ? (size_t)index[s0 + r / H] : (size_t)(s0 + r / H);
        xs[idx] = k < d.in ? X[(item * H + r % H) * d.in + k] : 0.0f;
    }
    const float *vin = xs;                              // input of the value mlp: the CADRL rows, or LSTM-RL's joint state
    int ld_vin = p.ld_x;
    float *gt = sm + p.gt, *dg = sm + p.dg, *cs = sm + p.c, *hs = sm + p.hs, *dh = sm + p.dh, *dc = sm + p.dc, *j = sm + p.j;
    const float *seq = xs;                              // LSTM input rows
    int ld_seq = p.ld_x;
    if (lstm) {
        for (int k = tid; k < p.ld_h; k += kThreads) hs[k] = 0.0f;             // h_0 (published by the next op's barrier)
        if (d.vn2) {                                                           // mlp1 (lstm_rl.py:37-38), no ReLU at its end
            float *m[4] = {sm + p.m[0], sm + p.m[1], sm + p.m[2], sm + p.m[3]};
            fwd(0, xs, p.ld_x, H, m[0], p.ld_m[0], true);
            fwd(1, m[0], p.ld_m[0], H, m[1], p.ld_m[1], true);
            fwd(2, m[1], p.ld_m[1], H, m[2], p.ld_m[2], true);
            fwd(3, m[2], p.ld_m[2], H, m[3], p.ld_m[3], false);
            seq = m[3]; ld_seq = p.ld_m[3];
        }
        fwd(d.ih, seq, ld_seq, H, gt, p.ld_g4, false);                         // x_t W_ih^T + b_ih for every step at once
        const float *whh = begin_op(d.hh, 0);                                  // W_hh^T | b_hh, kept for the whole loop
        const float *bhh = whh + pad4(nh * g4);
        for (int t = 0; t < H; ++t) {
            float *gtt = gt + (size_t)t * p.ld_g4;
            dense_staged(hs + (size_t)t * p.ld_h, p.ld_h, 1, nh, whh, bhh, g4, gtt, p.ld_g4, false, true, nullptr, 0);
            __syncthreads();
            for (int k = tid; k < nh; k += kThreads) {
                const float gi = sigmoidf_(gtt[k]), gf = sigmoidf_(gtt[nh + k]), gg = tanhf(gtt[2 * nh + k]),
                            go = sigmoidf_(gtt[3 * nh + k]);
                gtt[k] = gi; gtt[nh + k] = gf; gtt[2 * nh + k] = gg; gtt[3 * nh + k] = go;
                const float cp = t > 0 ? cs[(size_t)(t - 1) * p.ld_h + k] : 0.0f;
                const float c = fmaf(gf, cp, gi * gg);
                cs[(size_t)t * p.ld_h + k] = c;
                hs[(size_t)(t + 1) * p.ld_h + k] = go * tanhf(c);
            }
            __syncthreads();
        }
        end_op();
        for (int k = tid; k < p.ld_j; k += kThreads)                           // [state[:, 0, :self_dim] | h_n]
            j[k] = k < d.self_dim ? xs[k] : (k < d.self_dim + nh ? hs[(size_t)H * p.ld_h + k - d.self_dim] : 0.0f);
        vin = j; ld_vin = p.ld_j;
    }
    const int l0 = d.mlp0;
    fwd(l0, vin, ld_vin, ns, a[0], p.ld_a[0], true);       // (begin_op's barrier publishes j)
    fwd(l0 + 1, a[0], p.ld_a[0], ns, a[1], p.ld_a[1], true);
    fwd(l0 + 2, a[1], p.ld_a[1], ns, a[2], p.ld_a[2], true);
    fwd(l0 + 3, a[2], p.ld_a[2], ns, v, 1, false);

    // ---------------- loss and backward ----------------
    // MSELoss(mean): dL/dv_b = 2 (v_b - y_b) / B
    if (tid == 0) {
        float ls = 0.0f;
        for (int s = 0; s < ns; ++s) { const float df = v[s] - target[index ? index[s0 + s] : s0 + s]; ls += df * df; }
        loss_part[blockIdx.x] = ls;
    }
    float *dv = d0;
    if (tid < ns) dv[tid] = 2.0f * (v[tid] - target[index ? index[s0 + tid] : s0 + tid]) / (float)B;
    __syncthreads();
    wgrad(l0 + 3, dv, 1, a[2], p.ld_a[2], ns);
    bwd(l0 + 3, dv, 1, ns, d1, p.ld_a[2], a[2], p.ld_a[2]);
    wgrad(l0 + 2, d1, p.ld_a[2], a[1], p.ld_a[1], ns);
    bwd(l0 + 2, d1, p.ld_a[2], ns, d0, p.ld_a[1], a[1], p.ld_a[1]);
    wgrad(l0 + 1, d0, p.ld_a[1], a[0], p.ld_a[0], ns);
    bwd(l0 + 1, d0, p.ld_a[1], ns, d1, p.ld_a[0], a[0], p.ld_a[0]);
    wgrad(l0, d1, p.ld_a[0], vin, ld_vin, ns);
    if (!lstm) { assert(op == d.n_ops); return; }       // CADRL: no gradient w.r.t. the input

    float *dj = d0;
    bwd(l0, d1, p.ld_a[0], 1, dj, p.ld_j, nullptr, 0);
    // BPTT from dh_H = dj[self_dim:], dc_H = 0.  Thread k owns cell k in both phases of a step.
    for (int k = tid; k < nh; k += kThreads) { dh[k] = dj[d.self_dim + k]; dc[k] = 0.0f; }
    const float *whh = begin_op(d.hh, 1);               // W_hh [4h][h]: dh_{t-1} = dgates_t W_hh
    for (int t = H - 1; t >= 0; --t) {
        const float *gtt = gt + (size_t)t * p.ld_g4;
        float *dgt = dg + (size_t)t * p.ld_g4;
        for (int k = tid; k < nh; k += kThreads) {
            const float gi = gtt[k], gf = gtt[nh + k], gg = gtt[2 * nh + k], go = gtt[3 * nh + k];
            const float tc = tanhf(cs[(size_t)t * p.ld_h + k]);
            const float cp = t > 0 ? cs[(size_t)(t - 1) * p.ld_h + k] : 0.0f;
            const float dhk = dh[k];
            const float dck = dc[k] + dhk * go * (1.0f - tc * tc);
            dgt[k] = dck * gg * (gi * (1.0f - gi));
            dgt[nh + k] = dck * cp * (gf * (1.0f - gf));
            dgt[2 * nh + k] = dck * gi * (1.0f - gg * gg);
            dgt[3 * nh + k] = dhk * tc * (go * (1.0f - go));
            dc[k] = dck * gf;
        }
        __syncthreads();
        if (t > 0) {
            dense_staged(dgt, p.ld_g4, 1, g4, whh, nullptr, nh, dh, p.ld_h, false, false, nullptr, 0);
            __syncthreads();
        }
    }
    end_op();
    wgrad(d.ih, dg, p.ld_g4, seq, ld_seq, H);           // dW_ih, bias_ih
    wgrad(d.hh, dg, p.ld_g4, hs, p.ld_h, H);            // dW_hh over [h_0 .. h_{H-1}], bias_hh
    if (!d.vn2) { assert(op == d.n_ops); return; }
    float *m[4] = {sm + p.m[0], sm + p.m[1], sm + p.m[2], sm + p.m[3]};
    bwd(d.ih, dg, p.ld_g4, H, d0, p.ld_m[3], nullptr, 0);                // dx_t = dgates_t W_ih (mlp1's last layer: no ReLU)
    wgrad(3, d0, p.ld_m[3], m[2], p.ld_m[2], H);
    bwd(3, d0, p.ld_m[3], H, d1, p.ld_m[2], m[2], p.ld_m[2]);
    wgrad(2, d1, p.ld_m[2], m[1], p.ld_m[1], H);
    bwd(2, d1, p.ld_m[2], H, d0, p.ld_m[1], m[1], p.ld_m[1]);
    wgrad(1, d0, p.ld_m[1], m[0], p.ld_m[0], H);
    bwd(1, d0, p.ld_m[1], H, d1, p.ld_m[0], m[0], p.ld_m[0]);
    wgrad(0, d1, p.ld_m[0], xs, p.ld_x, H);
    assert(op == d.n_ops);                              // every staged block was consumed
}

}  // namespace

int trainer_nets_spc(const NetDims &d) { return d.net == CN_NET_CADRL ? kCadrlSPC : 1; }

size_t trainer_nets_smem(const NetDims &d, int H, int nbuf)
{
    return sizeof(float) * ((size_t)pad4(make_nplan(d, H, trainer_nets_spc(d)).total) + (size_t)nbuf * d.wbuf_floats);
}

cudaError_t trainer_nets_configure()
{
    return cudaFuncSetAttribute(trainer_nets_fwd_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
}

int trainer_nets_launch(const NetDims &d, const float *Wt, const float *Wa, const float *X, const float *target,
                        const int64_t *index, int batch, int H, float *gpart, float *loss_part, int *nparts, cudaStream_t s)
{
    const int spc = trainer_nets_spc(d);
    *nparts = (batch + spc - 1) / spc;
    // two staging buffers (the next weight block is copied while the current layer computes) when they fit, else one
    const int nbuf = trainer_nets_smem(d, H, 2) <= 232448 ? 2 : 1;
    trainer_nets_fwd_bwd_kernel<<<*nparts, kThreads, trainer_nets_smem(d, H, nbuf), s>>>(d, Wt, Wa, X, target, index, batch, H,
                                                                                      spc, nbuf, gpart, loss_part);
    CN_LAUNCH_CHECK();
    return CN_OK;
}
