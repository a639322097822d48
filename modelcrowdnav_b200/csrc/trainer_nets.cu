// trainer_nets.cu -- the forward + hand-written backward of every value network for the fused trainer.  trainer.cu owns the
// cn_trainer_* entry points, the reduce / SGD kernels and the parameter layout; the kernels here only produce the per-CTA
// partial gradients gpart[cta][n_params] and squared errors, with every activation in shared memory.
//
//   trainer_fwd_bwd_kernel        SARL / OM-SARL (sarl.py:28-65): one CTA per sample, its H rows through mlp1, mlp2,
//                                 attention, the masked softmax and mlp3.  FP32 FMA bound: ~3 x 62 k MAC per (sample,
//                                 human) row; 100 x 5 rows = 0.1 GFLOP per step.  Without the global state ([sarl]
//                                 with_global_state = false, sarl.py:40-47) attention.0 reads e_i itself: no [e | mean] input
//                                 is built and its gradient has no mean term.
//   trainer_nets_fwd_bwd_kernel   CADRL: value_network = mlp(13 -> a, b, c, 1) on single-human rows (cadrl.py:22-30,209),
//                                 kCadrlSPC samples per CTA.
//                                 LSTM-RL (lstm_rl.py:9-66): one sample per CTA: [ValueNetwork2: mlp1 on every row, no ReLU
//                                 after its last layer] -> nn.LSTM over the H rows in the given order (gates i, f, g, o) -> mlp
//                                 on [state[0, :self_dim] | h_H].  Backward = BPTT over the gates, c_t and h_t the forward left
//                                 in shared memory; W_hh stays staged for the whole recurrence (forward: transposed, backward:
//                                 original layout); the weight gradients are one weight_grad pass over all H rows after the
//                                 loop: dW_ih = dgates^T X, dW_hh = dgates^T [h_0 .. h_{H-1}] with h_0 = 0, and bias_ih and
//                                 bias_hh both receive sum_t dgates_t.
//
// Every weight block a step uses is STAGED into shared memory with cp.async, in the order of the op list the host builds
// (NetDims, trainer_net_dims in trainer.cu): while op k computes from one buffer, op k + 1's block (<= 80 kB, L2-resident)
// is copied into the other.  Streamed straight from L2, the dependent loads of a 256-thread CTA were all latency (226 us per
// SARL step in the ncu launch list, profiles/r02l_train_launches_summary.txt).  Device asserts check that each kernel
// consumes exactly that op list.
#include "cn_common.cuh"
#include "dense_f32.cuh"
#include "trainer_nets.cuh"

#include <assert.h>
#include <math.h>

namespace {

using namespace dense_f32;      // kThreads, pad4, dense_t, weight_grad, stage_async
// Samples per CTA.  SARL: 100 CTAs for the reference batch of 100; H <= 8 rows = one weight pass per layer.  CADRL: one row
// per sample, so a CTA of 8 samples runs every layer as ONE pass over its weight block (dense_t computes 8 rows per weight
// load) and the reduce sums 13 partial gradients instead of 100 for the reference batch of 100.  (Chosen from that
// reasoning, not from a measured sweep.)
constexpr int kSarlSPC = 1;
constexpr int kCadrlSPC = 8;

// SARL's shared-memory plan (floats); every row stride is a multiple of 4 floats
struct Plan {
    int R, ns;
    int ld_x, ld_a1, ld_e, ld_f1, ld_f, ld_u, ld_t, ld_j, ld_g1, ld_g;
    int x, a1, e, f1, f, u, t1, t2, sc, wt, c, j, g1, g2, g3, v, d0, d1, total;
};

__host__ __device__ inline Plan make_plan(const NetDims &d, int H, int ns)
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

// CADRL's and LSTM-RL's shared-memory plan (floats); every row stride is a multiple of 4 floats
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

// The step walks ~20 weighted ops and ~10 weight-gradient passes once, front to back: inlined, that is 32 k SASS instructions
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
// (the failure path of the op-order check: inlined at every op, the assert's call setup added ~15 instructions each)
__device__ __noinline__ void op_out_of_order() { assert(!"the kernel computes with a block the op list did not stage"); }

// The weight blocks of one step, staged in the order of d's op list.  An op is bracketed by begin_op / end_op; bwd runs one
// whole op, fwd too unless close = false leaves the op open for work that shares its barriers.
struct Staging {
    const NetDims &d;
    const float *Wt, *Wa;
    float *wbuf0, *wbuf1;      // not an array: indexing one at run time puts the struct, and the NetDims it refers to, on the stack
    int nbuf, op;

    // the staging buffers sit at `base`; with two of them op 0's block is on its way when the constructor returns
    __device__ __forceinline__ Staging(const NetDims &d_, const float *Wt_, const float *Wa_, float *base, int nbuf_)
        : d(d_), Wt(Wt_), Wa(Wa_), wbuf0(base), wbuf1(base + (nbuf_ == 2 ? d_.wbuf_floats : 0)), nbuf(nbuf_), op(0)
    {
        if (nbuf == 2) fetch(0, wbuf0);
    }
    __device__ __forceinline__ void fetch(int k, float *dst) const
    {
        const TLayer &l = d.L[d.op_layer[k]];
        const bool bwd = d.op_bwd[k];
        stage_block(dst, bwd ? Wa + l.a_off : Wt + l.t_off, pad4(l.in * l.out) + (bwd ? 0 : pad4(l.out)));
    }
    // Start of op `op`: with two buffers the NEXT block's copy is started (its buffer was released by the barrier that ended
    // op - 1) and this op's block, fetched one op ago, is waited for; with one buffer the block is fetched here.
    // (layer, bwd) = the block the caller computes with: it must be the one the host's op list staged for this op.
    __device__ __forceinline__ const float *begin_op(int layer, int bwd)
    {
        if (!(op < d.n_ops && d.op_layer[op] == layer && d.op_bwd[op] == bwd)) op_out_of_order();
        const int k = nbuf == 2 ? op + 1 : op;          // the block copied now
        const bool ahead = nbuf == 2 && k < d.n_ops;
        if (k < d.n_ops) fetch(k, ahead && (k & 1) ? wbuf1 : wbuf0);
        if (ahead) cp_async_wait<1>();
        else cp_async_wait<0>();
        __syncthreads();
        return nbuf == 2 && (op & 1) ? wbuf1 : wbuf0;
    }
    __device__ __forceinline__ void end_op() { __syncthreads(); ++op; }
    // Y = act(X W_i^T + b_i) over R rows
    __device__ __forceinline__ void fwd(int i, const float *X, int ldx, int R, float *Y, int ldy, bool relu, bool close = true)
    {
        const TLayer &l = d.L[i];
        const float *wb = begin_op(i, 0);
        dense_staged(X, ldx, R, l.in, wb, wb + pad4(l.in * l.out), l.out, Y, ldy, relu, false, nullptr, 0);
        if (close) end_op();
    }
    // dX[r][k] (+)= sum_o dY[r][o] W_i[o][k], times the ReLU mask of `gate` (the layer's input activation) when given: the
    // same routine with X = dY, "K" = out, "O" = in, no bias
    __device__ __forceinline__ void bwd(int i, const float *dY, int ldy, int R, float *dX, int ldx, const float *gate, int ldg,
                                        bool accumulate = false)
    {
        const float *wb = begin_op(i, 1);
        dense_staged(dY, ldy, R, d.L[i].out, wb, nullptr, d.L[i].in, dX, ldx, false, accumulate, gate, ldg);
        end_op();
    }
    __device__ __forceinline__ void finish() const { assert(op == d.n_ops); }      // every staged block was consumed
};

// dW_i, db_i of R rows into this CTA's partial gradient G
__device__ __forceinline__ void wgrad(const NetDims &d, float *G, int i, const float *dY, int ldy, const float *Xin, int ldx, int R)
{
    weight_grad_call(dY, ldy, Xin, ldx, R, d.L[i].out, d.L[i].in, G + d.L[i].w_off, G + d.L[i].b_off);
}

__global__ void __launch_bounds__(kThreads, 1)
trainer_fwd_bwd_kernel(NetDims d, const float *__restrict__ Wt, const float *__restrict__ Wa, const float *__restrict__ X,
                       const float *__restrict__ target, const int64_t *__restrict__ index, int B, int H, int nbuf,
                       float *__restrict__ gpart, float *__restrict__ loss_part)
{
    extern __shared__ __align__(16) float sm[];
    const int s0 = blockIdx.x * kSarlSPC;
    const int ns = min(kSarlSPC, B - s0);
    const Plan p = make_plan(d, H, ns);
    const Plan pmax = make_plan(d, H, kSarlSPC);        // the staging buffers sit behind the largest activation plan
    const int R = p.R, tid = threadIdx.x;
    float *xs = sm + p.x, *a1 = sm + p.a1, *e = sm + p.e, *f1 = sm + p.f1, *f = sm + p.f, *u = sm + p.u, *t1 = sm + p.t1,
          *t2 = sm + p.t2, *sc = sm + p.sc, *wt = sm + p.wt, *c = sm + p.c, *j = sm + p.j, *g1 = sm + p.g1, *g2 = sm + p.g2,
          *g3 = sm + p.g3, *v = sm + p.v, *d0 = sm + p.d0, *d1 = sm + p.d1;
    float *G = gpart + (size_t)blockIdx.x * d.n_params;
    const int E1 = d.L[1].out, F = d.L[3].out;
    // op list: forward layers 0..10, then the backward-data products of layers 10, 9, 8, 7, 3, 6, 5, 4, 2, 1
    Staging st(d, Wt, Wa, sm + pad4(pmax.total), nbuf);

    // ---------------- forward (sarl.py:28-65) ----------------
    // sample s of the batch = item index[s0 + s] of the replay tensors (index == NULL: the batch is X / target itself)
    for (int idx = tid; idx < R * p.ld_x; idx += kThreads) {
        const int r = idx / p.ld_x, k = idx - r * p.ld_x;
        const size_t item = index ? (size_t)index[s0 + r / H] : (size_t)(s0 + r / H);
        xs[idx] = k < d.in ? X[(item * H + r % H) * d.in + k] : 0.0f;
    }
    st.fwd(0, xs, p.ld_x, R, a1, p.ld_a1, true);                                // mlp1.0 + ReLU
    st.fwd(1, a1, p.ld_a1, R, e, p.ld_e, true);                                 // mlp1.2 + ReLU (last_relu)
    st.fwd(2, e, p.ld_e, R, f1, p.ld_f1, true, false);                          // mlp2.0 + ReLU
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
    st.end_op();
    st.fwd(3, f1, p.ld_f1, R, f, p.ld_f, false);                                // mlp2.2
    st.fwd(4, att_in, ld_att, R, t1, p.ld_t, true);                             // attention.0 + ReLU
    st.fwd(5, t1, p.ld_t, R, t2, p.ld_t, true);                                 // attention.2 + ReLU
    st.fwd(6, t2, p.ld_t, R, sc, 1, false);                                     // attention.4 -> score
    if (tid < ns) {                                                             // masked softmax (sarl.py:52-53)
        float z = 0.0f;
        for (int h = 0; h < H; ++h) {
            const float s = sc[tid * H + h];
            const float ex = expf(s) * (s != 0.0f ? 1.0f : 0.0f);
            wt[tid * H + h] = ex; z += ex;
        }
        for (int h = 0; h < H; ++h) wt[tid * H + h] /= z;
    }
    __syncthreads();
    for (int idx = tid; idx < ns * p.ld_j; idx += kThreads) {                   // joint = [self | weighted feature]
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
    st.fwd(7, j, p.ld_j, ns, g1, p.ld_g1, true);                                // mlp3.0   (begin_op's barrier publishes j)
    st.fwd(8, g1, p.ld_g1, ns, g2, p.ld_g, true);                               // mlp3.2
    st.fwd(9, g2, p.ld_g, ns, g3, p.ld_g, true);                                // mlp3.4
    st.fwd(10, g3, p.ld_g, ns, v, 1, false);                                    // mlp3.6 -> value

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
    wgrad(d, G, 10, dv, 1, g3, p.ld_g, ns);
    float *dg3 = d1;                                                // [ns][ld_g]
    st.bwd(10, dv, 1, ns, dg3, p.ld_g, g3, p.ld_g);
    // mlp3.4
    wgrad(d, G, 9, dg3, p.ld_g, g2, p.ld_g, ns);
    float *dg2 = d0;                                                // dv is dead
    st.bwd(9, dg3, p.ld_g, ns, dg2, p.ld_g, g2, p.ld_g);
    // mlp3.2
    wgrad(d, G, 8, dg2, p.ld_g, g1, p.ld_g1, ns);
    float *dg1 = d1;                                                // dg3 is dead
    st.bwd(8, dg2, p.ld_g, ns, dg1, p.ld_g1, g1, p.ld_g1);
    // mlp3.0
    wgrad(d, G, 7, dg1, p.ld_g1, j, p.ld_j, ns);
    float *dj = d0;                                                 // [ns][ld_j]; the self-state part has no parameters upstream
    st.bwd(7, dg1, p.ld_g1, ns, dj, p.ld_j, nullptr, 0);
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
    wgrad(d, G, 3, df, p.ld_f, f1, p.ld_f1, R);
    wgrad(d, G, 6, dsc, 1, t2, p.ld_t, R);
    float *df1 = d0;                                                // [R][ld_f1]  (dj is dead)
    st.bwd(3, df, p.ld_f, R, df1, p.ld_f1, f1, p.ld_f1);
    // mlp2.0's weights now; its data path joins de below
    wgrad(d, G, 2, df1, p.ld_f1, e, p.ld_e, R);
    float *dt2 = d1;                                                // [R][ld_t]  (df is dead)
    st.bwd(6, dsc, 1, R, dt2, p.ld_t, t2, p.ld_t);                  // dt2 = ds * W_att4[0][:]
    // attention.2
    wgrad(d, G, 5, dt2, p.ld_t, t1, p.ld_t, R);
    float *dt1 = t2;                                                // t2 is dead once its mask and attention.4's gradient are taken
    st.bwd(5, dt2, p.ld_t, R, dt1, p.ld_t, t1, p.ld_t);
    // attention.0 on u = [e | mean] (or on e)
    wgrad(d, G, 4, dt1, p.ld_t, att_in, ld_att, R);
    float *de = t1;                                                 // t1 is dead; rows of ld_t floats
    if (d.no_gs) {
        st.bwd(4, dt1, p.ld_t, R, de, p.ld_t, nullptr, 0);          // de_i = du_i
    } else {
        float *du = d1;                                             // [R][ld_u]  (dt2 is dead)
        st.bwd(4, dt1, p.ld_t, R, du, p.ld_u, nullptr, 0);
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
    st.bwd(2, df1, p.ld_f1, R, de, p.ld_t, e, p.ld_e, true);        // += df1 * W_mlp2.0   (begin_op's barrier publishes de)
    // mlp1.2
    wgrad(d, G, 1, de, p.ld_t, a1, p.ld_a1, R);
    float *da1 = d1;                                                // [R][ld_a1]  (du is dead)
    st.bwd(1, de, p.ld_t, R, da1, p.ld_a1, a1, p.ld_a1);
    // mlp1.0 (no gradient w.r.t. the input)
    wgrad(d, G, 0, da1, p.ld_a1, xs, p.ld_x, R);
    st.finish();
}

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
    float *G = gpart + (size_t)blockIdx.x * d.n_params;
    Staging st(d, Wt, Wa, sm + pad4(pmax.total), nbuf);

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
            st.fwd(0, xs, p.ld_x, H, m[0], p.ld_m[0], true);
            st.fwd(1, m[0], p.ld_m[0], H, m[1], p.ld_m[1], true);
            st.fwd(2, m[1], p.ld_m[1], H, m[2], p.ld_m[2], true);
            st.fwd(3, m[2], p.ld_m[2], H, m[3], p.ld_m[3], false);
            seq = m[3]; ld_seq = p.ld_m[3];
        }
        st.fwd(d.ih, seq, ld_seq, H, gt, p.ld_g4, false);                      // x_t W_ih^T + b_ih for every step at once
        const float *whh = st.begin_op(d.hh, 0);                               // W_hh^T | b_hh, kept for the whole loop
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
        st.end_op();
        for (int k = tid; k < p.ld_j; k += kThreads)                           // [state[:, 0, :self_dim] | h_n]
            j[k] = k < d.self_dim ? xs[k] : (k < d.self_dim + nh ? hs[(size_t)H * p.ld_h + k - d.self_dim] : 0.0f);
        vin = j; ld_vin = p.ld_j;
    }
    const int l0 = d.mlp0;
    st.fwd(l0, vin, ld_vin, ns, a[0], p.ld_a[0], true);    // (begin_op's barrier publishes j)
    st.fwd(l0 + 1, a[0], p.ld_a[0], ns, a[1], p.ld_a[1], true);
    st.fwd(l0 + 2, a[1], p.ld_a[1], ns, a[2], p.ld_a[2], true);
    st.fwd(l0 + 3, a[2], p.ld_a[2], ns, v, 1, false);

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
    wgrad(d, G, l0 + 3, dv, 1, a[2], p.ld_a[2], ns);
    st.bwd(l0 + 3, dv, 1, ns, d1, p.ld_a[2], a[2], p.ld_a[2]);
    wgrad(d, G, l0 + 2, d1, p.ld_a[2], a[1], p.ld_a[1], ns);
    st.bwd(l0 + 2, d1, p.ld_a[2], ns, d0, p.ld_a[1], a[1], p.ld_a[1]);
    wgrad(d, G, l0 + 1, d0, p.ld_a[1], a[0], p.ld_a[0], ns);
    st.bwd(l0 + 1, d0, p.ld_a[1], ns, d1, p.ld_a[0], a[0], p.ld_a[0]);
    wgrad(d, G, l0, d1, p.ld_a[0], vin, ld_vin, ns);
    if (!lstm) { st.finish(); return; }                 // CADRL: no gradient w.r.t. the input

    float *dj = d0;
    st.bwd(l0, d1, p.ld_a[0], 1, dj, p.ld_j, nullptr, 0);
    // BPTT from dh_H = dj[self_dim:], dc_H = 0.  Thread k owns cell k in both phases of a step.
    for (int k = tid; k < nh; k += kThreads) { dh[k] = dj[d.self_dim + k]; dc[k] = 0.0f; }
    const float *whh = st.begin_op(d.hh, 1);            // W_hh [4h][h]: dh_{t-1} = dgates_t W_hh
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
    st.end_op();
    wgrad(d, G, d.ih, dg, p.ld_g4, seq, ld_seq, H);     // dW_ih, bias_ih
    wgrad(d, G, d.hh, dg, p.ld_g4, hs, p.ld_h, H);      // dW_hh over [h_0 .. h_{H-1}], bias_hh
    if (!d.vn2) { st.finish(); return; }
    float *m[4] = {sm + p.m[0], sm + p.m[1], sm + p.m[2], sm + p.m[3]};
    st.bwd(d.ih, dg, p.ld_g4, H, d0, p.ld_m[3], nullptr, 0);             // dx_t = dgates_t W_ih (mlp1's last layer: no ReLU)
    wgrad(d, G, 3, d0, p.ld_m[3], m[2], p.ld_m[2], H);
    st.bwd(3, d0, p.ld_m[3], H, d1, p.ld_m[2], m[2], p.ld_m[2]);
    wgrad(d, G, 2, d1, p.ld_m[2], m[1], p.ld_m[1], H);
    st.bwd(2, d1, p.ld_m[2], H, d0, p.ld_m[1], m[1], p.ld_m[1]);
    wgrad(d, G, 1, d0, p.ld_m[1], m[0], p.ld_m[0], H);
    st.bwd(1, d0, p.ld_m[1], H, d1, p.ld_m[0], m[0], p.ld_m[0]);
    wgrad(d, G, 0, d1, p.ld_m[0], xs, p.ld_x, H);
    st.finish();
}

// ---------------- the world models (crowd_nav/policy/world_model.py:20-106) ----------------
// Loss of both: MSELoss(mean) over the batch x H x 2 predicted velocities.

// AttentionWorld's shared-memory plan (floats) for the R = H rows of one sample; every row stride is a multiple of 4 floats
struct WPlan {
    int ld_x, ld_a1, ld_e, ld_f1, ld_f, ld_u, ld_t, ld_j, ld_g1, ld_g, ld_o;
    int x, a1, e, f1, f, u, t1, t2, sc, wt, dc, j, g1, g2, g3, o, d0, d1, total;
};

__host__ __device__ inline WPlan make_wplan(const NetDims &d, int R)
{
    WPlan p;
    p.ld_x = pad4(d.in); p.ld_a1 = pad4(d.L[0].out); p.ld_e = pad4(d.L[1].out); p.ld_f1 = pad4(d.L[2].out);
    p.ld_f = pad4(d.L[3].out); p.ld_u = pad4(d.L[4].in);
    p.ld_t = pad4(max(max(d.L[4].out, d.L[5].out), d.L[1].out));      // t1 / t2 rows also host de (mlp1's output gradient)
    p.ld_j = pad4(d.L[7].in); p.ld_g1 = pad4(d.L[7].out); p.ld_g = pad4(max(d.L[8].out, d.L[9].out)); p.ld_o = pad4(d.L[10].out);
    int o = 0;
    p.x = o; o += R * p.ld_x;
    p.a1 = o; o += R * p.ld_a1;
    p.e = o; o += R * p.ld_e;
    p.f1 = o; o += R * p.ld_f1;
    p.f = o; o += R * p.ld_f;
    p.u = o; o += R * p.ld_u;
    p.t1 = o; o += R * p.ld_t;
    p.t2 = o; o += R * p.ld_t;
    p.sc = o; o += pad4(R);
    p.wt = o; o += pad4(R);
    p.dc = o; o += p.ld_f;
    p.j = o; o += R * p.ld_j;
    p.g1 = o; o += R * p.ld_g1;
    p.g2 = o; o += R * p.ld_g;
    p.g3 = o; o += R * p.ld_g;
    p.o = o; o += R * p.ld_o;
    // two gradient scratch buffers, each as wide as the widest gradient row they hold
    const int wide = max(max(max(p.ld_u, p.ld_a1), max(p.ld_g1, p.ld_j)), max(max(p.ld_t, p.ld_g), max(p.ld_f, p.ld_o)));
    p.d0 = o; o += R * wide;
    p.d1 = o; o += R * wide;
    p.total = o;
    return p;
}

// AttentionWorld: one CTA per sample, its H rows through SARL's blocks -- mlp1, mlp2, attention on [e_i | mean e], the masked
// softmax -- and then mlp3 on EVERY row, joint_i = [x_i | the sample's weighted feature] -> (vx, vy) of human i.  The op list
// is SARL's (forward 0..10, backward-data 10, 9, 8, 7, 3, 6, 5, 4, 2, 1).  Backward differences from SARL: mlp3's gradients
// run over R rows, d(feature) is the sum over the rows of the feature columns of d(joint_i), and the first d.in columns of
// d(joint_i) (the input itself) are dropped.  fwd_only: the squared errors alone (the op list then ends after layer 10).
__global__ void __launch_bounds__(kThreads, 1)
world_attention_fwd_bwd_kernel(NetDims d, const float *__restrict__ Wt, const float *__restrict__ Wa, const float *__restrict__ X,
                               const float *__restrict__ target, const int64_t *__restrict__ index, int B, int H, int nbuf,
                               int fwd_only, float *__restrict__ gpart, float *__restrict__ loss_part)
{
    extern __shared__ __align__(16) float sm[];
    const int R = H, tid = threadIdx.x;
    const WPlan p = make_wplan(d, H);
    float *xs = sm + p.x, *a1 = sm + p.a1, *e = sm + p.e, *f1 = sm + p.f1, *f = sm + p.f, *u = sm + p.u, *t1 = sm + p.t1,
          *t2 = sm + p.t2, *sc = sm + p.sc, *wt = sm + p.wt, *dcv = sm + p.dc, *j = sm + p.j, *g1 = sm + p.g1, *g2 = sm + p.g2,
          *g3 = sm + p.g3, *out = sm + p.o, *d0 = sm + p.d0, *d1 = sm + p.d1;
    const int E1 = d.L[1].out, F = d.L[3].out, IN = d.in, O = d.L[10].out;
    const size_t item = index ? (size_t)index[blockIdx.x] : (size_t)blockIdx.x;
    Staging st(d, Wt, Wa, sm + pad4(p.total), nbuf);

    // ---------------- forward (world_model.py:71-106), the arithmetic of attention_world_kernel ----------------
    for (int idx = tid; idx < R * p.ld_x; idx += kThreads) {
        const int r = idx / p.ld_x, k = idx - r * p.ld_x;
        xs[idx] = k < IN ? X[(item * H + r) * IN + k] : 0.0f;
    }
    st.fwd(0, xs, p.ld_x, R, a1, p.ld_a1, true);                                // mlp1.0 + ReLU
    st.fwd(1, a1, p.ld_a1, R, e, p.ld_e, true);                                 // mlp1.2 + ReLU
    st.fwd(2, e, p.ld_e, R, f1, p.ld_f1, true, false);                          // mlp2.0 + ReLU
    for (int k = tid; k < E1; k += kThreads) {                                  // u = [e_i | mean over the sample's humans]
        float m = 0.0f;
        for (int h = 0; h < H; ++h) m += e[(size_t)h * p.ld_e + k];
        m /= (float)H;
        for (int h = 0; h < H; ++h) {
            u[(size_t)h * p.ld_u + k] = e[(size_t)h * p.ld_e + k];
            u[(size_t)h * p.ld_u + E1 + k] = m;
        }
    }
    st.end_op();
    st.fwd(3, f1, p.ld_f1, R, f, p.ld_f, false);                                // mlp2.2
    st.fwd(4, u, p.ld_u, R, t1, p.ld_t, true);                                  // attention.0 + ReLU
    st.fwd(5, t1, p.ld_t, R, t2, p.ld_t, true);                                 // attention.2 + ReLU
    st.fwd(6, t2, p.ld_t, R, sc, 1, false);                                     // attention.4 -> score
    if (tid == 0) {                                                             // masked softmax (world_model.py:85-86)
        float z = 0.0f;
        for (int h = 0; h < H; ++h) {
            const float s = sc[h];
            const float ex = expf(s) * (s != 0.0f ? 1.0f : 0.0f);
            wt[h] = ex; z += ex;
        }
        for (int h = 0; h < H; ++h) wt[h] /= z;
    }
    __syncthreads();
    for (int idx = tid; idx < R * p.ld_j; idx += kThreads) {                    // joint_i = [x_i | weighted feature]
        const int r = idx / p.ld_j, k = idx - r * p.ld_j;
        float val = 0.0f;
        if (k < IN) val = xs[(size_t)r * p.ld_x + k];
        else if (k < IN + F)
            for (int h = 0; h < H; ++h) val = fmaf(wt[h], f[(size_t)h * p.ld_f + k - IN], val);
        j[idx] = val;
    }
    st.fwd(7, j, p.ld_j, R, g1, p.ld_g1, true);                                 // mlp3.0   (begin_op's barrier publishes j)
    st.fwd(8, g1, p.ld_g1, R, g2, p.ld_g, true);                                // mlp3.2
    st.fwd(9, g2, p.ld_g, R, g3, p.ld_g, true);                                 // mlp3.4
    st.fwd(10, g3, p.ld_g, R, out, p.ld_o, false);                              // mlp3.6 -> (vx, vy)

    // ---------------- loss and backward ----------------
    // MSELoss(mean) over B x H x O outputs: dL/dout = 2 (out - y) / (B H O)
    const float *y = target + item * H * O;
    if (tid == 0) {
        float ls = 0.0f;
        for (int i = 0; i < R * O; ++i) { const float df = out[(size_t)(i / O) * p.ld_o + i % O] - y[i]; ls += df * df; }
        loss_part[blockIdx.x] = ls;
    }
    if (fwd_only) { st.finish(); return; }
    float *G = gpart + (size_t)blockIdx.x * d.n_params;
    const float norm = 2.0f / (float)((int64_t)B * H * O);
    float *dout = d0;                                               // [R][ld_o]
    for (int i = tid; i < R * O; i += kThreads) {
        const size_t at = (size_t)(i / O) * p.ld_o + i % O;
        dout[at] = norm * (out[at] - y[i]);
    }
    __syncthreads();
    // mlp3 over every row
    wgrad(d, G, 10, dout, p.ld_o, g3, p.ld_g, R);
    float *dg3 = d1;
    st.bwd(10, dout, p.ld_o, R, dg3, p.ld_g, g3, p.ld_g);
    wgrad(d, G, 9, dg3, p.ld_g, g2, p.ld_g, R);
    float *dg2 = d0;                                                // dout is dead
    st.bwd(9, dg3, p.ld_g, R, dg2, p.ld_g, g2, p.ld_g);
    wgrad(d, G, 8, dg2, p.ld_g, g1, p.ld_g1, R);
    float *dg1 = d1;                                                // dg3 is dead
    st.bwd(8, dg2, p.ld_g, R, dg1, p.ld_g1, g1, p.ld_g1);
    wgrad(d, G, 7, dg1, p.ld_g1, j, p.ld_j, R);
    float *dj = d0;                                                 // [R][ld_j]; x_i's columns have no parameters upstream
    st.bwd(7, dg1, p.ld_g1, R, dj, p.ld_j, nullptr, 0);
    // d(feature) = sum over the rows of d(joint_i)[IN:]
    for (int k = tid; k < F; k += kThreads) {
        float s = 0.0f;
        for (int r = 0; r < R; ++r) s += dj[(size_t)r * p.ld_j + IN + k];
        dcv[k] = s;
    }
    __syncthreads();
    // weighted feature c = sum_i w_i f_i :  df_i = w_i dc,  dw_i = dc . f_i ;  softmax: ds_i = w_i (dw_i - sum_k w_k dw_k)
    float *df = d1;                                                 // [R][ld_f]  (dg1 is dead)
    float *dsc = sc;                                                // scores are dead after the softmax: reuse for ds
    if (tid < R) {
        float dw = 0.0f;
        for (int k = 0; k < F; ++k) dw = fmaf(dcv[k], f[(size_t)tid * p.ld_f + k], dw);
        dsc[tid] = dw;
    }
    for (int idx = tid; idx < R * F; idx += kThreads) {
        const int r = idx / F, k = idx - r * F;
        df[(size_t)r * p.ld_f + k] = wt[r] * dcv[k];
    }
    __syncthreads();
    if (tid == 0) {
        float dot = 0.0f;
        for (int h = 0; h < H; ++h) dot = fmaf(wt[h], dsc[h], dot);
        for (int h = 0; h < H; ++h) dsc[h] = wt[h] * (dsc[h] - dot);
    }
    __syncthreads();
    // from here on SARL's backward with one sample: mlp2.2 (no ReLU after it) and attention.4
    wgrad(d, G, 3, df, p.ld_f, f1, p.ld_f1, R);
    wgrad(d, G, 6, dsc, 1, t2, p.ld_t, R);
    float *df1 = d0;                                                // [R][ld_f1]  (dj is dead)
    st.bwd(3, df, p.ld_f, R, df1, p.ld_f1, f1, p.ld_f1);
    wgrad(d, G, 2, df1, p.ld_f1, e, p.ld_e, R);
    float *dt2 = d1;                                                // [R][ld_t]  (df is dead)
    st.bwd(6, dsc, 1, R, dt2, p.ld_t, t2, p.ld_t);
    wgrad(d, G, 5, dt2, p.ld_t, t1, p.ld_t, R);
    float *dt1 = t2;                                                // t2 is dead
    st.bwd(5, dt2, p.ld_t, R, dt1, p.ld_t, t1, p.ld_t);
    wgrad(d, G, 4, dt1, p.ld_t, u, p.ld_u, R);
    float *de = t1, *du = d1;                                       // t1 is dead; du: dt2 is dead
    st.bwd(4, dt1, p.ld_t, R, du, p.ld_u, nullptr, 0);
    for (int k = tid; k < E1; k += kThreads) {                      // de_i = du_i[:E1] + (1/H) sum_k du_k[E1:]
        float m = 0.0f;
        for (int h = 0; h < H; ++h) m += du[(size_t)h * p.ld_u + E1 + k];
        m /= (float)H;
        for (int h = 0; h < H; ++h) de[(size_t)h * p.ld_t + k] = du[(size_t)h * p.ld_u + k] + m;
    }
    st.bwd(2, df1, p.ld_f1, R, de, p.ld_t, e, p.ld_e, true);        // += df1 * W_mlp2.0   (begin_op's barrier publishes de)
    wgrad(d, G, 1, de, p.ld_t, a1, p.ld_a1, R);
    float *da1 = d1;
    st.bwd(1, de, p.ld_t, R, da1, p.ld_a1, a1, p.ld_a1);
    wgrad(d, G, 0, da1, p.ld_a1, xs, p.ld_x, R);
    st.finish();
}

// MlpWorld's shared-memory plan (floats) for ns samples = ns rows
struct MPlan { int ld_x, ld_a[3], ld_o; int x, a[3], o, d0, d1, total; };

__host__ __device__ inline MPlan make_mplan(const NetDims &d, int ns)
{
    MPlan p;
    int o = 0, wide = 0;
    p.ld_x = pad4(d.L[0].in); p.x = o; o += ns * p.ld_x;
    for (int i = 0; i < 3; ++i) { p.ld_a[i] = pad4(d.L[i].out); p.a[i] = o; o += ns * p.ld_a[i]; wide = max(wide, p.ld_a[i]); }
    p.ld_o = pad4(d.L[3].out); p.o = o; o += ns * p.ld_o; wide = max(wide, p.ld_o);
    p.d0 = o; o += ns * wide;
    p.d1 = o; o += ns * wide;
    p.total = o;
    return p;
}

// Inverted dropout (torch.nn.Dropout in training mode) on the post-ReLU activations a[ns][units] of `layer`: a unit is kept
// with probability 1 - p and then scaled by 1 / (1 - p).  The draw of (batch position s0 + s, layer, unit) is word 0 of the
// Philox block with counter (unit, layer, position, step) and key seed: independent of how the batch is split into CTAs.
__device__ __noinline__ void dropout_fwd(float *a, int ld, int ns, int units, int layer, int s0, const WorldStep &w, int mask_ld,
                                         int mask_off)
{
    const float scale = 1.0f / (1.0f - w.p);
    for (int idx = threadIdx.x; idx < ns * units; idx += kThreads) {
        const int s = idx / units, k = idx - s * units;
        Philox ph;
        ph.key[0] = (uint32_t)w.seed; ph.key[1] = (uint32_t)(w.seed >> 32);
        ph.ctr[0] = (uint32_t)k; ph.ctr[1] = (uint32_t)layer; ph.ctr[2] = (uint32_t)(s0 + s); ph.ctr[3] = w.step;
        uint32_t r[4];
        ph.block(r);
        const bool keep = (float)(r[0] >> 8) * (1.0f / 16777216.0f) >= w.p;
        float &v = a[(size_t)s * ld + k];
        v = keep ? v * scale : 0.0f;
        if (w.mask) w.mask[(size_t)(s0 + s) * mask_ld + mask_off + k] = keep ? 1 : 0;
    }
}

// d(post-ReLU activation) -> times 1 / (1 - p): the dropped units were already zeroed by the ReLU gate (their activation is 0)
__device__ __forceinline__ void dropout_bwd(float *g, int ld, int ns, int units, float p)
{
    const float scale = 1.0f / (1.0f - p);
    for (int idx = threadIdx.x; idx < ns * units; idx += kThreads) {
        const int s = idx / units, k = idx - s * units;
        g[(size_t)s * ld + k] *= scale;
    }
    __syncthreads();
}

// MlpWorld: mlp (4H -> 128 -> 64 -> 12 -> 2H) on one row per sample, ReLU + dropout after layers 0 and 1, ReLU after layer 2,
// tanh at the end; spc samples per CTA (CADRL's layout: every layer is one pass over its weight block).  Op list: forward
// 0..3, backward-data 3, 2, 1 (no gradient w.r.t. the input).
__global__ void __launch_bounds__(kThreads, 1)
world_mlp_fwd_bwd_kernel(NetDims d, const float *__restrict__ Wt, const float *__restrict__ Wa, const float *__restrict__ X,
                         const float *__restrict__ target, const int64_t *__restrict__ index, int B, int spc, int nbuf,
                         WorldStep w, float *__restrict__ gpart, float *__restrict__ loss_part)
{
    extern __shared__ __align__(16) float sm[];
    const int s0 = blockIdx.x * spc;
    const int ns = min(spc, B - s0);
    const MPlan p = make_mplan(d, ns);
    const MPlan pmax = make_mplan(d, spc);              // the staging buffers sit behind the largest activation plan
    const int tid = threadIdx.x, IN = d.L[0].in, O = d.L[3].out, U0 = d.L[0].out, U1 = d.L[1].out;
    float *xs = sm + p.x, *o = sm + p.o, *d0 = sm + p.d0, *d1 = sm + p.d1;
    float *a[3] = {sm + p.a[0], sm + p.a[1], sm + p.a[2]};
    const bool drop = w.p > 0.0f && !w.fwd_only;
    Staging st(d, Wt, Wa, sm + pad4(pmax.total), nbuf);

    for (int idx = tid; idx < ns * p.ld_x; idx += kThreads) {
        const int s = idx / p.ld_x, k = idx - s * p.ld_x;
        const size_t item = index ? (size_t)index[s0 + s] : (size_t)(s0 + s);
        xs[idx] = k < IN ? X[item * IN + k] : 0.0f;
    }
    st.fwd(0, xs, p.ld_x, ns, a[0], p.ld_a[0], true);
    if (drop) dropout_fwd(a[0], p.ld_a[0], ns, U0, 0, s0, w, U0 + U1, 0);
    st.fwd(1, a[0], p.ld_a[0], ns, a[1], p.ld_a[1], true);     // (begin_op's barrier publishes the dropout)
    if (drop) dropout_fwd(a[1], p.ld_a[1], ns, U1, 1, s0, w, U0 + U1, U0);
    st.fwd(2, a[1], p.ld_a[1], ns, a[2], p.ld_a[2], true);
    st.fwd(3, a[2], p.ld_a[2], ns, o, p.ld_o, false);
    for (int idx = tid; idx < ns * O; idx += kThreads) {
        float &v = o[(size_t)(idx / O) * p.ld_o + idx % O];
        v = tanhf(v);
    }
    __syncthreads();

    // MSELoss(mean) over B x O outputs; tanh' = 1 - out^2
    if (tid == 0) {
        float ls = 0.0f;
        for (int s = 0; s < ns; ++s) {
            const float *y = target + (index ? (size_t)index[s0 + s] : (size_t)(s0 + s)) * O;
            for (int k = 0; k < O; ++k) { const float df = o[(size_t)s * p.ld_o + k] - y[k]; ls += df * df; }
        }
        loss_part[blockIdx.x] = ls;
    }
    if (w.fwd_only) { st.finish(); return; }
    float *G = gpart + (size_t)blockIdx.x * d.n_params;
    const float norm = 2.0f / (float)((int64_t)B * O);
    for (int idx = tid; idx < ns * O; idx += kThreads) {
        const int s = idx / O, k = idx - s * O;
        const float *y = target + (index ? (size_t)index[s0 + s] : (size_t)(s0 + s)) * O;
        const float v = o[(size_t)s * p.ld_o + k];
        d0[(size_t)s * p.ld_o + k] = norm * (v - y[k]) * (1.0f - v * v);
    }
    __syncthreads();
    wgrad(d, G, 3, d0, p.ld_o, a[2], p.ld_a[2], ns);
    st.bwd(3, d0, p.ld_o, ns, d1, p.ld_a[2], a[2], p.ld_a[2]);
    wgrad(d, G, 2, d1, p.ld_a[2], a[1], p.ld_a[1], ns);
    st.bwd(2, d1, p.ld_a[2], ns, d0, p.ld_a[1], a[1], p.ld_a[1]);
    if (drop) dropout_bwd(d0, p.ld_a[1], ns, U1, w.p);
    wgrad(d, G, 1, d0, p.ld_a[1], a[0], p.ld_a[0], ns);
    st.bwd(1, d0, p.ld_a[1], ns, d1, p.ld_a[0], a[0], p.ld_a[0]);
    if (drop) dropout_bwd(d1, p.ld_a[0], ns, U0, w.p);
    wgrad(d, G, 0, d1, p.ld_a[0], xs, p.ld_x, ns);
    st.finish();
}

constexpr int kWorldMlpSPC = kCadrlSPC;

}  // namespace

int trainer_spc(const NetDims &d)
{
    if (d.net == kNetWorldMlp) return kWorldMlpSPC;
    return d.net == CN_NET_SARL ? kSarlSPC : d.net == CN_NET_CADRL ? kCadrlSPC : 1;
}

size_t trainer_smem(const NetDims &d, int H, int nbuf)
{
    int act;
    if (d.net == kNetWorldAttention) act = make_wplan(d, H).total;
    else if (d.net == kNetWorldMlp) act = make_mplan(d, kWorldMlpSPC).total;
    else act = d.net == CN_NET_SARL ? make_plan(d, H, kSarlSPC).total : make_nplan(d, H, trainer_spc(d)).total;
    return sizeof(float) * ((size_t)pad4(act) + (size_t)nbuf * d.wbuf_floats);
}

cudaError_t trainer_configure(const NetDims &d)
{
    const void *kernel = d.net == CN_NET_SARL ? (const void *)trainer_fwd_bwd_kernel
                         : d.net == kNetWorldAttention ? (const void *)world_attention_fwd_bwd_kernel
                         : d.net == kNetWorldMlp ? (const void *)world_mlp_fwd_bwd_kernel
                                                 : (const void *)trainer_nets_fwd_bwd_kernel;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTrainerMaxSmem);
}

int trainer_launch(const NetDims &d, const float *Wt, const float *Wa, const float *X, const float *target,
                   const int64_t *index, int batch, int H, float *gpart, float *loss_part, int *nparts, cudaStream_t s,
                   const WorldStep *w)
{
    const int spc = trainer_spc(d);
    *nparts = (batch + spc - 1) / spc;
    // two staging buffers (the next weight block is copied while the current op computes) when they fit, else one
    const int nbuf = trainer_smem(d, H, 2) <= kTrainerMaxSmem ? 2 : 1;
    const size_t smem = trainer_smem(d, H, nbuf);
    if (d.net == CN_NET_SARL)
        trainer_fwd_bwd_kernel<<<*nparts, kThreads, smem, s>>>(d, Wt, Wa, X, target, index, batch, H, nbuf, gpart, loss_part);
    else if (d.net == kNetWorldAttention)
        world_attention_fwd_bwd_kernel<<<*nparts, kThreads, smem, s>>>(d, Wt, Wa, X, target, index, batch, H, nbuf, w->fwd_only,
                                                                       gpart, loss_part);
    else if (d.net == kNetWorldMlp)
        world_mlp_fwd_bwd_kernel<<<*nparts, kThreads, smem, s>>>(d, Wt, Wa, X, target, index, batch, spc, nbuf, *w, gpart,
                                                                 loss_part);
    else
        trainer_nets_fwd_bwd_kernel<<<*nparts, kThreads, smem, s>>>(d, Wt, Wa, X, target, index, batch, H, spc, nbuf, gpart,
                                                                    loss_part);
    CN_LAUNCH_CHECK();
    return CN_OK;
}
