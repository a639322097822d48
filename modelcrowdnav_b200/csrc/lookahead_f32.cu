// lookahead_f32.cu -- SARL one-step lookahead, FP32 CUDA-core path (CN_PREC_F32).
//
// One CTA evaluates a chunk of candidate actions of one environment entirely on chip:
//   K3  propagate + reward + rotate      -> X   (rows = actions x humans, 13 features)   smem
//   K4  mlp1 -> mlp2 / attention -> mlp3 -> V                                              smem
//   K5  value = reward + gamma_bar * V   -> values[E][A] (HBM), then argmax_kernel
// No per-layer activation ever reaches HBM.  This path is the arithmetic twin of torch's fp32
// ValueNetwork (used for parity at 1e-5 and for TD targets); the tensor-core path lives in
// lookahead_tc.cu.
//
// Reference (file:line relative to the reference root):
//   MultiHumanRL.predict            crowd_nav/policy/multi_human_rl.py:11-63
//   MultiHumanRL.compute_reward     crowd_nav/policy/multi_human_rl.py:65-88
//   MultiHumanRL.transform          crowd_nav/policy/multi_human_rl.py:90-104
//   CADRL.propagate / rotate        crowd_nav/policy/cadrl.py:104-129,217-252
//   ValueNetwork.forward            crowd_nav/policy/sarl.py:28-65
//   CrowdSim.onestep_lookahead      crowd_sim/envs/crowd_sim.py:325-329 (query_env)
//   Policy.reach_destination        crowd_sim/envs/policy/policy.py:43-49
#include "env_math.cuh"

#include <math.h>

namespace {

constexpr int kThreads = 256;
constexpr int kRowsCap = 64;  // rows (action x human) per CTA
constexpr size_t kMaxDynSmem = 232448;   // 227 KB: the opt-in dynamic shared memory limit of sm_100

__host__ __device__ inline int pad4(int x) { return (x + 3) & ~3; }

struct F32Plan {
    int H, A, CA;             // humans, actions, actions per chunk
    int wX, wT0, wM1, wF, wJ; // padded smem row widths (floats)
    int oX, oT0, oM1, oF, oG, oJ, oS, oW, oV, oEnv, oOrd, oOm, total_floats;  // smem offsets (floats)
};

// out[r][n] = act( (accum ? out[r][n] : 0) + sum_k in[r / in_div][k] * Wt[k_off + k][n] (+ b[n]) )
// 4x4 register tile per thread; weights streamed from L1/L2 as float4, activations broadcast from smem.
__device__ void layer(const LinearDev L, int k_off, int K, const float *__restrict__ in, int ldin, int in_div,
                      float *__restrict__ out, int ldout, int rows, bool accum, bool add_bias, bool relu)
{
    const int N = L.out;
    const int ntc = (N + 3) >> 2, ntr = (rows + 3) >> 2;
    for (int tile = threadIdx.x; tile < ntr * ntc; tile += blockDim.x) {
        const int tr = tile / ntc, tc = tile - tr * ntc;
        const int r0 = tr * 4, n0 = tc * 4;
        const float *ip[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int r = r0 + i;
            if (r >= rows) r = rows - 1;
            ip[i] = in + (size_t)(r / in_div) * ldin;
        }
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
        const float *wp = L.wt + (size_t)k_off * L.ld + n0;
#pragma unroll 4
        for (int k = 0; k < K; ++k) {
            const float4 w = __ldg(reinterpret_cast<const float4 *>(wp + (size_t)k * L.ld));
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float a = ip[i][k];
                acc[i][0] = fmaf(a, w.x, acc[i][0]);
                acc[i][1] = fmaf(a, w.y, acc[i][1]);
                acc[i][2] = fmaf(a, w.z, acc[i][2]);
                acc[i][3] = fmaf(a, w.w, acc[i][3]);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = r0 + i;
            if (r >= rows) break;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int n = n0 + j;
                if (n >= N) break;
                float v = acc[i][j];
                if (accum) v += out[(size_t)r * ldout + n];
                if (add_bias) v += __ldg(L.b + n);
                if (relu) v = fmaxf(v, 0.0f);
                out[(size_t)r * ldout + n] = v;
            }
        }
    }
}

// N == 1 head: out[r] = in[r] . w + b
__device__ void head(const LinearDev L, const float *__restrict__ in, int ldin, float *__restrict__ out, int rows)
{
    for (int r = threadIdx.x; r < rows; r += blockDim.x) {
        float acc = 0.0f;
        const float *x = in + (size_t)r * ldin;
        for (int k = 0; k < L.in; ++k) acc = fmaf(x[k], __ldg(L.wt + (size_t)k * L.ld), acc);
        out[r] = acc + __ldg(L.b);
    }
}

// ValueNetwork.forward on `ng` groups of H rows whose 13-feature rows are already in X (sarl.py:28-65).
// Result: V[g] for g in [0, ng).
__device__ void sarl_forward_smem(const SarlWeightsDev &W, const SarlDims &d, const F32Plan &pl, float *sm, int ng)
{
    const int H = pl.H, rows = ng * H;
    float *X = sm + pl.oX, *T0 = sm + pl.oT0, *M1 = sm + pl.oM1, *F = sm + pl.oF, *G = sm + pl.oG;
    float *J = sm + pl.oJ, *S = sm + pl.oS, *Wt = sm + pl.oW, *Vv = sm + pl.oV;
    const int G1 = d.m1[1], FD = d.m2[1];

    layer(W.m1[0], 0, d.in, X, pl.wX, 1, T0, pl.wT0, rows, false, true, true);       // mlp1.0 + ReLU
    __syncthreads();
    layer(W.m1[1], 0, d.m1[0], T0, pl.wT0, 1, M1, pl.wM1, rows, false, true, true);  // mlp1.2 + ReLU (last_relu)
    __syncthreads();
    // global state = mean over humans (sarl.py:42), unless with_global_state = false; self_state = x[:, 0, :6] (sarl.py:36)
    if (!d.no_gs)
        for (int i = threadIdx.x; i < ng * G1; i += blockDim.x) {
            const int g = i / G1, k = i - g * G1;
            float s = 0.0f;
            for (int h = 0; h < H; ++h) s += M1[(size_t)(g * H + h) * pl.wM1 + k];
            G[(size_t)g * pl.wM1 + k] = s / (float)H;
        }
    for (int i = threadIdx.x; i < ng * d.self_dim; i += blockDim.x) {
        const int g = i / d.self_dim, k = i - g * d.self_dim;
        J[(size_t)g * pl.wJ + k] = X[(size_t)(g * H) * pl.wX + k];
    }
    layer(W.m2[0], 0, G1, M1, pl.wM1, 1, T0, pl.wT0, rows, false, true, true);       // mlp2.0 + ReLU
    __syncthreads();
    layer(W.m2[1], 0, d.m2[0], T0, pl.wT0, 1, F, pl.wF, rows, false, true, false);   // mlp2.2
    __syncthreads();
    if (d.no_gs) {
        // attention.0 on mlp1_out alone (sarl.py:47)
        layer(W.at[0], 0, G1, M1, pl.wM1, 1, T0, pl.wT0, rows, false, true, true);
    } else {
        // attention.0 on cat([mlp1_out, global]) (sarl.py:45): two partial products
        layer(W.at[0], 0, G1, M1, pl.wM1, 1, T0, pl.wT0, rows, false, false, false);
        __syncthreads();
        layer(W.at[0], G1, G1, G, pl.wM1, H, T0, pl.wT0, rows, true, true, true);
    }
    __syncthreads();
    layer(W.at[1], 0, d.at[0], T0, pl.wT0, 1, M1, pl.wM1, rows, false, true, true);  // attention.2 + ReLU
    __syncthreads();
    head(W.at[2], M1, pl.wM1, S, rows);                                              // attention.4 -> scores
    __syncthreads();
    // masked, un-stabilised softmax over humans (sarl.py:52-53)
    for (int g = threadIdx.x; g < ng; g += blockDim.x) {
        float ssum = 0.0f;
        for (int h = 0; h < H; ++h) {
            const float sc = S[g * H + h];
            const float se = expf(sc) * (sc != 0.0f ? 1.0f : 0.0f);
            Wt[g * H + h] = se;
            ssum += se;
        }
        for (int h = 0; h < H; ++h) Wt[g * H + h] = Wt[g * H + h] / ssum;
    }
    __syncthreads();
    // weighted feature (sarl.py:57-60) -> joint state (sarl.py:63)
    for (int i = threadIdx.x; i < ng * FD; i += blockDim.x) {
        const int g = i / FD, k = i - g * FD;
        float s = 0.0f;
        for (int h = 0; h < H; ++h) s += Wt[g * H + h] * F[(size_t)(g * H + h) * pl.wF + k];
        J[(size_t)g * pl.wJ + d.self_dim + k] = s;
    }
    __syncthreads();
    // mlp3 (sarl.py:64); U0 aliases T0, U1 aliases M1
    float *U0 = T0, *U1 = M1;
    layer(W.m3[0], 0, d.self_dim + FD, J, pl.wJ, 1, U0, pl.wT0, ng, false, true, true);
    __syncthreads();
    layer(W.m3[1], 0, d.m3[0], U0, pl.wT0, 1, U1, pl.wM1, ng, false, true, true);
    __syncthreads();
    layer(W.m3[2], 0, d.m3[1], U1, pl.wM1, 1, U0, pl.wT0, ng, false, true, true);
    __syncthreads();
    head(W.m3[3], U0, pl.wT0, Vv, ng);
    __syncthreads();
}

// CADRL (cadrl.py:22-30,160-166): value_network = mlp(13 -> m3) on every (robot, human) row; V[g] = min over the humans.
__device__ void cadrl_forward_smem(const SarlWeightsDev &W, const SarlDims &d, const F32Plan &pl, float *sm, int ng)
{
    const int H = pl.H, rows = ng * H;
    float *X = sm + pl.oX, *T0 = sm + pl.oT0, *M1 = sm + pl.oM1, *S = sm + pl.oS, *Vv = sm + pl.oV;
    layer(W.m3[0], 0, d.in, X, pl.wX, 1, T0, pl.wT0, rows, false, true, true);
    __syncthreads();
    layer(W.m3[1], 0, d.m3[0], T0, pl.wT0, 1, M1, pl.wM1, rows, false, true, true);
    __syncthreads();
    layer(W.m3[2], 0, d.m3[1], M1, pl.wM1, 1, T0, pl.wT0, rows, false, true, true);
    __syncthreads();
    head(W.m3[3], T0, pl.wT0, S, rows);
    __syncthreads();
    for (int g = threadIdx.x; g < ng; g += blockDim.x) {
        float m = S[g * H];
        for (int h = 1; h < H; ++h) m = fminf(m, S[g * H + h]);
        Vv[g] = m;
    }
    __syncthreads();
}

// LSTM-RL (lstm_rl.py:9-66): nn.LSTM over the H rows of a group (gate order i, f, g, o; h0 = c0 = 0), fed by the rows
// themselves (ValueNetwork1) or by mlp1(rows) (ValueNetwork2), then mlp(cat(self_state, h_n)).  Rows are already in
// network order (the lookahead sorts the humans, lstm_rl.py:99-104).
__device__ void lstm_forward_smem(const SarlWeightsDev &W, const SarlDims &d, const F32Plan &pl, float *sm, int ng)
{
    const int H = pl.H, rows = ng * H, Hh = d.lstm_h;
    float *X = sm + pl.oX, *T0 = sm + pl.oT0, *M1 = sm + pl.oM1, *Cc = sm + pl.oF, *Hs = sm + pl.oG;
    float *J = sm + pl.oJ, *Vv = sm + pl.oV;
    const float *in = X;
    int ldin = pl.wX;
    if (d.lm1[0] > 0) {                                                              // lstm_rl.py:56-58, no last ReLU
        layer(W.lm1[0], 0, d.in, X, pl.wX, 1, T0, pl.wT0, rows, false, true, true);
        __syncthreads();
        layer(W.lm1[1], 0, d.lm1[0], T0, pl.wT0, 1, M1, pl.wM1, rows, false, true, true);
        __syncthreads();
        layer(W.lm1[2], 0, d.lm1[1], M1, pl.wM1, 1, T0, pl.wT0, rows, false, true, true);
        __syncthreads();
        layer(W.lm1[3], 0, d.lm1[2], T0, pl.wT0, 1, M1, pl.wM1, rows, false, true, false);
        __syncthreads();
        in = M1; ldin = pl.wM1;
    }
    for (int i = threadIdx.x; i < ng * Hh; i += blockDim.x) {
        const int g = i / Hh, k = i - g * Hh;
        Hs[(size_t)g * pl.wM1 + k] = 0.0f;
        Cc[(size_t)g * pl.wF + k] = 0.0f;
    }
    for (int i = threadIdx.x; i < ng * d.self_dim; i += blockDim.x) {               // self_state = state[:, 0, :6]
        const int g = i / d.self_dim, k = i - g * d.self_dim;
        J[(size_t)g * pl.wJ + k] = X[(size_t)(g * H) * pl.wX + k];
    }
    __syncthreads();
    for (int t = 0; t < H; ++t) {
        // gates = W_ih x_t + b_ih + W_hh h + b_hh, one row per group (row stride H * ldin picks step t of every group)
        layer(W.lih, 0, d.lstm_in, in + (size_t)t * ldin, H * ldin, 1, T0, pl.wT0, ng, false, true, false);
        __syncthreads();
        layer(W.lhh, 0, Hh, Hs, pl.wM1, 1, T0, pl.wT0, ng, true, true, false);
        __syncthreads();
        for (int i = threadIdx.x; i < ng * Hh; i += blockDim.x) {
            const int g = i / Hh, k = i - g * Hh;
            const float *gt = T0 + (size_t)g * pl.wT0;
            const float ig = 1.0f / (1.0f + expf(-gt[k])), fg = 1.0f / (1.0f + expf(-gt[Hh + k]));
            const float gg = tanhf(gt[2 * Hh + k]), og = 1.0f / (1.0f + expf(-gt[3 * Hh + k]));
            const float c = fg * Cc[(size_t)g * pl.wF + k] + ig * gg;
            Cc[(size_t)g * pl.wF + k] = c;
            Hs[(size_t)g * pl.wM1 + k] = og * tanhf(c);
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < ng * Hh; i += blockDim.x) {
        const int g = i / Hh, k = i - g * Hh;
        J[(size_t)g * pl.wJ + d.self_dim + k] = Hs[(size_t)g * pl.wM1 + k];
    }
    __syncthreads();
    float *U0 = T0, *U1 = M1;
    layer(W.m3[0], 0, d.self_dim + Hh, J, pl.wJ, 1, U0, pl.wT0, ng, false, true, true);
    __syncthreads();
    layer(W.m3[1], 0, d.m3[0], U0, pl.wT0, 1, U1, pl.wM1, ng, false, true, true);
    __syncthreads();
    layer(W.m3[2], 0, d.m3[1], U1, pl.wM1, 1, U0, pl.wT0, ng, false, true, true);
    __syncthreads();
    head(W.m3[3], U0, pl.wT0, Vv, ng);
    __syncthreads();
}

__device__ __forceinline__ void net_forward_smem(const SarlWeightsDev &W, const SarlDims &d, const F32Plan &pl, float *sm, int ng)
{
    if (d.net == CN_NET_CADRL) cadrl_forward_smem(W, d, pl, sm, ng);
    else if (d.net == CN_NET_LSTM_RL) lstm_forward_smem(W, d, pl, sm, ng);
    else sarl_forward_smem(W, d, pl, sm, ng);
}

// grid = (E, chunks)
__global__ void __launch_bounds__(kThreads, 2)
lookahead_values_kernel(EnvParams p, SarlWeightsDev W, SarlDims d, F32Plan pl, const double *__restrict__ st,
                        const double *__restrict__ time, const double *__restrict__ human_v,
                        const uint8_t *__restrict__ frozen, const double *__restrict__ actions, int query_env,
                        double gamma, double gamma_bar_host, double v_pref_host, double *__restrict__ values,
                        const double *__restrict__ theta)
{
    extern __shared__ __align__(16) float sm[];
    const int e = blockIdx.x;
    if (frozen[e]) return;
    const EnvDims ed = p.d;
    const int H = pl.H;
    const int a0 = blockIdx.y * pl.CA;
    const int na = min(pl.CA, pl.A - a0);
    const int rows = na * H;
    double *env = reinterpret_cast<double *>(sm + pl.oEnv);  // [A1][8] + human next (px,py,vx,vy)[H] + reward[CA]
    double *hnext = env + (size_t)ed.A1 * F_COUNT;
    double *rew = hnext + (size_t)H * 4;
    float *X = sm + pl.oX;

    for (int i = threadIdx.x; i < ed.A1 * F_COUNT; i += blockDim.x) {
        const int a = i / F_COUNT, f = i - a * F_COUNT;
        env[i] = st[st_idx(ed, f, a, e)];
    }
    __syncthreads();
    auto ag = [&](int f, int a) { return env[a * F_COUNT + f]; };
    // network order of the humans: LstmRL.predict sorts them by DECREASING distance to the robot (stable, lstm_rl.py:99-104);
    // with query_env the next human states come back from the env in env order (multi_human_rl.py:37-38)
    int *ord = reinterpret_cast<int *>(sm + pl.oOrd);
    if (threadIdx.x == 0) {
        for (int h = 0; h < H; ++h) ord[h] = h;
        if (d.net == CN_NET_LSTM_RL && !query_env) {
            for (int i = 1; i < H; ++i) {
                const int oi = ord[i];
                const double di = norm2d(ag(F_PX, oi + 1) - ag(F_PX, 0), ag(F_PY, oi + 1) - ag(F_PY, 0));
                int j = i - 1;
                while (j >= 0 && norm2d(ag(F_PX, ord[j] + 1) - ag(F_PX, 0), ag(F_PY, ord[j] + 1) - ag(F_PY, 0)) < di) {
                    ord[j + 1] = ord[j];
                    --j;
                }
                ord[j + 1] = oi;
            }
        }
    }
    const double dt = p.time_step;
    const int kin = p.kinematics;
    const double th = kin != CN_KIN_HOLONOMIC ? theta[e] : 0.0;      // robot heading (cadrl.py:119: next_theta = theta + r)
    // next human states: query_env -> ORCA action (agent.py:63-74), else constant velocity (cadrl.py:107-109)
    for (int h = threadIdx.x; h < H; h += blockDim.x) {
        double hvx, hvy;
        if (query_env) { hvx = human_v[(size_t)(0 * H + h) * ed.E + e]; hvy = human_v[(size_t)(1 * H + h) * ed.E + e]; }
        else { hvx = ag(F_VX, h + 1); hvy = ag(F_VY, h + 1); }
        hnext[h * 4 + 0] = ag(F_PX, h + 1) + hvx * dt;
        hnext[h * 4 + 1] = ag(F_PY, h + 1) + hvy * dt;
        hnext[h * 4 + 2] = hvx;
        hnext[h * 4 + 3] = hvy;
    }
    __syncthreads();
    // reward per action
    for (int i = threadIdx.x; i < na; i += blockDim.x) {
        double ax, ay;
        cn_effective_velocity(kin, th, actions[2 * (a0 + i)], actions[2 * (a0 + i) + 1], ax, ay);
        double reward;
        if (query_env) {
            reward = cn_step_outcome(p, ag, H, time[e], ax, ay).reward;   // crowd_sim.py:325-329
        } else {
            // multi_human_rl.py:65-88 (end-point distances, constants hard-coded there)
            const double npx = ag(F_PX, 0) + ax * dt, npy = ag(F_PY, 0) + ay * dt, rr = ag(F_R, 0);
            double dmin = INFINITY;
            bool collision = false;
            for (int h = 0; h < H; ++h) {
                const double dist = norm2d(npx - hnext[h * 4 + 0], npy - hnext[h * 4 + 1]) - rr - ag(F_R, h + 1);
                if (dist < 0) { collision = true; break; }
                if (dist < dmin) dmin = dist;
            }
            const bool reaching_goal = norm2d(npx - ag(F_GX, 0), npy - ag(F_GY, 0)) < rr;
            if (collision) reward = -0.25;
            else if (reaching_goal) reward = 1;
            else if (dmin < 0.2) reward = (dmin - 0.2) * 0.5 * dt;
            else reward = 0;
        }
        rew[i] = reward;
    }
    // occupancy maps: built once per predict() from the next human states, in network order (multi_human_rl.py:47-49)
    float *OM = sm + pl.oOm;
    if (d.om_dim > 0) {
        for (int i = threadIdx.x; i < H; i += blockDim.x)
            occupancy_map_row(d, H, i, [&](int j, int f) { return hnext[ord[j] * 4 + f]; }, OM + (size_t)i * d.om_dim);
        __syncthreads();
    }
    // rotated joint-state rows (multi_human_rl.py:43-45): torch.Tensor([...]) rounds the doubles to fp32
    for (int r = threadIdx.x; r < rows; r += blockDim.x) {
        const int i = r / H, h = ord[r - i * H];
        double ax, ay;
        cn_effective_velocity(kin, th, actions[2 * (a0 + i)], actions[2 * (a0 + i) + 1], ax, ay);
        float s[14], o[13];
        s[0] = (float)(ag(F_PX, 0) + ax * dt); s[1] = (float)(ag(F_PY, 0) + ay * dt);
        s[2] = (float)ax; s[3] = (float)ay; s[4] = (float)ag(F_R, 0);
        s[5] = (float)ag(F_GX, 0); s[6] = (float)ag(F_GY, 0); s[7] = (float)ag(F_VPREF, 0);
        s[8] = kin != CN_KIN_HOLONOMIC ? (float)(th + actions[2 * (a0 + i) + 1]) : 0.0f;
        s[9] = (float)hnext[h * 4 + 0]; s[10] = (float)hnext[h * 4 + 1];
        s[11] = (float)hnext[h * 4 + 2]; s[12] = (float)hnext[h * 4 + 3]; s[13] = (float)ag(F_R, h + 1);
        cn_rotate(s, o, kin);
#pragma unroll
        for (int k = 0; k < 13; ++k) X[(size_t)r * pl.wX + k] = o[k];
        for (int k = 0; k < d.om_dim; ++k) X[(size_t)r * pl.wX + 13 + k] = OM[(size_t)(r - i * H) * d.om_dim + k];
    }
    __syncthreads();
    net_forward_smem(W, d, pl, sm, na);
    const float *Vv = sm + pl.oV;
    const double vp = ag(F_VPREF, 0);
    const double gamma_bar = (vp == v_pref_host) ? gamma_bar_host : pow(gamma, dt * vp);
    for (int i = threadIdx.x; i < na; i += blockDim.x)
        values[(size_t)e * pl.A + a0 + i] = rew[i] + gamma_bar * (double)Vv[i];   // multi_human_rl.py:52
}

// first-strict-max argmax + reach_destination + epsilon-greedy (multi_human_rl.py:22-30,53-58)
// One WARP per env: the A values of an env are one contiguous, coalesced read; lane l scans a = l, l + 32, ...
// (ascending, strict >: the lowest index wins inside a lane), then a shuffle reduction keeps the larger value and,
// on equal values, the lower index -- the reference's "first strict maximum".  NaN never wins; all-NaN -> best = -1.
__global__ void __launch_bounds__(128)
argmax_kernel(EnvParams p, int A, const double *__restrict__ st, const uint8_t *__restrict__ frozen,
              const double *__restrict__ values, const double *__restrict__ actions, double epsilon,
              uint32_t *__restrict__ step_ctr, double *__restrict__ action_xy,
              int32_t *__restrict__ action_idx, int32_t *__restrict__ bad_flag)
{
    const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const EnvDims d = p.d;
    // programmatic dependent launch (cn_lookahead_argmax): the grid may be resident before the value kernel has finished
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (e >= d.E || frozen[e]) return;       // warp-uniform
    double max_value = -INFINITY;
    int best = -1;
    for (int a = lane; a < A; a += 32) {
        const double v = values[(size_t)e * A + a];
        if (v > max_value) { max_value = v; best = a; }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, max_value, off);
        const int ob = __shfl_xor_sync(0xffffffffu, best, off);
        // a lane that saw only NaN / nothing has best = -1 and never wins; ties go to the lower action index
        if (ob >= 0 && (best < 0 || ov > max_value || (ov == max_value && ob < best))) { max_value = ov; best = ob; }
    }
    if (lane != 0) return;
    // policy.py:43-49: norm((py - gy, px - gx)) < radius
    const bool reached = norm2d(st[st_idx(d, F_PY, 0, e)] - st[st_idx(d, F_GY, 0, e)],
                                st[st_idx(d, F_PX, 0, e)] - st[st_idx(d, F_GX, 0, e)]) < st[st_idx(d, F_R, 0, e)];
    if (reached) best = 0;
    else {
        bool random_pick = false;
        if (epsilon > 0.0) {
            PhiloxStream rng;
            rng.init(p.seed, (uint64_t)(p.env_id_offset + e), step_ctr[e], 1u);
            step_ctr[e] += 1;
            if (rng.next() < epsilon) { best = min(A - 1, (int)(rng.next() * A)); random_pick = true; }
        }
        if (!random_pick && best < 0) { atomicExch(bad_flag, 1); atomicAdd(bad_flag + 1, 1); best = 0; }   // [1]: sticky count
    }
    action_idx[e] = best;
    action_xy[e] = actions[2 * best];
    action_xy[d.E + e] = actions[2 * best + 1];
}

// MultiHumanRL.transform (multi_human_rl.py:90-104): current joint state -> E x H x 13 fp32
// sort_humans: rows in LstmRL.predict's order (decreasing distance to the robot, stable: lstm_rl.py:99-104) -- what
// predict() leaves in last_state for LSTM-RL; 0 = env order (MultiHumanRL.transform itself never sorts).
__global__ void transform_kernel(EnvParams p, SarlDims nd, const double *__restrict__ st, const double *__restrict__ theta,
                                 float *__restrict__ out, int sort_humans)
{
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const EnvDims d = p.d;
    if (tid >= d.E * d.H) return;
    const int h = tid / d.E, e = tid - h * d.E;
    auto ag = [&](int f, int a) { return (float)st[st_idx(d, f, a, e)]; };
    float s[14], o[13];
    s[0] = ag(F_PX, 0); s[1] = ag(F_PY, 0); s[2] = ag(F_VX, 0); s[3] = ag(F_VY, 0); s[4] = ag(F_R, 0);
    s[5] = ag(F_GX, 0); s[6] = ag(F_GY, 0); s[7] = ag(F_VPREF, 0);
    s[8] = p.kinematics != CN_KIN_HOLONOMIC ? (float)theta[e] : 0.0f;
    s[9] = ag(F_PX, h + 1); s[10] = ag(F_PY, h + 1); s[11] = ag(F_VX, h + 1); s[12] = ag(F_VY, h + 1);
    s[13] = ag(F_R, h + 1);
    cn_rotate(s, o, p.kinematics);
    const double rx = st[st_idx(d, F_PX, 0, e)], ry = st[st_idx(d, F_PY, 0, e)];
    auto dist = [&](int k) { return norm2d(st[st_idx(d, F_PX, k + 1, e)] - rx, st[st_idx(d, F_PY, k + 1, e)] - ry); };
    auto rank = [&](int k) {                 // position of human k in the sorted order
        if (!sort_humans) return k;
        const double dh = dist(k);
        int r = 0;
        for (int j = 0; j < d.H; ++j)
            if (j != k) { const double dj = dist(j); r += (dj > dh || (dj == dh && j < k)) ? 1 : 0; }
        return r;
    };
    const int pos = rank(h);
    const int D = 13 + nd.om_dim;
    float *row = out + ((size_t)e * d.H + pos) * D;
    for (int k = 0; k < 13; ++k) row[k] = o[k];
    // with_om (multi_human_rl.py:98-101): map of the CURRENT human states around this human, the others visited in the order
    // of the human list the reference builds it from -- sorted for a sorted last_state (lstm_rl.py:99-105).  The order of the
    // float64 velocity sums can change a mean's float32 rounding.
    if (nd.om_dim > 0) {
        int ord[CN_MAX_HUMANS];
        for (int k = 0; k < d.H; ++k) ord[rank(k)] = k;
        occupancy_map_row(nd, d.H, pos, [&](int j, int f) {
            return st[st_idx(d, f == 0 ? F_PX : f == 1 ? F_PY : f == 2 ? F_VX : F_VY, ord[j] + 1, e)]; }, row + 13);
    }
}

// ValueNetwork.forward on a device batch (B x H x 13 -> B); grid = chunks of CA items
__global__ void __launch_bounds__(kThreads, 2)
forward_kernel(SarlWeightsDev W, SarlDims d, F32Plan pl, const float *__restrict__ x, int B, float *__restrict__ out)
{
    extern __shared__ __align__(16) float sm[];
    const int b0 = blockIdx.x * pl.CA;
    const int nb = min(pl.CA, B - b0);
    const int H = pl.H;
    float *X = sm + pl.oX;
    const int D = d.in;                                   // 13, or 13 + occupancy map
    for (int i = threadIdx.x; i < nb * H * D; i += blockDim.x) {
        const int r = i / D, k = i - r * D;
        X[(size_t)r * pl.wX + k] = x[(size_t)b0 * H * D + i];
    }
    __syncthreads();
    net_forward_smem(W, d, pl, sm, nb);
    const float *Vv = sm + pl.oV;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) out[b0 + i] = Vv[i];
}

F32Plan plan_for(const SarlDims &d, int H, int A, int A1, int CA)
{
    F32Plan pl;
    pl.H = H; pl.A = A;
    pl.CA = CA;
    const int rows = pl.CA * H;
    auto mx = [](int a, int b) { return a > b ? a : b; };
    pl.wX = d.in <= 16 ? 16 : pad4(d.in);          // 13 rotated features (+ occupancy map)
    pl.wT0 = pad4(mx(mx(d.m1[0], d.m2[0]), mx(mx(d.at[0], d.m3[0]), d.m3[2])));
    pl.wM1 = pad4(mx(mx(d.m1[1], d.at[1]), d.m3[1]));
    pl.wF = pad4(d.m2[1]);
    pl.wJ = pad4(d.self_dim + d.m2[1]);
    if (d.net == CN_NET_LSTM_RL) {          // gates (4h) in T0, h in G (ld wM1), c in F, joint = [self | h_n] in J
        pl.wT0 = pad4(mx(pl.wT0, mx(4 * d.lstm_h, mx(d.lm1[0], d.lm1[2]))));
        pl.wM1 = pad4(mx(pl.wM1, mx(d.lstm_h, mx(d.lm1[1], d.lm1[3]))));
        pl.wF = pad4(mx(pl.wF, d.lstm_h));
        pl.wJ = pad4(d.self_dim + mx(d.m2[1], d.lstm_h));
    }
    int o = 0;
    pl.oX = o; o += rows * pl.wX;
    pl.oT0 = o; o += rows * pl.wT0;
    pl.oM1 = o; o += rows * pl.wM1;
    pl.oF = o; o += rows * pl.wF;
    pl.oG = o; o += pl.CA * pl.wM1;
    pl.oJ = o; o += pl.CA * pl.wJ;
    pl.oS = o; o += pad4(rows);
    pl.oW = o; o += pad4(rows);
    pl.oV = o; o += pad4(pl.CA);
    o = (o + 3) & ~3;
    pl.oEnv = o; o += 2 * (A1 * F_COUNT + H * 4 + pl.CA);
    pl.oOrd = o; o += pad4(H);                      // LSTM-RL: humans in network order
    pl.oOm = o; o += pad4(H * d.om_dim);            // with_om: one map per human
    pl.total_floats = o;
    return pl;
}

// kRowsCap rows per CTA (CA actions or samples of H rows each); layers too wide for that many rows in shared memory get
// fewer actions per CTA, down to one.  A plan that still does not fit is refused by the caller.
F32Plan make_plan(const SarlDims &d, int H, int A, int A1)
{
    int ca = kRowsCap / H;
    if (ca < 1) ca = 1;
    if (ca > A) ca = A;
    F32Plan pl = plan_for(d, H, A, A1, ca);
    while (ca > 1 && sizeof(float) * (size_t)pl.total_floats > kMaxDynSmem) pl = plan_for(d, H, A, A1, --ca);
    return pl;
}

}  // namespace

int cn_lookahead_argmax(cn_policy *p, cn_env *env, double epsilon, cudaStream_t s, bool pdl)
{
    // pdl = false for pipelined shards (several handles sharing the SMs): plain launches
    return cn_launch(argmax_kernel, (env->p.d.E + 3) / 4, 128, 0, s, pdl, env->p, p->d.A, env->state, env->frozen, p->values,
                     p->action_dev, epsilon, env->step_ctr, env->action_xy, env->action_idx, p->bad_flag);
}

// cudaFuncSetAttribute applies to the CURRENT device only: called from cn_policy_create after cudaSetDevice, so that every
// device a policy handle lives on can launch the > 48 KB configurations (a process-wide "configured" flag would skip the
// second device).
int cn_f32_configure_device(void)
{
    CN_CUDA_CHECK(cudaFuncSetAttribute(lookahead_values_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDynSmem));
    CN_CUDA_CHECK(cudaFuncSetAttribute(forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDynSmem));
    return CN_OK;
}

int cn_lookahead_prepare(cn_policy *p, cn_env *env, cudaStream_t s)
{
    int rc = cn_grow(p->values, p->values_cap, env->p.d.E, sizeof(double) * p->d.A);
    if (rc) return rc;
    CN_CUDA_CHECK(cudaMemsetAsync(p->bad_flag, 0, sizeof(int32_t), s));
    return CN_OK;
}

int cn_lookahead_f32(cn_policy *p, cn_env *env, int query_env, double epsilon, cudaStream_t s)
{
    const EnvDims ed = env->p.d;
    if (ed.H > kRowsCap) { cn_set_error("FP32 lookahead supports human_num <= %d", kRowsCap); return CN_EUNSUPPORTED; }
    int rc = cn_lookahead_prepare(p, env, s);
    if (rc) return rc;
    const F32Plan pl = make_plan(p->d, ed.H, p->d.A, ed.A1);
    const size_t smem = sizeof(float) * (size_t)pl.total_floats;
    if (smem > kMaxDynSmem) { cn_set_error("FP32 lookahead needs %zu bytes of shared memory (layer widths too large)", smem); return CN_EUNSUPPORTED; }
    const double gamma_bar = pow(p->cfg.gamma, env->p.time_step * p->cfg.v_pref);
    dim3 grid(ed.E, (p->d.A + pl.CA - 1) / pl.CA);
    lookahead_values_kernel<<<grid, kThreads, smem, s>>>(env->p, p->w, p->d, pl, env->state, env->time, env->human_v,
                                                         env->frozen, p->action_dev, query_env, p->cfg.gamma, gamma_bar,
                                                         p->cfg.v_pref, p->values, env->theta);
    CN_LAUNCH_CHECK();
    return cn_lookahead_argmax(p, env, epsilon, s, true);
}

int cn_transform_f32(cn_policy *p, cn_env *env, float *out_dev, int sort_humans, cudaStream_t s)
{
    const int n = env->p.d.E * env->p.d.H;
    // the heading feature follows the POLICY's kinematics (cadrl.py:236-240), not the env's robot dynamics: in imitation
    // learning a holonomic ORCA robot drives the env while target_policy.transform() may be a unicycle SARL (explorer.py:163)
    EnvParams ep = env->p;
    ep.kinematics = p->cfg.kinematics;
    transform_kernel<<<(n + 127) / 128, 128, 0, s>>>(ep, p->d, env->state, env->theta, out_dev, sort_humans);
    CN_LAUNCH_CHECK();
    return CN_OK;
}

int cn_forward_f32(cn_policy *p, const float *x_dev, int batch, int H, float *out_dev, cudaStream_t s)
{
    if (H > kRowsCap || H < 1) { cn_set_error("forward supports 1 <= human_num <= %d", kRowsCap); return CN_EUNSUPPORTED; }
    if (batch <= 0) return CN_OK;
    const F32Plan pl = make_plan(p->d, H, batch, 1);
    const size_t smem = sizeof(float) * (size_t)pl.total_floats;
    if (smem > kMaxDynSmem) { cn_set_error("FP32 forward needs %zu bytes of shared memory (layer widths too large)", smem); return CN_EUNSUPPORTED; }
    forward_kernel<<<(batch + pl.CA - 1) / pl.CA, kThreads, smem, s>>>(p->w, p->d, pl, x_dev, batch, out_dev);
    CN_LAUNCH_CHECK();
    return CN_OK;
}
