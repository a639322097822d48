// tc_rows_pair.cuh -- the row network of the SARL lookahead on CTA PAIRS (tcgen05 cta_group::2).
// Included by lookahead_tc.cu inside its anonymous namespace (shares the padded shapes and the input helpers).
//
// Why pairs: with one CTA per SM the fp16 weights of the row network (157 KB) leave room for the activations
// of only ONE 128-row tile, so the tensor pipe idles during every epilogue (tc_rows_kernel: 21 % tensor-active).
// A cta_group::2 UMMA splits the B operand (the weights) in halves between the two SMs of a cluster, so each SM
// keeps 78.5 KB of weights and has room for TWO tile contexts (2 x 68 KB of activations, 2 x 224 TMEM columns).
// Per SM: 16 epilogue warps = 2 contexts x 2 column halves x 4 TMEM lane quarters (the epilogues are latency
// bound per warp, so every context gets 8 warps), and warp 16 of the rank-0 CTA issues every UMMA of the pair
// (M = 256 = tile of CTA 0 + tile of CTA 1 for the same context).
// Hand-over is pure dataflow through mbarriers, no CTA-wide barrier in the tile loop:
//   req[c]  (rank-0 CTA, 16 arrivals = 8 warps x 2 CTAs)  "operand of context c's next stage is in shared memory"
//   reqm[c] (same, for stage 3 only: stages 2 and 3 are requested without a completion wait in between, and
//            the two CTAs are not in lock step, so a shared barrier could see stage-3 arrivals in stage 2's phase)
//   done[c] (both CTAs, multicast tcgen05.commit)          "accumulator of context c's stage is complete"
//
// Per context and tile (rows = (env, action, human); D = TMEM columns relative to the context base):
//   stage  UMMA (M=256 over the pair)                         A operand        D          epilogue (CUDA cores)
//   0      mlp1.0                K=32   N=160                 X    (R1 tail)   [0,160)    ReLU -> H1, fp16 packed IN PLACE in TMEM
//   1      mlp1.2                K=160  N=112                 H1   (TMEM, TS)  [120,232)  ReLU -> mlp1_out (R2)
//   2      [attn.0a | mlp2.0]    K=112  N=224                 mlp1_out (R2)    [0,224)    group mean of mlp1_out in smem
//   3      attn.0b (mean half)   K=112  N=112, accumulate     mean (R1)        [0,112)    ReLU -> Ha1 fp16 IN PLACE in TMEM [0,56), H3 (R1)
//   4      attn.2 ; mlp2.2       K=112  N=112 ; N=64          Ha1 (TMEM, TS) ; H3 (R1)   [56,168) ; [168,232)
//          attention.4 as an fp32 dot -> masked softmax over the group -> w * F (fp32, smem) -> sum over the
//          humans of the group in shared memory -> joint state J (fp16) -> HBM
// The next tile's propagate / rotate features, clearances and rewards are computed under stages 2-3.
//
// GS = false ([sarl] with_global_state = false, sarl.py:40-47: attention.0 reads mlp1_out only) drops the group mean and
// stage 3, so a tile has FOUR stages and one cross-CTA hand-over less; the shared-memory and TMEM maps are the same:
//   stage  UMMA                                                A operand        D          epilogue
//   0, 1   as above
//   2      [attn.0 | mlp2.0]     K=112  N=224, own commit      mlp1_out (R2)    [0,224)    ReLU -> Ha1 fp16 IN PLACE in TMEM [0,56), H3 (R1)
//   3      attn.2 ; mlp2.2       as stage 4 above                                          as stage 4 above
// The number of completions per tile stays four (stage 2 commits itself instead of riding on stage 3's commit).
//
// Reference: crowd_nav/policy/sarl.py:28-65 (value network), cadrl.py:104-129,217-252 (propagate, rotate),
// multi_human_rl.py:65-88 / crowd_sim.py:344-403 (lookahead reward).

// Timing ablations (developer builds only, never in the shipped library; see scripts/row_kernel_ablation.sh and
// profiles/r02v_row_kernel_ablation*.txt): -DCN_ABLATE_EPI drops every epilogue's arithmetic and data movement (waits, barriers
// and hand-over signals stay), -DCN_ABLATE_MMA drops the UMMAs (commits stay).  The values are garbage; the kernel time is the
// point: hand-overs alone 0.164 ms, + UMMAs 0.456 ms, + epilogues instead 0.346 ms, everything 0.531 ms.
constexpr int kThreadsPair = 608;        // 16 epilogue warps (2 contexts x 2 column halves x 4 lane quarters) + issuer warp + 2 loader warps
constexpr int N_S2 = 2 * N_M1;             // stage 2: [mlp2.0 (rank-0 half) | attention.0 on mlp1_out (rank-1 half)]
constexpr int PAIR_CTX_COLS = 256;         // TMEM columns per tile context
constexpr int T_H1B = 80;                  // H1 as packed fp16 (TS-mode A operand): K 0..79 at [0,40), K 80..159 at [80,120)
constexpr int T_D1 = 120;                  // mlp1.2 accumulator [120,232)
constexpr int T_A2 = N_M1 / 2;             // attention.2 accumulator [56,168): right behind Ha1 packed in place at [0,56)
constexpr int T_F = T_A2 + N_M1;           // mlp2.2 accumulator (the pairwise features F) [168,232)

// per-CTA HALF weight image: rows [rank * N/2, (rank+1) * N/2) of every layer, chunked K-major with R = N/2
constexpr uint32_t H_W1 = 0;                                        //  80 x 32
constexpr uint32_t H_W2 = H_W1 + bytes_of(N_H1 / 2, K_X);           //  56 x 160
constexpr uint32_t H_W3A = H_W2 + bytes_of(N_M1 / 2, N_H1);         // 112 x 112  (rank 0: attention.0 first half, rank 1: mlp2.0)
constexpr uint32_t H_WB = H_W3A + bytes_of(N_M1, N_M1);             //  56 x 112  attention.0, group-mean half (GS only)
constexpr uint32_t H_W4 = H_WB + bytes_of(N_M1 / 2, N_M1);          //  32 x 112
constexpr uint32_t H_WA2 = H_W4 + bytes_of(N_F / 2, N_M1);          //  56 x 112
constexpr uint32_t H_TAIL = H_WA2 + bytes_of(N_M1 / 2, N_M1);       // fp32: attention.4 weight[100], bias
constexpr uint32_t IMG_H_BYTES = H_TAIL + TAIL_BYTES;

// shared-memory map of tc_rows_pair_kernel
constexpr uint32_t Q_R1_BYTES = bytes_of(ROWS, N_H1);               // 40 KB: H1 | mean, next X | H3 | w*F (fp32)
constexpr uint32_t Q_R2_BYTES = bytes_of(ROWS, N_M1);               // 28 KB: mlp1_out | Ha1
constexpr uint32_t Q_X_OFF = bytes_of(ROWS, N_M1);                  // next tile's X inside R1 (behind the 112-column tiles)
constexpr uint32_t Q_CTX_BYTES = Q_R1_BYTES + Q_R2_BYTES;
constexpr uint32_t Q_CTX0 = (IMG_H_BYTES + 127) & ~127u;
constexpr uint32_t Q_MISC = Q_CTX0 + 2 * Q_CTX_BYTES;               // S[2][2][128] f32 | D[2][128] f64 | 10 mbarriers | tmem slot
constexpr uint32_t Q_SMEM = Q_MISC + 2048 + 2048 + 96 + 16;
static_assert(Q_X_OFF + bytes_of(ROWS, K_X) <= Q_R1_BYTES, "next-tile X must fit behind the 112-column tiles");
static_assert(Q_SMEM <= 232448, "tc_rows_pair_kernel exceeds 227 KB of shared memory");

struct RowInPP {
    double rpx, rpy, rgx, rgy, rr, rvp, hpx, hpy, hvx, hvy, cvx, cvy, hr, ax, ay, t;
    float ntheta;          // robot heading after the action (cadrl.py:119), fp32 like the reference's state tensor
    int valid;
};

__device__ __forceinline__ void pp_load_inputs(RowInPP &in, const EnvDims &ed, const double *__restrict__ st,
                                               const double *__restrict__ time, const double *__restrict__ human_v,
                                               const double *__restrict__ actions, int A, int query_env, int NG, int G,
                                               int tile, int gl, int h, int kinematics, const double *__restrict__ theta)
{
    const int H = ed.H;
    const int g = tile * G + gl;          // the host keeps (total tiles + 1) * G below 2^31
    in.valid = (gl < G && g < NG) ? 1 : 0;
    if (!in.valid) return;
    const int e = A == 81 ? g / 81 : g / A, a = g - e * A;        // 81 = the holonomic action space: a multiply instead of a division
    // st[(field * A1 + agent) * E + env]: one base per agent, the field strides are uniform
    const size_t fs = (size_t)ed.A1 * ed.E;
    const double *__restrict__ pr = st + e, *__restrict__ ph = pr + (size_t)(h + 1) * ed.E;
    in.rpx = pr[F_PX * fs]; in.rpy = pr[F_PY * fs];
    in.rgx = pr[F_GX * fs]; in.rgy = pr[F_GY * fs];
    in.rr = pr[F_R * fs];   in.rvp = pr[F_VPREF * fs];
    in.hpx = ph[F_PX * fs]; in.hpy = ph[F_PY * fs];
    in.hr = ph[F_R * fs];
    in.cvx = ph[F_VX * fs]; in.cvy = ph[F_VY * fs];
    if (query_env) {                                                                    // agent.py:63-74
        in.hvx = human_v[(size_t)(0 * H + h) * ed.E + e]; in.hvy = human_v[(size_t)(1 * H + h) * ed.E + e];
        in.t = time[e];
    } else {                                                                            // cadrl.py:107-109
        in.hvx = in.cvx; in.hvy = in.cvy; in.t = 0.0;
    }
    // (ax, ay) = the velocity the robot moves with: the action itself (holonomic) or v (cos, sin)(theta + r)
    const double a0 = actions[2 * a], a1 = actions[2 * a + 1];
    const double th = kinematics != CN_KIN_HOLONOMIC ? theta[e] : 0.0;
    cn_effective_velocity(kinematics, th, a0, a1, in.ax, in.ay);
    in.ntheta = kinematics != CN_KIN_HOLONOMIC ? (float)(th + a1) : 0.0f;
}

// clearance of this row's human for the lookahead reward (see group_compute in lookahead_tc.cu for the equivalence with the
// reference's break-on-first-collision loops)
__device__ __forceinline__ double pp_clearance(const RowInPP &in, double dt, int query_env)
{
    if (!in.valid) return INFINITY;
    if (query_env) {   // crowd_sim.py:347-359
        const double px = in.hpx - in.rpx, py = in.hpy - in.rpy;
        const double vx = in.cvx - in.ax, vy = in.cvy - in.ay;
        const double ex = px + vx * dt, ey = py + vy * dt;
        return cn_point_to_segment_dist0(px, py, ex, ey) - in.hr - in.rr;
    }
    // multi_human_rl.py:69-70
    const double npx = in.rpx + in.ax * dt, npy = in.rpy + in.ay * dt;
    const double nhx = in.hpx + in.cvx * dt, nhy = in.hpy + in.cvy * dt;
    const double dx = npx - nhx, dy = npy - nhy;
    // The reward only asks "clearance < 0" and "min clearance < 0.2" (multi_human_rl.py:71-86): a row whose fp32 distance is
    // clear of that by a wide margin needs no float64 square root -- any value >= 0.2 gives the same reward.
    const float fx = (float)dx, fy = (float)dy, fr = (float)in.rr + (float)in.hr + 0.25f;
    if (fx * fx + fy * fy > fr * fr) return 1.0e30;
    return norm2d(dx, dy) - in.rr - in.hr;
}

// CADRL.rotate with the rotation taken from the normalised goal direction instead of atan2 -> sincos
// (cos(atan2(dy, dx)) = dx / |d|): same quantity to ~1e-7, a fraction of the instructions.  The FP32 twin keeps
// torch's atan2/cos/sin order (env_math.cuh); this path is fp16 downstream anyway.
__device__ __forceinline__ void rotate_dir(const float *s, float *o, int kinematics)
{
    const float dx = s[5] - s[0], dy = s[6] - s[1];
    const float d = sqrtf(dx * dx + dy * dy);
    float c = 1.0f, sn = 0.0f;
    if (d > 0.0f) { const float inv = 1.0f / d; c = dx * inv; sn = dy * inv; }
    o[0] = d;
    o[1] = s[7];
    o[2] = kinematics == CN_KIN_UNICYCLE ? s[8] - atan2f(dy, dx) : 0.0f;      // cadrl.py:236-240
    o[3] = s[4];
    o[4] = s[2] * c + s[3] * sn;
    o[5] = s[3] * c - s[2] * sn;
    o[6] = (s[9] - s[0]) * c + (s[10] - s[1]) * sn;
    o[7] = (s[10] - s[1]) * c - (s[9] - s[0]) * sn;
    o[8] = s[11] * c + s[12] * sn;
    o[9] = s[12] * c - s[11] * sn;
    o[10] = s[13];
    const float ax = s[0] - s[9], ay = s[1] - s[10];
    o[11] = sqrtf(ax * ax + ay * ay);
    o[12] = s[4] + s[13];
}

__device__ __forceinline__ void pair_features(const RowInPP &in, double dt, int kinematics, uint4 &c0, uint4 &c1, uint4 &c2,
                                              uint4 &c3)
{
    c0 = make_uint4(0, 0, 0, 0); c1 = c0; c2 = c0; c3 = c0;
    if (!in.valid) return;
    float s[14], o[13];
    s[0] = (float)(in.rpx + in.ax * dt); s[1] = (float)(in.rpy + in.ay * dt);
    s[2] = (float)in.ax; s[3] = (float)in.ay; s[4] = (float)in.rr;
    s[5] = (float)in.rgx; s[6] = (float)in.rgy; s[7] = (float)in.rvp; s[8] = in.ntheta;
    s[9] = (float)(in.hpx + in.hvx * dt); s[10] = (float)(in.hpy + in.hvy * dt);
    s[11] = (float)in.hvx; s[12] = (float)in.hvy; s[13] = (float)in.hr;
    rotate_dir(s, o, kinematics);
    float hi[13], lo[13];
#pragma unroll
    for (int k = 0; k < 13; ++k) split_hl(o[k], hi[k], lo[k]);
    c0 = make_uint4(h2(hi[0], hi[1]), h2(hi[2], hi[3]), h2(hi[4], hi[5]), h2(hi[6], hi[7]));
    c1 = make_uint4(h2(hi[8], hi[9]), h2(hi[10], hi[11]), h2(hi[12], 1.0f), h2(1.0f, 0.0f));
    c2 = make_uint4(h2(lo[0], lo[1]), h2(lo[2], lo[3]), h2(lo[4], lo[5]), h2(lo[6], lo[7]));
    c3 = make_uint4(h2(lo[8], lo[9]), h2(lo[10], lo[11]), h2(lo[12], 0.0f), 0u);
}

// lookahead reward of one (env, action) group from the H clearances in D (see group_compute in lookahead_tc.cu for the equivalence
// with the reference's break-on-first-collision loops)
__device__ __forceinline__ double pair_reward(const EnvParams &p, const RowInPP &in, const double *__restrict__ D, int H,
                                              int query_env)
{
    const double dt = p.time_step;
    double dmin = INFINITY;
    bool collision = false;
    for (int k = 0; k < H; ++k) {
        const double c = D[k];
        if (c < 0) collision = true;
        else if (c < dmin) dmin = c;
    }
    const double npx = in.rpx + in.ax * dt, npy = in.rpy + in.ay * dt;
    const bool reaching_goal = norm2d(npx - in.rgx, npy - in.rgy) < in.rr;
    if (query_env) {                                                                 // crowd_sim.py:382-403
        if (in.t >= p.time_limit - 1) return 0;
        if (collision) return p.collision_penalty;
        if (reaching_goal) return p.success_reward;
        if (dmin < p.discomfort_dist) return (dmin - p.discomfort_dist) * p.discomfort_penalty_factor * dt;
        return 0;
    }
    if (collision) return -0.25;                                                     // multi_human_rl.py:77-86
    if (reaching_goal) return 1;
    if (dmin < 0.2) return (dmin - 0.2) * 0.5 * dt;
    return 0;
}


struct TailW { float w[104]; };   // attention.4: weight[100], bias at [100]; passed by value (constant bank operands)

constexpr uint32_t X_TILE_BYTES = bytes_of(ROWS, K_X);   // 8 KB: one tile of the layer-1 operand, already in UMMA order

// Feature kernel: everything a row tile needs before its stage 0, for ALL tiles of the lookahead at once (one block
// per tile, one thread per row): propagate + rotate -> X operand tile in HBM (consumed through TMA bulk copies by
// tc_rows_pair_kernel), self-state chunks of J, lookahead rewards.  3.3 M rows of independent work: the massively
// parallel form this needs -- inside the row kernel it sat on a few latency-bound warps (measured 4.6-7 k cycles
// per tile against a 6-8 k cycle tile budget; three dedicated producer warps per CTA, re-measured with the final
// kernel: 8.8e6 vs 1.07e7 env-steps/s).  Costs one 64 B / row round trip through L2 / HBM.
template <int HT>
__global__ void __launch_bounds__(ROWS, 9)
tc_features_kernel(EnvParams p, const double *__restrict__ st, const double *__restrict__ time,
                   const double *__restrict__ human_v, const double *__restrict__ actions, int A, int query_env, int NG,
                   int G_rt, const double *__restrict__ theta, uint8_t *__restrict__ X, uint8_t *__restrict__ J,
                   double *__restrict__ rew)
{
    __shared__ double D[ROWS];
    pdl_launch_dependents();               // the row kernel's CTAs may take the SMs this grid frees (they wait before reading X)
    const EnvDims ed = p.d;
    const int H = HT ? HT : ed.H;
    const int G = HT ? ROWS / HT : G_rt;
    const int tile = blockIdx.x, r = threadIdx.x;
    const int gl = r / H, h = r - gl * H;
    const double dt = p.time_step;
    RowInPP in;
    pp_load_inputs(in, ed, st, time, human_v, actions, A, query_env, NG, G, tile, gl, h, p.kinematics, theta);
    D[r] = pp_clearance(in, dt, query_env);
    uint4 c0, c1, c2, c3;
    pair_features(in, dt, p.kinematics, c0, c1, c2, c3);
    uint8_t *xt = X + (size_t)tile * X_TILE_BYTES;
    *reinterpret_cast<uint4 *>(xt + chunk_off(ROWS, r, 0)) = c0;
    *reinterpret_cast<uint4 *>(xt + chunk_off(ROWS, r, 1)) = c1;
    *reinterpret_cast<uint4 *>(xt + chunk_off(ROWS, r, 2)) = c2;
    *reinterpret_cast<uint4 *>(xt + chunk_off(ROWS, r, 3)) = c3;
    const bool lead = in.valid && h == 0;
    const int g = tile * G + gl;
    if (lead) {
        // c0 = hi[0..7], c2 = lo[0..7]: the self state is columns 0..5 of the rotated row (sarl.py:36)
        uint8_t *jt = J + (size_t)(g >> 7) * J_TILE_BYTES;
        const int rb = g & 127;
        *reinterpret_cast<uint4 *>(jt + chunk_off(ROWS, rb, 7)) = make_uint4(c0.x, c0.y, c0.z, h2(1.0f, 1.0f));
        *reinterpret_cast<uint4 *>(jt + chunk_off(ROWS, rb, 8)) = make_uint4(c2.x, c2.y, c2.z, 0u);
        *reinterpret_cast<uint4 *>(jt + chunk_off(ROWS, rb, 9)) = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    // the G rewards of the tile by its first G threads (whole warps instead of every H-th lane of every warp)
    if (r < G && tile * G + r < NG) {
        RowInPP in0;
        pp_load_inputs(in0, ed, st, time, human_v, actions, A, query_env, NG, G, tile, r, 0, p.kinematics, theta);
        rew[tile * G + r] = pair_reward(p, in0, D + r * H, H, query_env);
    }
}

// acc[8] += sum over n 16-byte chunks of 8 fp16 at base + i * stride.  Loads go out four at a time before anything is added:
// under a streaming UMMA one ld.shared round trip costs ~150-250 cycles (measured), so dependent one-at-a-time loops crawl.
__device__ __forceinline__ void sum_f16x8_rows(const uint8_t *base, int n, uint32_t stride, float (&acc)[8])
{
    for (int i0 = 0; i0 < n; i0 += 4) {
        uint4 u[4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
            u[j] = (i0 + j < n) ? *reinterpret_cast<const uint4 *>(base + (size_t)(i0 + j) * stride) : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const __half2 *hv = reinterpret_cast<const __half2 *>(&u[j]);
#pragma unroll
            for (int k = 0; k < 4; ++k) { const float2 f = __half22float2(hv[k]); acc[2 * k] += f.x; acc[2 * k + 1] += f.y; }
        }
    }
}

__device__ __forceinline__ void ctx_barrier(int ctx)
{
    if (ctx == 0) asm volatile("bar.sync 1, 256;" ::: "memory");
    else asm volatile("bar.sync 2, 256;" ::: "memory");
}

// HT = compile-time human count (5, 10: the benchmark configurations) or 0 = run-time H
// OM = occupancy maps (multi_human_rl.py:109-163): the map of a human does not depend on the robot's action, so its product
// with mlp1.0's map columns is one fp32 row bias per (env, human) (omP, from tc_om_bias_kernel), added in the E0 epilogue
// GS = the global state: attention.0 on [mlp1_out | group mean] (five stages per tile), or on mlp1_out alone (four stages)
template <int HT, bool OM, bool GS>
// __maxnreg__(88), not __launch_bounds__ (the two exclude each other): see cn_small_block() in cn_common.cuh -- 88 registers
// leave room for one <= 72-register warp of another shard's small kernels in every SM sub-partition; no measurable cost here.
__global__ void __cluster_dims__(2, 1, 1) __maxnreg__(88)
tc_rows_pair_kernel(EnvParams p,
                    const uint8_t *__restrict__ wimg, const uint8_t *__restrict__ X, uint8_t *__restrict__ J, int NG, int G_rt,
                    int rounds, const TailW tw, long long *__restrict__ dbg, const float *__restrict__ omP, int A)
{
#define QPROBE(slot, i) do { if (dbg && blockIdx.x < 2 && probe_round) dbg[(blockIdx.x * 4 + (slot)) * 32 + (i)] = clock64(); } while (0)
    extern __shared__ __align__(128) uint8_t smem[];
    const EnvDims ed = p.d;
    const int H = HT ? HT : ed.H;
    const int G = HT ? ROWS / HT : G_rt;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool is_issuer_warp = warp == 16, is_producer_warp = warp > 16;
    const int q = warp & 3, ctx = (warp >> 2) & 1, hf = (warp >> 3) & 1;     // lane quarter, tile context, column half
    const uint32_t rank = cluster_ctarank();
    const int cluster_id = blockIdx.x >> 1, nclusters = gridDim.x >> 1;
    const int row = q * 32 + lane;                  // tile row == TMEM lane of this thread
    const int t256 = hf * 128 + row;                // thread index within the context
    const int my_gl = row / H, my_h = row - my_gl * H;
    const int rows = G * H;
    uint8_t *R1 = smem + Q_CTX0 + (uint32_t)ctx * Q_CTX_BYTES, *R2 = R1 + Q_R1_BYTES;
    float *S0 = reinterpret_cast<float *>(smem + Q_MISC) + ctx * 256, *S1 = S0 + 128;   // partial scores of the column halves
    const uint32_t bar0 = smem_u32(smem + Q_MISC + 4096);
    const uint32_t req0 = bar0, req1 = bar0 + 8, done0 = bar0 + 16, done1 = bar0 + 24, reqm0 = bar0 + 32, reqm1 = bar0 + 40;
    const uint32_t xfull0 = bar0 + 48, xfull1 = bar0 + 56;     // rank-0 CTA: X of the context's next tile has landed in both CTAs
    const uint32_t xland0 = bar0 + 80, xland1 = bar0 + 88;     // per CTA: TMA transaction barrier of the X slot
    const uint32_t xfree0 = bar0 + 64, xfree1 = bar0 + 72;     // per CTA: stage 0 of the context's tile is complete -> the X slot may be rewritten
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + Q_MISC + 4096 + 96);

    copy_image_to_smem(smem, wimg + (size_t)rank * IMG_H_BYTES, IMG_H_BYTES);
    for (uint32_t i = tid * 16; i < 2 * Q_CTX_BYTES; i += kThreadsPair * 16)       // padding rows stay finite
        *reinterpret_cast<uint4 *>(smem + Q_CTX0 + i) = make_uint4(0, 0, 0, 0);
    if (tid == 0) {
        mbar_init(req0, 16); mbar_init(req1, 16); mbar_init(done0, 1); mbar_init(done1, 1);
        mbar_init(reqm0, 16); mbar_init(reqm1, 16);
        mbar_init(xfull0, 2); mbar_init(xfull1, 2); mbar_init(xfree0, 1); mbar_init(xfree1, 1);
        mbar_init(xland0, 1); mbar_init(xland1, 1);
        fence_mbar_init();
    }
    if (warp == 0) tmem_alloc_2(smem_u32(tmem_slot), 512);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    cluster_sync_all();
    fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    pdl_launch_dependents();               // mlp3's CTAs may be placed as this grid's CTAs exit
    pdl_wait();                            // everything above overlapped the feature kernel's tail; X / J / rewards are complete from here

    if (is_issuer_warp) {
        // ================= issuer warp (rank-0 CTA only) =================
        // ONE issuing thread polls both contexts.  (Two issuer warps, one blocking per context, were measured: the
        // contexts then run in lock step, contend for the same resources at the same time, and the kernel is 3 % slower.)
        if (rank == 0 && lane == 0) {
            const uint32_t sW1 = smem_u32(smem + H_W1), sW2 = smem_u32(smem + H_W2), sW3A = smem_u32(smem + H_W3A);
            const uint32_t sWB = smem_u32(smem + H_WB), sW4 = smem_u32(smem + H_W4), sWA2 = smem_u32(smem + H_WA2);
            constexpr int NS = GS ? 5 : 4;                  // UMMA stages per tile
            const int total = NS * rounds;
            int stage0 = 0, stage1 = 0;
            uint32_t ph0 = 0, ph1 = 0, phm0 = 0, phm1 = 0, phx0 = 0, phx1 = 0;
            uint32_t idle_polls = 0;
            while (stage0 < total || stage1 < total) {
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    int &stage = c ? stage1 : stage0;
                    if (stage >= total) continue;
                    const int s = stage % NS;
                    uint32_t &ph = (GS && s == 3) ? (c ? phm1 : phm0) : (c ? ph1 : ph0);
                    if (!mbar_test_wait_cluster((GS && s == 3) ? (c ? reqm1 : reqm0) : (c ? req1 : req0), ph)) continue;
                    if (s == 0) {                                   // stage 0 also needs the TMA-landed X of both CTAs
                        uint32_t &phx = c ? phx1 : phx0;
                        if (!mbar_test_wait_cluster(c ? xfull1 : xfull0, phx)) continue;
                        phx ^= 1;
                    }
                    ph ^= 1;
                    const bool probe_round = stage / NS == 3;
                    QPROBE(2 + c, 2 * s);
                    fence_after_sync();
                    const uint32_t tm = tmem + (uint32_t)c * PAIR_CTX_COLS;
                    const uint32_t sR1 = smem_u32(smem + Q_CTX0 + (uint32_t)c * Q_CTX_BYTES), sR2 = sR1 + Q_R1_BYTES;
                    const uint32_t done = c ? done1 : done0;
#ifdef CN_ABLATE_MMA
                    if (!GS || s != 2) commit_2(done, 3);
                    if (1) {
                    } else if (s == 0) {
#else
                    if (s == 0) {
#endif
                        mma_layer_2(tm, sR1 + Q_X_OFF, ROWS, sW1, K_X, N_H1, false);
                        commit_2(done, 3);
                    } else if (s == 1) {
                        // A = H1 straight from TMEM (two packed halves, written in place by the two column-half warps)
                        mma_steps_2_ts(tm + T_D1, tm, sW2, 0, N_H1 / 32, N_M1, false);
                        mma_steps_2_ts(tm + T_D1, tm + T_H1B, sW2, N_H1 / 32, N_H1 / 16, N_M1, true);
                        commit_2(done, 3);
                    } else if (s == 2) {
                        mma_layer_2(tm, sR2, ROWS, sW3A, N_M1, N_S2, false);          // GS: completion rides on stage 3's commit
                        if constexpr (!GS) commit_2(done, 3);
                    } else if (GS && s == 3) {
                        mma_layer_2(tm, sR1, ROWS, sWB, N_M1, N_M1, true);             // attention.0 accumulator = [0,112)
                        commit_2(done, 3);
                    } else {
                        // A of attention.2 = Ha1 straight from TMEM (packed in place by the hf-0 warps)
                        mma_steps_2_ts(tm + T_A2, tm, sWA2, 0, N_M1 / 16, N_M1, false);
                        mma_layer_2(tm + T_F, sR1, ROWS, sW4, N_M1, N_F, false);
                        commit_2(done, 3);
                    }
                    QPROBE(2 + c, 2 * s + 1);
                    ++stage;
                    idle_polls = 0;
                }
                // protocol bug guard: never hang the GPU.  (Counted in polls, not clock64() reads: the poll loop IS the hand-over
                // latency of every stage.  A __nanosleep here was measured and costs 1.5 % at 20 ns, 2.5 % at 100 ns.)
                if (++idle_polls > (1u << 28)) __trap();
            }
        }
    } else if (is_producer_warp) {
        // ================= loader warps (both CTAs): warp 17 + c streams context c's X tiles from HBM by TMA bulk copy =================
        if (lane == 0) {
            const int c = warp - 17;
            const uint32_t xl = c ? xland1 : xland0, xfree = c ? xfree1 : xfree0;
            const uint32_t xfull_leader = mapa(c ? xfull1 : xfull0, 0);
            const uint32_t dst = smem_u32(smem + Q_CTX0 + (uint32_t)c * Q_CTX_BYTES + Q_X_OFF);
            const int tile_stride = 4 * nclusters;
            int tile = (cluster_id * 2 + (int)rank) * 2 + c;
            uint32_t phf = 0, phl = 0;
            for (int rnd = 0; rnd < rounds; ++rnd, tile += tile_stride) {
                if (rnd > 0) { mbar_wait_guarded(xfree, phf); phf ^= 1; }              // stage 0 of the previous tile is complete
                bulk_load(dst, X + (size_t)tile * X_TILE_BYTES, X_TILE_BYTES, xl);
                mbar_wait_guarded(xl, phl); phl ^= 1;                                   // the tile has landed in this CTA
                mbar_arrive_cluster(xfull_leader);
            }
        }
    } else {
        // ================= epilogue warps: context `ctx`, column half `hf` (both CTAs) =================
        const uint32_t done = ctx ? done1 : done0;
        const uint32_t req_leader = mapa(ctx ? req1 : req0, 0), reqm_leader = mapa(ctx ? reqm1 : reqm0, 0);
        const uint32_t tl = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)ctx * PAIR_CTX_COLS;
        uint32_t ph = 0;
        const float invH = 1.0f / (float)H;
        const int tile_stride = 4 * nclusters;
        int tile = (cluster_id * 2 + (int)rank) * 2 + ctx;
        // loop-invariant work items of the two shared-memory group reductions (consecutive threads -> consecutive groups)
        // (HT: at most 2 mean items and 1 sum item per thread, decomposed once; run-time H: any count, decomposed in the loop)
        constexpr int kMeanIters = HT ? 2 : 4;      // G <= 64 -> at most 896 mean items / 256 threads
        int mean_off[kMeanIters];
#pragma unroll
        for (int i = 0; i < kMeanIters; ++i) {
            const int it = t256 + i * 256;
            const int c = it / G, gl = it - c * G;
            mean_off[i] = (it < G * (N_M1 / 8)) ? (int)chunk_off(ROWS, gl * H, c) : -1;
        }
        constexpr int kSumIters = HT ? 1 : 2;       // at most 448 sum items / 256 threads
        // Run-time H with FEW, LARGE groups (H = 50: 2 groups of 50 rows): one thread per (group, chunk) item would leave 28
        // threads walking 50 rows each (measured: 5.5 k cycles for the mean, 3.3 k for the sums, of a 20 k cycle tile).  The
        // rows of a group are then split over P threads per item so that (nearly) all 256 threads of the context work.
        // P = a power of two, so that the P threads of an item are adjacent lanes of one warp: they take the rows h = seg,
        // seg + P, ... (adjacent lanes -> adjacent 16-byte rows: conflict-free) and combine their partial sums by shuffles.
        auto pow2_floor = [](int x) { int p = 1; while (2 * p <= x && p < 16) p *= 2; return p; };
        const int mean_split = HT ? 1 : pow2_floor(256 / (G * (N_M1 / 8)));   // 8 for G = 2 (H = 50), >= 2 <=> G <= 9 <=> H >= 13
        const int sum_split = HT ? 1 : pow2_floor(256 / (G * 7));             // 16 for G = 2, >= 2 <=> G <= 18 <=> H >= 8
        uint8_t *mean_scratch = R1 + Q_X_OFF + X_TILE_BYTES;        // the 4 KB of R1 behind the X slot (softmax scratch)
        static_assert(Q_X_OFF + X_TILE_BYTES + 2 * ROWS * 4 <= Q_R1_BYTES, "softmax scratch must fit behind the X slot");
        // operand hand-over: generic-proxy writes -> async proxy, TMEM reads ordered, one arrival per warp
#define PAIR_SIGNAL_TO(bar) do { fence_async_smem(); fence_before_sync(); __syncwarp(); if (lane == 0) mbar_arrive_cluster(bar); } while (0)
#define PAIR_SIGNAL() PAIR_SIGNAL_TO(req_leader)
#define PAIR_WAIT() do { mbar_wait_guarded(done, ph); ph ^= 1; fence_after_sync(); } while (0)
        // OM: the 320 bytes of this thread's row bias are pulled into L1 one tile ahead (the loads in E0 sit on the tile's critical
        // path; from L2 they cost +56 % on the kernel, measured)
        auto om_prefetch = [&](int tl_idx) {
            const long long g2 = (long long)tl_idx * G + my_gl;
            if (row < rows && g2 < NG) {
                const float *b = omP + ((size_t)(g2 / A) * H + my_h) * N_H1 + hf * 80;
                asm volatile("prefetch.global.L1 [%0];" :: "l"(b));
                asm volatile("prefetch.global.L1 [%0];" :: "l"(b + 32));
                asm volatile("prefetch.global.L1 [%0];" :: "l"(b + 64));
            }
        };
        if constexpr (OM) om_prefetch(tile);
        PAIR_SIGNAL();                                                             // stage 0 of the first tile
        for (int rnd = 0; rnd < rounds; ++rnd, tile += tile_stride) {
            const bool has_next = rnd + 1 < rounds;
            const bool probe_round = (t256 == 0) && rnd == 3;
            const long long g = (long long)tile * G + my_gl;
            const bool row_valid = (row < rows) && (g < NG);
            QPROBE(ctx, 0);
            // ---- stage 0 was requested at the end of the previous tile (before its group sums) / before the loop ----
            // ---- E0: H1 = relu(acc[0,160)) -> R1 ----
            PAIR_WAIT(); QPROBE(ctx, 1);
            if (warp == 4 * ctx && lane == 0) mbar_arrive(ctx ? xfree1 : xfree0);      // stage 0 is complete (H1 lives in TMEM): the X slot may be refilled
            if constexpr (OM) {
                const float *bias = row_valid ? omP + ((size_t)(g / A) * H + my_h) * N_H1 + hf * 80 : nullptr;
                compact_to_tmem_bias(tl, hf * 80, 80, hf * T_H1B, bias);
            } else
#ifndef CN_ABLATE_EPI
            compact_to_tmem<true, true>(tl, hf * 80, 80, hf * T_H1B, 1.0f);        // in place: no shared-memory traffic for H1
#endif
            PAIR_SIGNAL(); QPROBE(ctx, 2);
            if constexpr (OM) { if (has_next) om_prefetch(tile + tile_stride); }
            // ---- E1: mlp1_out = relu(acc[0,112)) -> R2 ----
            PAIR_WAIT(); QPROBE(ctx, 3);
#ifndef CN_ABLATE_EPI
            if (hf == 0) epilogue_to_smem<true>(tl, T_D1, 64, R2, row, 0);
            else epilogue_to_smem<true>(tl, T_D1 + 64, 48, R2, row, 8);
#endif
            PAIR_SIGNAL(); QPROBE(ctx, 4);                                         // stage 2 may start
            if constexpr (GS) {
                QPROBE(ctx, 12);
                // ---- group mean of mlp1_out over the humans of a group (sarl.py:42), replicated on the group's rows -> R1 ----
                ctx_barrier(ctx);
                QPROBE(ctx, 13);
#ifdef CN_ABLATE_EPI
                if (0) {
#else
                if (!HT && mean_split >= 2) {
#endif
                    const int P = mean_split, nitems = G * (N_M1 / 8);
                    const int it = t256 / P, seg = t256 & (P - 1);
                    const bool on = it < nitems;
                    const int c = on ? it / G : 0, gl = on ? it - c * G : 0;
                    const int n = on ? (H - seg + P - 1) / P : 0;                    // rows seg, seg + P, ... of the group
                    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                    sum_f16x8_rows(R2 + chunk_off(ROWS, gl * H + seg, c), n, 16u * P, acc);
                    for (int off = 1; off < P; off <<= 1)                                // whole warps take part (it may be off)
#pragma unroll
                        for (int k = 0; k < 8; ++k) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], off);
                    const uint4 o = make_uint4(h2(acc[0] * invH, acc[1] * invH), h2(acc[2] * invH, acc[3] * invH),
                                               h2(acc[4] * invH, acc[5] * invH), h2(acc[6] * invH, acc[7] * invH));
                    for (int h = seg; h < H && on; h += P)                               // replicate on the same rows
                        *reinterpret_cast<uint4 *>(R1 + chunk_off(ROWS, gl * H + h, c)) = o;
                } else
#pragma unroll
                for (int i = 0; i < kMeanIters; ++i) {
#ifdef CN_ABLATE_EPI
                    break;
#endif
                    if (mean_off[i] < 0) continue;
                    const uint8_t *src = R2 + mean_off[i];
                    uint4 v[HT ? HT : 1];
                    __half2 acc[4];
                    if (HT) {
#pragma unroll
                        for (int h = 0; h < HT; ++h) v[h] = *reinterpret_cast<const uint4 *>(src + h * 16);
                        const __half2 *h0 = reinterpret_cast<const __half2 *>(&v[0]);
                        acc[0] = h0[0]; acc[1] = h0[1]; acc[2] = h0[2]; acc[3] = h0[3];
#pragma unroll
                        for (int h = 1; h < HT; ++h) {
                            const __half2 *hv = reinterpret_cast<const __half2 *>(&v[h]);
#pragma unroll
                            for (int k = 0; k < 4; ++k) acc[k] = __hadd2(acc[k], hv[k]);
                        }
                    } else {
                        v[0] = *reinterpret_cast<const uint4 *>(src);
                        const __half2 *h0 = reinterpret_cast<const __half2 *>(&v[0]);
                        acc[0] = h0[0]; acc[1] = h0[1]; acc[2] = h0[2]; acc[3] = h0[3];
                        for (int h = 1; h < H; ++h) {
                            const uint4 u = *reinterpret_cast<const uint4 *>(src + h * 16);
                            const __half2 *hv = reinterpret_cast<const __half2 *>(&u);
#pragma unroll
                            for (int k = 0; k < 4; ++k) acc[k] = __hadd2(acc[k], hv[k]);
                        }
                    }
                    uint4 o;
                    {
                        const float2 f0 = __half22float2(acc[0]), f1 = __half22float2(acc[1]);
                        const float2 f2 = __half22float2(acc[2]), f3 = __half22float2(acc[3]);
                        o.x = h2(f0.x * invH, f0.y * invH); o.y = h2(f1.x * invH, f1.y * invH);
                        o.z = h2(f2.x * invH, f2.y * invH); o.w = h2(f3.x * invH, f3.y * invH);
                    }
                    uint8_t *dst = R1 + mean_off[i];
                    if (HT) {
#pragma unroll
                        for (int h = 0; h < HT; ++h) *reinterpret_cast<uint4 *>(dst + h * 16) = o;
                    } else {
                        for (int h = 0; h < H; ++h) *reinterpret_cast<uint4 *>(dst + h * 16) = o;
                    }
                }
                QPROBE(ctx, 14);
                PAIR_SIGNAL_TO(reqm_leader); QPROBE(ctx, 5);
                if (dbg && blockIdx.x < 2 && rnd == 3 && ctx == 0 && lane == 0) dbg[192 + blockIdx.x * 8 + hf * 4 + q] = clock64();                           // stage 3 may start
            }
            QPROBE(ctx, 6);
            // ---- E3: Ha1 = relu(acc[0,112)) fp16 in place in TMEM (hf 0) ; H3 = relu(acc[112,224)) -> R1 (hf 1) ----
            // (GS: after stage 3, whose commit covers stage 2; otherwise after stage 2's own commit)
            PAIR_WAIT(); QPROBE(ctx, 7);
#ifndef CN_ABLATE_EPI
            if (hf == 0) compact_to_tmem<true, true>(tl, 0, N_M1, 0, 1.0f);         // Ha1: fp16 pairs in place, [0,56)
            else epilogue_to_smem<true>(tl, N_M1, N_M1, R1, row, 0);
#endif
            PAIR_SIGNAL(); QPROBE(ctx, 8);
            // ---- E4: attention.4 dot (split over the column halves), masked softmax (sarl.py:48-53), w * F ----
            PAIR_WAIT(); QPROBE(ctx, 9);
#ifdef CN_ABLATE_EPI
            if (has_next) PAIR_SIGNAL();
            ctx_barrier(ctx);
            QPROBE(ctx, 11);
            continue;
#endif
            {
                float part = 0.0f;
                if (hf == 0) {
                    uint32_t v[32];
                    ld32(tl + T_A2, v);
                    wait_ld();
#pragma unroll
                    for (int k = 0; k < 32; ++k) part = fmaf(fmaxf(__uint_as_float(v[k]), 0.0f), tw.w[k], part);
                    ld32(tl + T_A2 + 32, v);
                    wait_ld();
#pragma unroll
                    for (int k = 0; k < 32; ++k) part = fmaf(fmaxf(__uint_as_float(v[k]), 0.0f), tw.w[32 + k], part);
                    S0[row] = part;
                } else {
                    uint32_t x[32], y[16];
                    ld32(tl + T_A2 + 64, x);
                    wait_ld();
#pragma unroll
                    for (int k = 0; k < 32; ++k) part = fmaf(fmaxf(__uint_as_float(x[k]), 0.0f), tw.w[64 + k], part);
                    ld16(tl + T_A2 + 96, y);
                    wait_ld();
#pragma unroll
                    for (int k = 0; k < 4; ++k) part = fmaf(fmaxf(__uint_as_float(y[k]), 0.0f), tw.w[96 + k], part);
                    S1[row] = part;
                }
            }
            QPROBE(ctx, 15);
            // Every TMEM read of [0,168) of this tile is done (Ha1 was consumed by the stage-4 UMMA, the attention.2 accumulator
            // by the loads above); F at [168,232) is still live but stage 0 only writes [0,160): request the next tile's stage 0
            // NOW, so that its UMMA runs under the softmax / w * F / group sums below.  (Stage 1 writes [120,232) and is only
            // requested after the next E0, i.e. after every warp has finished this tile.)
            if (has_next) PAIR_SIGNAL();
            // the pairwise features F of this thread's row: the load stays in flight across the barrier and the softmax
            // (a tcgen05.ld + wait round trip is ~290 cycles of this, the longest, epilogue)
            uint32_t fv[32];
            ld32(tl + T_F + hf * 32, fv);
            ctx_barrier(ctx);
            QPROBE(ctx, 16);
            float w = 0.0f;
            if (!HT && H >= 8) {
                // large groups: one exp per row instead of H per row -- every thread exponentiates its own row's score into SE
                // (both column-half threads of a row write the same value), then sums its group's H entries
                float *SE = reinterpret_cast<float *>(mean_scratch);              // 128 floats of the (idle) mean scratch
                float mine = 0.0f;
                if (row_valid) {
                    const float sc = S0[row] + S1[row] + tw.w[100];
                    mine = __expf(sc) * (sc != 0.0f ? 1.0f : 0.0f);
                    SE[row] = mine;
                }
                ctx_barrier(ctx);
                float *SP = SE + ROWS;                                            // partial sums of 8 consecutive rows of a group
                if (row_valid && (my_h & 7) == 0) {
                    float p8 = 0.0f;
#pragma unroll
                    for (int k = 0; k < 8; ++k) p8 += (my_h + k < H) ? SE[row + k] : 0.0f;
                    SP[row] = p8;
                }
                ctx_barrier(ctx);
                if (row_valid) {
                    float ssum = 0.0f;
                    const int r0 = my_gl * H;
                    for (int h = 0; h < H; h += 8) ssum += SP[r0 + h];
                    w = mine / ssum;
                }
            } else if (row_valid) {
                float ssum = 0.0f, mine = 0.0f;
                const int r0 = my_gl * H;
                if (HT) {
#pragma unroll
                    for (int h = 0; h < HT; ++h) {
                        const float sc = S0[r0 + h] + S1[r0 + h] + tw.w[100];
                        const float se = __expf(sc) * (sc != 0.0f ? 1.0f : 0.0f);
                        ssum += se;
                        if (h == my_h) mine = se;
                    }
                } else {
                    for (int h = 0; h < H; ++h) {
                        const float sc = S0[r0 + h] + S1[r0 + h] + tw.w[100];
                        const float se = __expf(sc) * (sc != 0.0f ? 1.0f : 0.0f);
                        ssum += se;
                        if (h == my_h) mine = se;
                    }
                }
                w = mine / ssum;
            }
            {
                // w * F as fp16 (fp32 product rounded once), chunked like an operand over the (dead) Ha1 tile in R2 -- not R1:
                // the next tile's H1 epilogue may start while slower warps still sum: hf 0 -> features 0..31, hf 1 -> 32..55
                wait_ld();
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    if (hf == 1 && c == 3) break;
                    const float *f = reinterpret_cast<const float *>(fv) + c * 8;
                    *reinterpret_cast<uint4 *>(R2 + chunk_off(ROWS, row, hf * 4 + c)) =
                        make_uint4(h2(w * f[0], w * f[1]), h2(w * f[2], w * f[3]), h2(w * f[4], w * f[5]), h2(w * f[6], w * f[7]));
                }
            }
            QPROBE(ctx, 17);
            fence_before_sync();
            ctx_barrier(ctx);
            QPROBE(ctx, 10);
            // (R2 is next written by the next tile's E1, which needs every warp's stage-1 request, issued after its sums.)
            // ---- weighted feature of the group (sarl.py:57-60): sum over its humans -> J chunks 0..6 ----
            if (!HT && sum_split >= 2) {
                const int P = sum_split, nitems = G * 7;
                const int it = t256 / P, seg = t256 & (P - 1);
                const bool on = it < nitems;
                const int sum_c = on ? it / G : 0, sum_gl = on ? it - sum_c * G : 0;
                const int n = on ? (H - seg + P - 1) / P : 0;
                float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                sum_f16x8_rows(R2 + chunk_off(ROWS, sum_gl * H + seg, sum_c), n, 16u * P, acc);
                for (int off = 1; off < P; off <<= 1)
#pragma unroll
                    for (int k = 0; k < 8; ++k) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], off);
                const long long gg = (long long)tile * G + sum_gl;
                if (on && seg == 0 && gg < NG) {
                    uint8_t *jt = J + (size_t)(gg >> 7) * J_TILE_BYTES;
                    *reinterpret_cast<uint4 *>(jt + chunk_off(ROWS, (uint32_t)(gg & 127), sum_c)) =
                        make_uint4(h2(acc[0], acc[1]), h2(acc[2], acc[3]), h2(acc[4], acc[5]), h2(acc[6], acc[7]));
                }
            } else
#pragma unroll
            for (int si = 0; si < kSumIters; ++si) {
                const int it = t256 + si * 256;
                const int sum_c = it / G, sum_gl = it - sum_c * G;
                const long long gg = (long long)tile * G + sum_gl;
                if (it < G * 7 && gg < NG) {
                    const uint8_t *src = R2 + chunk_off(ROWS, sum_gl * H, sum_c);
                    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                    if (HT) {
                        uint4 u[HT ? HT : 1];
#pragma unroll
                        for (int h = 0; h < HT; ++h) u[h] = *reinterpret_cast<const uint4 *>(src + h * 16);
#pragma unroll
                        for (int h = 0; h < HT; ++h) {
                            const __half2 *hv = reinterpret_cast<const __half2 *>(&u[h]);
#pragma unroll
                            for (int k = 0; k < 4; ++k) { const float2 f = __half22float2(hv[k]); acc[2 * k] += f.x; acc[2 * k + 1] += f.y; }
                        }
                    } else {
                        for (int h = 0; h < H; ++h) {
                            const uint4 u = *reinterpret_cast<const uint4 *>(src + h * 16);
                            const __half2 *hv = reinterpret_cast<const __half2 *>(&u);
#pragma unroll
                            for (int k = 0; k < 4; ++k) { const float2 f = __half22float2(hv[k]); acc[2 * k] += f.x; acc[2 * k + 1] += f.y; }
                        }
                    }
                    const float4 a0 = make_float4(acc[0], acc[1], acc[2], acc[3]), a1 = make_float4(acc[4], acc[5], acc[6], acc[7]);
                    uint8_t *jt = J + (size_t)(gg >> 7) * J_TILE_BYTES;
                    *reinterpret_cast<uint4 *>(jt + chunk_off(ROWS, (uint32_t)(gg & 127), sum_c)) =
                        make_uint4(h2(a0.x, a0.y), h2(a0.z, a0.w), h2(a1.x, a1.y), h2(a1.z, a1.w));
                }
            }
            QPROBE(ctx, 11);
        }
#undef PAIR_SIGNAL
#undef PAIR_SIGNAL_TO
#undef PAIR_WAIT
    }
    fence_before_sync();
    __syncthreads();
    cluster_sync_all();
    if (warp == 0) tmem_dealloc_2(tmem, 512);
#undef QPROBE
}

// =====================================================================================================
// self-test of the CTA-pair building block: D[256 x N] = A[256 x K] * B[N x K]^T, including the remote
// "operand ready" arrival and the multicast completion used by tc_rows_pair_kernel
// =====================================================================================================
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(160, 1)
umma_pair_selftest_kernel(const uint8_t *__restrict__ a_img /*2 x [128 x K]*/, const uint8_t *__restrict__ b_img /*2 x [N/2 x K]*/,
                          float *__restrict__ d, int N, int K, int reps, long long *__restrict__ cycles)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    const uint32_t a_bytes = bytes_of(ROWS, K), b_bytes = bytes_of(N / 2, K);
    uint8_t *sa = smem, *sb = smem + a_bytes;
    uint8_t *misc = smem + ((a_bytes + b_bytes + 15) & ~15u);
    const uint32_t req = smem_u32(misc), done = smem_u32(misc + 8);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(misc + 16);
    copy_image_to_smem(sa, a_img + (size_t)rank * a_bytes, a_bytes);
    copy_image_to_smem(sb, b_img + (size_t)rank * b_bytes, b_bytes);
    if (tid == 0) { mbar_init(req, 8); mbar_init(done, 1); fence_mbar_init(); }
    if (warp == 0) tmem_alloc_2(smem_u32(tmem_slot), 512);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    cluster_sync_all();
    fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    long long t0 = clock64();
    if (warp == 4) {
        if (rank == 0 && lane == 0) {
            uint32_t ph = 0;
            for (int rep = 0; rep < reps; ++rep) {
                mbar_wait_cluster(req, ph); ph ^= 1;
                fence_after_sync();
                mma_layer_2(tmem, smem_u32(sa), ROWS, smem_u32(sb), K, N, false);
                commit_2(done, 3);
            }
        }
    } else {
        const uint32_t req_leader = mapa(req, 0);
        const uint32_t tlane = tmem + ((uint32_t)(warp * 32) << 16);
        uint32_t ph = 0;
        for (int rep = 0; rep < reps; ++rep) {
            fence_async_smem();
            fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(req_leader);
            mbar_wait_guarded(done, ph); ph ^= 1;
            fence_after_sync();
        }
        if (tid == 0 && rank == 0 && cycles) *cycles = clock64() - t0;
        for (int c0 = 0; c0 < N; c0 += 16) {
            uint32_t v[16];
            ld16(tlane + c0, v);
            wait_ld();
            for (int k = 0; k < 16; ++k) d[((size_t)rank * ROWS + tid) * N + c0 + k] = __uint_as_float(v[k]);
        }
    }
    fence_before_sync();
    __syncthreads();
    cluster_sync_all();
    if (warp == 0) tmem_dealloc_2(tmem, 512);
}
