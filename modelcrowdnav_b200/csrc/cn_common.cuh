// cn_common.cuh -- internal definitions shared by the kernels and the C ABI (sm_100a only).
#pragma once
#include <atomic>
#include <stdlib.h>
#include <utility>
#include <vector>

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/crowdnav_b200.h"

// ---- field-major SoA state in HBM: state[(field * A1 + agent) * E + env] (f64) -----------------
enum { F_PX = 0, F_PY, F_VX, F_VY, F_GX, F_GY, F_R, F_VPREF, F_COUNT };

struct EnvDims {
    int E;   // envs on this GPU
    int H;   // humans
    int A1;  // H + 1 agents, agent 0 = robot
};

__host__ __device__ __forceinline__ size_t st_idx(const EnvDims &d, int field, int agent, int env)
{
    return ((size_t)field * d.A1 + agent) * d.E + env;
}

struct EnvParams {
    EnvDims d;
    double time_limit, time_step;
    double success_reward, collision_penalty, discomfort_dist, discomfort_penalty_factor;
    float neighbor_dist, time_horizon, time_step_f;
    int max_neighbors;
    double human_safety_space;
    int robot_visible;
    int sim_rule;
    double circle_radius, square_width, human_radius, human_v_pref, robot_radius, robot_v_pref;
    uint64_t seed;
    int64_t env_id_offset;
    int auto_reset;
    double gamma;
    int randomize_attributes;
    int kinematics;       // CN_KIN_*: robot kinematics
};

// per-env episode accumulators (explorer.py:41-51,92-108,124-141)
struct EnvAccum {
    int32_t *ep_steps;       // steps in the running episode
    double *ep_return;       // running discounted return
    int64_t *episodes, *success, *collision, *timeout, *steps, *too_close;
    double *sum_min_dist, *sum_success_time, *sum_collision_time, *sum_timeout_time, *sum_return;
    uint32_t *episode_ctr;   // Philox subsequence of the next device reset
};

struct cn_env {
    int device;
    EnvParams p;
    double *state;        // 8 x A1 x E
    double *time;         // E
    double *human_v;      // 2 x H x E
    double *action_xy;    // 2 x E (pending robot action)
    int32_t *action_idx;  // E
    double *reward;       // E
    uint8_t *done;        // E
    uint8_t *info;        // E
    double *dmin;         // E
    double *next_obs;     // 5 x H x E
    uint8_t *frozen;      // E: episode finished and auto_reset off -> env no longer advances
    EnvAccum acc;
    void *accum_block;    // single allocation backing acc.*
    double *stage;        // device staging, E x A1 x 8 (AoS exchange layout)
    uint32_t *step_ctr;   // E: lookahead draws (epsilon-greedy Philox subsequence)
    double *theta;        // E: robot heading (only read when p.kinematics != CN_KIN_HOLONOMIC)
    int orca_valid;
    // fork/join resources of cn_rollout_step: ORCA runs beside the lookahead when the lookahead does not read it
    cudaStream_t side_stream;
    cudaEvent_t ev_fork, ev_join;
    cudaStream_t tail_stream;          // highest-priority stream for everything after the row kernel (pipelined host steps)
    cudaEvent_t ev_rows, ev_tail;
    double *io_block;     // device image of the packed host exchange block (cn_rollout_step_host_packed), lazily allocated
    // cn_rollout_episodes: "how many envs are still running" read back asynchronously (2 slots, checked one interval late)
    int32_t *active_dev, *active_host;
    cudaEvent_t ev_active[2];
};

struct SarlDims {
    int in, self_dim;
    int m1[2], m2[2], at[3], m3[4];
    int A;  // actions
    int net;        // CN_NET_*: SARL, CADRL (m3 = its mlp on every row), LSTM-RL (m3 = the mlp on cat(self, h_n))
    int lstm_h;     // LSTM hidden size
    int lm1[4];     // LSTM-RL ValueNetwork2's mlp1 widths, lm1[0] = 0 -> ValueNetwork1
    int lstm_in;    // LSTM input width (input_dim or lm1[3])
    int om_dim;     // occupancy-map floats per row (0 = with_om off), cell_num^2 * om_ch
    int cell_num, om_ch;
    double cell_size;
    int no_gs;      // SARL without the global state: attention.0 reads mlp1_out only (in = m1[1])
};

// build_occupancy_maps for ONE human (multi_human_rl.py:109-163): grid of cell_num x cell_num cells of cell_size metres
// centred on the human, x axis along its velocity; per cell [occupied, mean vx, mean vy] (om_ch = 3) of the OTHER humans,
// velocities in the same frame.  get(j, f): f = 0..3 -> px, py, vx, vy of the j-th human in network order.  float64 like
// numpy, one float32 rounding at the end (torch .float()).
// occupancy_map_pair: the cell of human j in human i's grid (-1 = outside) and j's velocity in i's frame.
template <typename Get>
__device__ __forceinline__ int occupancy_map_pair(const SarlDims &d, int i, int j, Get get, double &vxr, double &vyr)
{
    const int cn = d.cell_num;
    const double pxi = get(i, 0), pyi = get(i, 1);
    const double angle = atan2(get(i, 3), get(i, 2));
    const double opx = get(j, 0) - pxi, opy = get(j, 1) - pyi;
    const double rotation = atan2(opy, opx) - angle;
    const double distance = sqrt(opx * opx + opy * opy);
    const double xi = floor(cos(rotation) * distance / d.cell_size + cn / 2.0);
    const double yi = floor(sin(rotation) * distance / d.cell_size + cn / 2.0);
    if (xi < 0 || xi >= cn || yi < 0 || yi >= cn) return -1;
    const double vx = get(j, 2), vy = get(j, 3);
    const double vrot = atan2(vy, vx) - angle, speed = sqrt(vx * vx + vy * vy);
    vxr = cos(vrot) * speed; vyr = sin(vrot) * speed;
    return (int)(cn * yi + xi);
}

// out[c * om_ch ...] of one cell from its sums
__device__ __forceinline__ void occupancy_map_store(int ch, int c, double cnt, double sx, double sy, float *__restrict__ out)
{
    const bool on = cnt > 0.0;
    if (ch == 1) out[c] = on ? 1.0f : 0.0f;
    else if (ch == 2) { out[2 * c] = on ? (float)(sx / cnt) : 0.0f; out[2 * c + 1] = on ? (float)(sy / cnt) : 0.0f; }
    else { out[3 * c] = on ? 1.0f : 0.0f; out[3 * c + 1] = on ? (float)(sx / cnt) : 0.0f; out[3 * c + 2] = on ? (float)(sy / cnt) : 0.0f; }
}

template <typename Get>
__device__ void occupancy_map_row(const SarlDims &d, int H, int i, Get get, float *__restrict__ out)
{
    // every other human's cell and rotated velocity once, then the cells in order (same sums as occupancy_map_cell per cell)
    int cell[CN_MAX_HUMANS];
    double vxr[CN_MAX_HUMANS], vyr[CN_MAX_HUMANS];
    for (int j = 0; j < H; ++j) {
        cell[j] = -1; vxr[j] = 0.0; vyr[j] = 0.0;
        if (j != i) cell[j] = occupancy_map_pair(d, i, j, get, vxr[j], vyr[j]);
    }
    const int cells = d.cell_num * d.cell_num;
    for (int c = 0; c < cells; ++c) {
        double cnt = 0.0, sx = 0.0, sy = 0.0;
        for (int j = 0; j < H; ++j)
            if (cell[j] == c) { cnt += 1.0; sx += vxr[j]; sy += vyr[j]; }
        occupancy_map_store(d.om_ch, c, cnt, sx, sy, out);
    }
}

// fp32 weights on the device, transposed to [in][out_padded] (out padded to a multiple of 4)
struct LinearDev {
    const float *wt;
    const float *b;
    int in, out, ld;
};

struct SarlWeightsDev {
    LinearDev m1[2], m2[2], at[3], m3[4];
    LinearDev lm1[4], lih, lhh;      // LSTM-RL: mlp1 (ValueNetwork2), weight_ih / bias_ih, weight_hh / bias_hh as [in][4h]
};

// One layer of a value network's state dict: a Linear (weight [out][in], then bias [out]) whose device copy is *dst, or
// (dst_hh != nullptr) LSTM-RL's LSTM block: weight_ih_l0 [out][in], weight_hh_l0 [out][out / 4], bias_ih_l0, bias_hh_l0 with
// out = 4 * hidden, device copies *dst (weight_ih / bias_ih) and *dst_hh (weight_hh / bias_hh).
struct LayerSpec {
    int in, out;
    LinearDev *dst, *dst_hh;
};
SarlDims cn_dims_of(const cn_sarl_cfg *c, int om_dim);                   // the network shape of a configuration (capi.cu)
std::vector<LayerSpec> cn_layers(const SarlDims &d, SarlWeightsDev &w);   // state-dict order of d.net (capi.cu)
inline size_t cn_layer_floats(const LayerSpec &l)
{
    return (size_t)l.in * l.out + l.out + (l.dst_hh ? (size_t)(l.out / 4) * l.out + l.out : 0);
}

struct cn_policy {
    int device;
    cn_sarl_cfg cfg;
    SarlDims d;
    double action_host[CN_MAX_ACTIONS * 2];
    double *action_dev;        // A x 2
    float *w_raw;              // flat state-dict order copy (device)
    float *w_t;                // transposed/padded fp32 block
    SarlWeightsDev w;
    int64_t n_params;
    int weights_loaded;
    // lookahead outputs
    double *values;            // E x A
    int32_t *bad_flag;         // [0]: some env of the LAST lookahead had no finite value (cleared per lookahead); [1]: sticky count
                               // of such envs since the handle was created / cn_policy_bad_count(reset)
    size_t values_cap;         // envs `values` has room for
    // tcgen05 path (lookahead_tc.cu)
    void *tc;                  // opaque, owned by the TC module
};

// ---- error plumbing --------------------------------------------------------------------------
void cn_set_error(const char *fmt, ...);
extern std::atomic<int64_t> g_cn_launches;

#define CN_CUDA_CHECK(call)                                                                     \
    do {                                                                                        \
        cudaError_t _e = (call);                                                                \
        if (_e != cudaSuccess) {                                                                \
            cn_set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return CN_ECUDA;                                                                    \
        }                                                                                       \
    } while (0)

// Block size of the small per-env kernels (ORCA, step, reset).  Co-residency with another env shard's persistent kernel
// (PipelinedHostRollout) is decided per SM SUB-PARTITION: tc_rows_pair / tc_mlp3_pair run 19 warps (5,5,5,4 per
// sub-partition) and are capped at 88 registers (__maxnreg__), which leaves 16384 - 5*88*32 = 2304 registers = one warp of
// <= 72 registers in every sub-partition.  So one warp per sub-partition of step (70), reset (52), ORCA (46) or the feature
// kernel (56, one 128-thread block per SM) runs UNDER the persistent kernel; at 96 registers only <= 32-register warps did
// (measured with cn_debug_trace: step + reset of a shard took 258 us, i.e. waited for the other shard's row kernel to exit,
// against 25 us now).  A preferred-carveout hint was tried first and changes nothing.
static inline int cn_small_block() { return 32; }

// developer timeline (cn_debug_trace): when enabled, records a CUDA event named `name` on stream `s`; a no-op otherwise
void cn_trace_mark(const char *name, cudaStream_t s);

#define CN_LAUNCH_CHECK()                                                                       \
    do {                                                                                        \
        ++g_cn_launches;                                                                        \
        cudaError_t _e = cudaGetLastError();                                                    \
        if (_e != cudaSuccess) {                                                                \
            cn_set_error("kernel launch failed at %s:%d: %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return CN_ECUDA;                                                                    \
        }                                                                                       \
    } while (0)

// Kernel launch with an optional programmatic dependent launch (pdl): the grid may become resident while the previous
// kernel on s is still running, so the kernel must griddepcontrol.wait before it reads that kernel's output.
template <typename... KArgs, typename... Args>
int cn_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl, Args &&...args)
{
    cudaLaunchConfig_t lc = {};
    lc.gridDim = grid; lc.blockDim = block; lc.dynamicSmemBytes = smem; lc.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = at; lc.numAttrs = pdl ? 1 : 0;
    CN_CUDA_CHECK(cudaLaunchKernelEx(&lc, kern, std::forward<Args>(args)...));
    CN_LAUNCH_CHECK();
    return CN_OK;
}

// Grow-on-demand scratch buffer: makes buf hold at least n items of item_bytes each.  A buffer that grows loses its contents;
// zero = true clears the new one on stream s.
template <typename T>
int cn_grow(T *&buf, size_t &cap, size_t n, size_t item_bytes, bool zero = false, cudaStream_t s = 0)
{
    if (n <= cap) return CN_OK;
    if (buf) cudaFree(buf);
    buf = nullptr; cap = 0;
    CN_CUDA_CHECK(cudaMalloc((void **)&buf, n * item_bytes));
    if (zero) CN_CUDA_CHECK(cudaMemsetAsync(buf, 0, n * item_bytes, s));
    cap = n;
    return CN_OK;
}

// ---- Philox4x32-10 (counter-based RNG; Salmon et al. 2011) ------------------------------------
struct Philox {
    uint32_t key[2];
    uint32_t ctr[4];
    __host__ __device__ static inline void mulhilo(uint32_t a, uint32_t b, uint32_t &hi, uint32_t &lo)
    {
        const uint64_t p = (uint64_t)a * b;
        hi = (uint32_t)(p >> 32);
        lo = (uint32_t)p;
    }
    __host__ __device__ inline void block(uint32_t out[4]) const
    {
        uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
        uint32_t k0 = key[0], k1 = key[1];
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
        for (int r = 0; r < 10; ++r) {
            uint32_t hi0, lo0, hi1, lo1;
            mulhilo(0xD2511F53u, c0, hi0, lo0);
            mulhilo(0xCD9E8D57u, c2, hi1, lo1);
            const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
            c0 = n0; c1 = n1; c2 = n2; c3 = n3;
            k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
        }
        out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
    }
};

// Uniform double in [0,1) with 53 random bits (same construction as MT19937 genrand_res53).
struct PhiloxStream {
    Philox ph;
    uint32_t buf[4];
    int have;
    uint32_t draw;
    __host__ __device__ inline void init(uint64_t seed, uint64_t env_gid, uint32_t subseq, uint32_t domain)
    {
        ph.key[0] = (uint32_t)seed; ph.key[1] = (uint32_t)(seed >> 32);
        ph.ctr[1] = subseq; ph.ctr[2] = (uint32_t)env_gid;
        ph.ctr[3] = (uint32_t)(env_gid >> 32) ^ (domain << 24);
        have = 0; draw = 0;
    }
    __host__ __device__ inline double next()
    {
        if (have < 2) { ph.ctr[0] = draw++; ph.block(buf); have = 4; }
        const uint32_t a = buf[4 - have] >> 5, b = buf[5 - have] >> 6;
        have -= 2;
        return ((double)a * 67108864.0 + (double)b) / 9007199254740992.0;
    }
};

// Robot action -> the velocity the reference's non-holonomic branches use for collision checking, compute_position and
// propagate: v * cos(theta + r), v * sin(theta + r) (crowd_sim.py:353-354, agent.py:115-117, cadrl.py:119-121).
// Holonomic actions are already velocities.  (CUDA's double cos/sin are within 1-2 ulp of glibc's: positions of the
// non-holonomic modes agree with the reference to ~1e-15 relative, not bit for bit.)
__device__ __forceinline__ void cn_effective_velocity(int kinematics, double theta, double a0, double a1, double &ax, double &ay)
{
    if (kinematics == CN_KIN_HOLONOMIC) { ax = a0; ay = a1; }
    else { ax = a0 * cos(a1 + theta); ay = a0 * sin(a1 + theta); }
}

// np.linalg.norm of a 2-vector as numpy evaluates it: sqrt(fma(b, b, a*a))
__host__ __device__ __forceinline__ double norm2d(double a, double b) { return sqrt(fma(b, b, a * a)); }

// ---- module entry points (each .cu) -----------------------------------------------------------
int cn_launch_orca(cn_env *env, cudaStream_t s);
int cn_launch_robot_orca(cn_env *env, double safety_space, cudaStream_t s);
int cn_launch_step(cn_env *env, const double *action_xy_dev, int update, cudaStream_t s, int fuse_reset = 0);
int cn_launch_reset(cn_env *env, int only_done, cudaStream_t s);
int cn_launch_pack(cn_env *env, int to_soa, cudaStream_t s);  // stage (AoS) <-> state (SoA)
int cn_launch_io(cn_env *env, double *blk, int unpack, cudaStream_t s);   // packed host exchange block <-> device state

int cn_lookahead_f32(cn_policy *p, cn_env *env, int query_env, double epsilon, cudaStream_t s);
int cn_transform_f32(cn_policy *p, cn_env *env, float *out_dev, int sort_humans, cudaStream_t s);
int cn_forward_f32(cn_policy *p, const float *x_dev, int batch, int H, float *out_dev, cudaStream_t s);
int cn_f32_configure_device(void);   // per-device kernel attributes (call after cudaSetDevice)

int cn_tc_init(cn_policy *p);
void cn_tc_destroy(cn_policy *p);
int cn_tc_load_weights(cn_policy *p, const float *flat_host, cudaStream_t s);
// tail != nullptr: the scoring stage (mlp3, or CADRL's minimum over the humans) and the argmax of every network go to `tail`,
// ordered after `s` by env->ev_rows
int cn_lookahead_tc(cn_policy *p, cn_env *env, int query_env, double epsilon, cudaStream_t s, cudaStream_t tail = nullptr);
