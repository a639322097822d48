// capi.cu -- the extern "C" surface declared in include/crowdnav_b200.h.
#include "cn_common.cuh"

#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

std::atomic<int64_t> g_cn_launches{0};
static thread_local char g_err[512] = "";

void cn_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cn_launch_transpose_out(int E, int H, int C, const double *src, double *dst, cudaStream_t s);
int cn_launch_set_actions(cn_env *env, const double *aos_dev, cudaStream_t s);
int cn_launch_set_human_v(cn_env *env, const double *aos_dev, cudaStream_t s);
int cn_launch_pack_keep(cn_env *env, cudaStream_t s);

// ---- developer timeline: named CUDA events on whatever streams the work runs on -----------------
struct TraceRec { const char *name; cudaStream_t stream; cudaEvent_t ev; };
static std::vector<TraceRec> g_trace;
static bool g_trace_on = false;

void cn_trace_mark(const char *name, cudaStream_t s)
{
    if (!g_trace_on || g_trace.size() >= 4096) return;
    cudaEvent_t ev;
    if (cudaEventCreate(&ev) != cudaSuccess) return;
    cudaEventRecord(ev, s);
    g_trace.push_back({name, s, ev});
}

// ---- network shapes and state-dict layer lists ---------------------------------------------------
// The network shape of a configuration (om_dim = 0 without occupancy maps)
SarlDims cn_dims_of(const cn_sarl_cfg *c, int om_dim)
{
    SarlDims d;
    memset(&d, 0, sizeof(d));
    d.in = c->input_dim; d.self_dim = c->self_state_dim;
    for (int i = 0; i < 2; ++i) { d.m1[i] = c->mlp1_dims[i]; d.m2[i] = c->mlp2_dims[i]; }
    for (int i = 0; i < 3; ++i) d.at[i] = c->attn_dims[i];
    for (int i = 0; i < 4; ++i) d.m3[i] = c->mlp3_dims[i];
    d.net = c->network; d.lstm_h = c->network == CN_NET_LSTM_RL ? c->lstm_hidden : 0;
    for (int i = 0; i < 4; ++i) d.lm1[i] = c->network == CN_NET_LSTM_RL ? c->lstm_mlp1_dims[i] : 0;
    d.lstm_in = d.lm1[0] > 0 ? d.lm1[3] : d.in;
    d.om_dim = om_dim; d.cell_num = c->cell_num; d.om_ch = c->om_channel_size; d.cell_size = c->cell_size;
    d.no_gs = c->network == CN_NET_SARL && c->without_global_state ? 1 : 0;
    return d;
}

std::vector<LayerSpec> cn_layers(const SarlDims &d, SarlWeightsDev &w)
{
    std::vector<LayerSpec> L;
    int in = d.in;
    auto chain = [&](int n, const int *outs, LinearDev *dst) {
        for (int i = 0; i < n; ++i) { L.push_back({in, outs[i], &dst[i], nullptr}); in = outs[i]; }
    };
    if (d.net == CN_NET_CADRL) {                          // value_network.{0,2,4,6} (cadrl.py:22-26)
        chain(4, d.m3, w.m3);
    } else if (d.net == CN_NET_LSTM_RL) {                 // [mlp1.*] mlp.* lstm.* (lstm_rl.py:9-16,37-45)
        if (d.lm1[0] > 0) chain(4, d.lm1, w.lm1);
        in = d.self_dim + d.lstm_h;
        chain(4, d.m3, w.m3);
        L.push_back({d.lstm_in, 4 * d.lstm_h, &w.lih, &w.lhh});
    } else {                                              // mlp1.* mlp2.* attention.* mlp3.*
        chain(2, d.m1, w.m1);
        chain(2, d.m2, w.m2);
        in = d.no_gs ? d.m1[1] : 2 * d.m1[1];           // attention.0 on [mlp1_out | mean] or mlp1_out (sarl.py:40-47)
        chain(3, d.at, w.at);
        in = d.m2[1] + d.self_dim;
        chain(4, d.m3, w.m3);
    }
    return L;
}

extern "C" {

/* Developer diagnostic: on = 1 starts recording a timeline of the library's stream operations (one CUDA event per mark),
 * on = 0 stops.  cn_debug_trace_dump synchronises the device and writes "ms_since_first_mark stream name" lines. */
int cn_debug_trace(int on)
{
    for (auto &r : g_trace) cudaEventDestroy(r.ev);
    g_trace.clear();
    g_trace_on = on != 0;
    return CN_OK;
}

int cn_debug_trace_dump(char *buf, int64_t cap)
{
    if (!buf || cap < 1) { cn_set_error("null buffer"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaDeviceSynchronize());
    int64_t off = 0;
    buf[0] = 0;
    for (size_t i = 0; i < g_trace.size(); ++i) {
        float ms = 0.0f;
        cudaEventElapsedTime(&ms, g_trace[0].ev, g_trace[i].ev);
        const int n = snprintf(buf + off, (size_t)(cap - off), "%.4f %p %s\n", ms, (void *)g_trace[i].stream, g_trace[i].name);
        if (n < 0 || off + n >= cap) break;
        off += n;
    }
    return CN_OK;
}

const char *cn_last_error(void) { return g_err; }
int cn_version(void) { return 100; }
int64_t cn_launch_count(void) { return g_cn_launches.load(); }

int cn_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void cn_env_cfg_default(cn_env_cfg *c)
{
    memset(c, 0, sizeof(*c));
    c->num_envs = 1; c->human_num = 5;
    c->time_limit = 25; c->time_step = 0.25;
    c->success_reward = 1; c->collision_penalty = -0.25; c->discomfort_dist = 0.2; c->discomfort_penalty_factor = 0.5;
    c->neighbor_dist = 10; c->max_neighbors = 10; c->time_horizon = 5; c->human_safety_space = 0;
    c->robot_visible = 0;
    c->sim_rule = CN_CIRCLE_CROSSING; c->circle_radius = 4; c->square_width = 10;
    c->human_radius = 0.3; c->human_v_pref = 1; c->robot_radius = 0.3; c->robot_v_pref = 1;
    c->seed = 0; c->env_id_offset = 0; c->auto_reset = 0; c->gamma = 0.9;
    c->randomize_attributes = 0;
    c->robot_kinematics = CN_KIN_HOLONOMIC;
}

void cn_sarl_cfg_default(cn_sarl_cfg *c)
{
    memset(c, 0, sizeof(*c));
    c->input_dim = 13; c->self_state_dim = 6;
    c->mlp1_dims[0] = 150; c->mlp1_dims[1] = 100;
    c->mlp2_dims[0] = 100; c->mlp2_dims[1] = 50;
    c->attn_dims[0] = 100; c->attn_dims[1] = 100; c->attn_dims[2] = 1;
    c->mlp3_dims[0] = 150; c->mlp3_dims[1] = 100; c->mlp3_dims[2] = 100; c->mlp3_dims[3] = 1;
    c->speed_samples = 5; c->rotation_samples = 16;
    c->gamma = 0.9; c->v_pref = 1.0; c->precision = CN_PREC_F32;
    c->kinematics = CN_KIN_HOLONOMIC;
    c->network = CN_NET_SARL; c->lstm_hidden = 50;      // [lstm_rl] global_state_dim; lstm_mlp1_dims = {0}: ValueNetwork1
    c->with_om = 0; c->cell_num = 4; c->cell_size = 1.0; c->om_channel_size = 3;   // [om]
}

static int use_device(int device)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        cn_set_error("no CUDA device available (%s); libcrowdnav_b200 has no CPU fallback",
                     e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        return CN_ECUDA;
    }
    if (device < 0 || device >= n) { cn_set_error("device %d out of range (0..%d)", device, n - 1); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CN_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        cn_set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
        return CN_ECUDA;
    }
    return CN_OK;
}

// ---------------------------------------------------------------------------------------------
// environment
// ---------------------------------------------------------------------------------------------

int cn_env_create(const cn_env_cfg *cfg, int device, cn_env **out)
{
    if (!cfg || !out) { cn_set_error("null argument"); return CN_EINVAL; }
    if (cfg->num_envs < 1 || cfg->human_num < 1 || cfg->human_num > CN_MAX_HUMANS) {
        cn_set_error("num_envs >= 1 and 1 <= human_num <= %d required", CN_MAX_HUMANS);
        return CN_EINVAL;
    }
    if (cfg->max_neighbors < 0 || cfg->max_neighbors > CN_MAX_NEIGHBORS) {
        cn_set_error("max_neighbors must be in [0, %d]", CN_MAX_NEIGHBORS);
        return CN_EINVAL;
    }
    if (!(cfg->time_step > 0)) { cn_set_error("time_step must be positive"); return CN_EINVAL; }
    int rc = use_device(device);
    if (rc) return rc;

    cn_env *env = new cn_env();
    memset(env, 0, sizeof(*env));
    env->device = device;
    EnvParams &p = env->p;
    p.d.E = cfg->num_envs; p.d.H = cfg->human_num; p.d.A1 = cfg->human_num + 1;
    p.time_limit = cfg->time_limit; p.time_step = cfg->time_step;
    p.success_reward = cfg->success_reward; p.collision_penalty = cfg->collision_penalty;
    p.discomfort_dist = cfg->discomfort_dist; p.discomfort_penalty_factor = cfg->discomfort_penalty_factor;
    // rvo2 takes C floats: Python doubles are rounded at the Cython boundary (orca.py:94,99)
    p.neighbor_dist = (float)cfg->neighbor_dist; p.time_horizon = (float)cfg->time_horizon;
    p.time_step_f = (float)cfg->time_step; p.max_neighbors = cfg->max_neighbors;
    p.human_safety_space = cfg->human_safety_space; p.robot_visible = cfg->robot_visible;
    p.sim_rule = cfg->sim_rule; p.circle_radius = cfg->circle_radius; p.square_width = cfg->square_width;
    p.human_radius = cfg->human_radius; p.human_v_pref = cfg->human_v_pref;
    p.robot_radius = cfg->robot_radius; p.robot_v_pref = cfg->robot_v_pref;
    p.seed = cfg->seed; p.env_id_offset = cfg->env_id_offset; p.auto_reset = cfg->auto_reset;
    p.gamma = cfg->gamma;
    p.randomize_attributes = cfg->randomize_attributes;
    p.kinematics = cfg->robot_kinematics;

    const size_t E = p.d.E, H = p.d.H, A1 = p.d.A1;
#define CN_ALLOC(ptr, bytes)                                                     \
    do {                                                                         \
        cudaError_t _e = cudaMalloc((void **)&(ptr), (bytes));                   \
        if (_e != cudaSuccess) {                                                 \
            cn_set_error("cudaMalloc(%zu) failed: %s", (size_t)(bytes), cudaGetErrorString(_e)); \
            cn_env_destroy(env);                                                 \
            return CN_ENOMEM;                                                    \
        }                                                                        \
        cudaMemset((ptr), 0, (bytes));                                           \
    } while (0)
    CN_ALLOC(env->state, sizeof(double) * F_COUNT * A1 * E);
    CN_ALLOC(env->time, sizeof(double) * E);
    CN_ALLOC(env->human_v, sizeof(double) * 2 * H * E);
    CN_ALLOC(env->action_xy, sizeof(double) * 2 * E);
    CN_ALLOC(env->action_idx, sizeof(int32_t) * E);
    CN_ALLOC(env->reward, sizeof(double) * E);
    CN_ALLOC(env->done, E);
    CN_ALLOC(env->info, E);
    CN_ALLOC(env->dmin, sizeof(double) * E);
    CN_ALLOC(env->next_obs, sizeof(double) * 5 * H * E);
    CN_ALLOC(env->frozen, E);
    CN_ALLOC(env->stage, sizeof(double) * F_COUNT * A1 * E);
    CN_ALLOC(env->step_ctr, sizeof(uint32_t) * E);
    CN_ALLOC(env->theta, sizeof(double) * E);
    // accumulators: 6 int64 + 6 double + 1 double + int32 + uint32 per env
    const size_t acc_bytes = E * (6 * 8 + 6 * 8 + 4 + 4);
    CN_ALLOC(env->accum_block, acc_bytes);
#undef CN_ALLOC
    char *b = (char *)env->accum_block;
    EnvAccum &a = env->acc;
    a.episodes = (int64_t *)b; b += 8 * E;
    a.success = (int64_t *)b; b += 8 * E;
    a.collision = (int64_t *)b; b += 8 * E;
    a.timeout = (int64_t *)b; b += 8 * E;
    a.steps = (int64_t *)b; b += 8 * E;
    a.too_close = (int64_t *)b; b += 8 * E;
    a.sum_min_dist = (double *)b; b += 8 * E;
    a.sum_success_time = (double *)b; b += 8 * E;
    a.sum_collision_time = (double *)b; b += 8 * E;
    a.sum_timeout_time = (double *)b; b += 8 * E;
    a.sum_return = (double *)b; b += 8 * E;
    a.ep_return = (double *)b; b += 8 * E;
    a.ep_steps = (int32_t *)b; b += 4 * E;
    a.episode_ctr = (uint32_t *)b; b += 4 * E;
    *out = env;
    return CN_OK;
}

int cn_env_destroy(cn_env *env)
{
    if (!env) return CN_OK;
    cudaSetDevice(env->device);
    void *ptrs[] = {env->state, env->time, env->human_v, env->action_xy, env->action_idx, env->reward, env->done,
                    env->info, env->dmin, env->next_obs, env->frozen, env->stage, env->step_ctr, env->accum_block, env->theta};
    for (void *q : ptrs) if (q) cudaFree(q);
    if (env->io_block) cudaFree(env->io_block);
    if (env->side_stream) cudaStreamDestroy(env->side_stream);
    if (env->ev_fork) cudaEventDestroy(env->ev_fork);
    if (env->ev_join) cudaEventDestroy(env->ev_join);
    if (env->tail_stream) cudaStreamDestroy(env->tail_stream);
    if (env->ev_rows) cudaEventDestroy(env->ev_rows);
    if (env->ev_tail) cudaEventDestroy(env->ev_tail);
    if (env->active_dev) cudaFree(env->active_dev);
    if (env->active_host) cudaFreeHost(env->active_host);
    for (cudaEvent_t ev : env->ev_active) if (ev) cudaEventDestroy(ev);
    delete env;
    return CN_OK;
}

#define CN_ENV_ENTER(env)                                              \
    if (!(env)) { cn_set_error("null env handle"); return CN_EINVAL; } \
    CN_CUDA_CHECK(cudaSetDevice((env)->device));                       \
    cudaStream_t s = (cudaStream_t)stream

int cn_env_set_theta(cn_env *env, const double *theta_host, void *stream)
{
    CN_ENV_ENTER(env);
    if (!theta_host) { cn_set_error("theta_host is null"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaMemcpyAsync(env->theta, theta_host, sizeof(double) * env->p.d.E, cudaMemcpyHostToDevice, s));
    CN_CUDA_CHECK(cudaStreamSynchronize(s));
    return CN_OK;
}

int cn_env_get_theta(cn_env *env, double *theta_host, void *stream)
{
    CN_ENV_ENTER(env);
    if (!theta_host) { cn_set_error("theta_host is null"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaMemcpyAsync(theta_host, env->theta, sizeof(double) * env->p.d.E, cudaMemcpyDeviceToHost, s));
    CN_CUDA_CHECK(cudaStreamSynchronize(s));
    return CN_OK;
}

int cn_env_set_state(cn_env *env, const double *agents_host, const double *times_host, void *stream)
{
    CN_ENV_ENTER(env);
    if (!agents_host) { cn_set_error("agents_host is null"); return CN_EINVAL; }
    const size_t E = env->p.d.E, A1 = env->p.d.A1;
    CN_CUDA_CHECK(cudaMemcpyAsync(env->stage, agents_host, sizeof(double) * E * A1 * F_COUNT, cudaMemcpyHostToDevice, s));
    int rc = cn_launch_pack(env, 1, s);
    if (rc) return rc;
    if (times_host) CN_CUDA_CHECK(cudaMemcpyAsync(env->time, times_host, sizeof(double) * E, cudaMemcpyHostToDevice, s));
    else CN_CUDA_CHECK(cudaMemsetAsync(env->time, 0, sizeof(double) * E, s));
    return CN_OK;
}

int cn_env_get_state(cn_env *env, double *agents_host, double *times_host, void *stream)
{
    CN_ENV_ENTER(env);
    const size_t E = env->p.d.E, A1 = env->p.d.A1;
    if (agents_host) {
        int rc = cn_launch_pack(env, 0, s);
        if (rc) return rc;
        CN_CUDA_CHECK(cudaMemcpyAsync(agents_host, env->stage, sizeof(double) * E * A1 * F_COUNT, cudaMemcpyDeviceToHost, s));
    }
    if (times_host) CN_CUDA_CHECK(cudaMemcpyAsync(times_host, env->time, sizeof(double) * E, cudaMemcpyDeviceToHost, s));
    CN_CUDA_CHECK(cudaStreamSynchronize(s));
    return CN_OK;
}

int cn_env_reset(cn_env *env, void *stream)
{
    CN_ENV_ENTER(env);
    return cn_launch_reset(env, 0, s);
}

int cn_env_orca(cn_env *env, void *stream)
{
    CN_ENV_ENTER(env);
    return cn_launch_orca(env, s);
}

int cn_env_robot_orca(cn_env *env, double safety_space, void *stream)
{
    CN_ENV_ENTER(env);
    return cn_launch_robot_orca(env, safety_space, s);
}

int cn_env_step(cn_env *env, const double *action_xy_dev, int update, void *stream)
{
    CN_ENV_ENTER(env);
    if (!env->orca_valid) {
        cn_set_error("cn_env_step: call cn_env_orca for the current state first");
        return CN_EINVAL;
    }
    int rc = cn_launch_step(env, action_xy_dev, update, s);
    if (rc) return rc;
    if (update && env->p.auto_reset) rc = cn_launch_reset(env, 1, s);
    return rc;
}

int cn_env_get_views(cn_env *env, cn_env_views *out)
{
    if (!env || !out) { cn_set_error("null argument"); return CN_EINVAL; }
    out->reward = env->reward; out->done = env->done; out->info = env->info; out->dmin = env->dmin;
    out->human_v = env->human_v; out->next_obs = env->next_obs; out->state = env->state; out->time = env->time;
    out->action_idx = env->action_idx; out->action_xy = env->action_xy;
    return CN_OK;
}

int cn_env_read_outputs(cn_env *env, double *reward, uint8_t *done, uint8_t *info, double *dmin, void *stream)
{
    CN_ENV_ENTER(env);
    const size_t E = env->p.d.E;
    if (reward) CN_CUDA_CHECK(cudaMemcpyAsync(reward, env->reward, sizeof(double) * E, cudaMemcpyDeviceToHost, s));
    if (done) CN_CUDA_CHECK(cudaMemcpyAsync(done, env->done, E, cudaMemcpyDeviceToHost, s));
    if (info) CN_CUDA_CHECK(cudaMemcpyAsync(info, env->info, E, cudaMemcpyDeviceToHost, s));
    if (dmin) CN_CUDA_CHECK(cudaMemcpyAsync(dmin, env->dmin, sizeof(double) * E, cudaMemcpyDeviceToHost, s));
    CN_CUDA_CHECK(cudaStreamSynchronize(s));
    return CN_OK;
}

int cn_env_read_human_actions(cn_env *env, double *human_vxy_host, void *stream)
{
    CN_ENV_ENTER(env);
    if (!env->orca_valid) { cn_set_error("no cached ORCA result; call cn_env_orca"); return CN_EINVAL; }
    const size_t E = env->p.d.E, H = env->p.d.H;
    int rc = cn_launch_transpose_out((int)E, (int)H, 2, env->human_v, env->stage, s);
    if (rc) return rc;
    CN_CUDA_CHECK(cudaMemcpyAsync(human_vxy_host, env->stage, sizeof(double) * E * H * 2, cudaMemcpyDeviceToHost, s));
    CN_CUDA_CHECK(cudaStreamSynchronize(s));
    return CN_OK;
}

int cn_env_read_next_obs(cn_env *env, double *obs_host, void *stream)
{
    CN_ENV_ENTER(env);
    const size_t E = env->p.d.E, H = env->p.d.H;
    int rc = cn_launch_transpose_out((int)E, (int)H, 5, env->next_obs, env->stage, s);
    if (rc) return rc;
    CN_CUDA_CHECK(cudaMemcpyAsync(obs_host, env->stage, sizeof(double) * E * H * 5, cudaMemcpyDeviceToHost, s));
    CN_CUDA_CHECK(cudaStreamSynchronize(s));
    return CN_OK;
}

int cn_env_read_actions(cn_env *env, double *action_xy_host, int32_t *action_idx_host, void *stream)
{
    CN_ENV_ENTER(env);
    const size_t E = env->p.d.E;
    if (action_xy_host) {
        // pending action is 2 x E on the device; transpose through the staging buffer
        int rc = cn_launch_transpose_out((int)E, 1, 2, env->action_xy, env->stage, s);
        if (rc) return rc;
        CN_CUDA_CHECK(cudaMemcpyAsync(action_xy_host, env->stage, sizeof(double) * 2 * E, cudaMemcpyDeviceToHost, s));
    }
    if (action_idx_host)
        CN_CUDA_CHECK(cudaMemcpyAsync(action_idx_host, env->action_idx, sizeof(int32_t) * E, cudaMemcpyDeviceToHost, s));
    CN_CUDA_CHECK(cudaStreamSynchronize(s));
    return CN_OK;
}

int cn_env_set_actions(cn_env *env, const double *action_xy_host, void *stream)
{
    CN_ENV_ENTER(env);
    if (!action_xy_host) { cn_set_error("action_xy_host is null"); return CN_EINVAL; }
    const size_t E = env->p.d.E;
    CN_CUDA_CHECK(cudaMemcpyAsync(env->stage, action_xy_host, sizeof(double) * 2 * E, cudaMemcpyHostToDevice, s));
    return cn_launch_set_actions(env, env->stage, s);
}

int cn_env_set_human_actions(cn_env *env, const double *human_vxy_host, void *stream)
{
    CN_ENV_ENTER(env);
    if (!human_vxy_host) { cn_set_error("human_vxy_host is null"); return CN_EINVAL; }
    const size_t n = (size_t)env->p.d.E * env->p.d.H * 2;
    CN_CUDA_CHECK(cudaMemcpyAsync(env->stage, human_vxy_host, sizeof(double) * n, cudaMemcpyHostToDevice, s));
    return cn_launch_set_human_v(env, env->stage, s);
}

int cn_env_read_stats(cn_env *env, cn_stats *out, int reset, void *stream)
{
    CN_ENV_ENTER(env);
    if (!out) { cn_set_error("null stats"); return CN_EINVAL; }
    const size_t E = env->p.d.E;
    const size_t bytes = E * 8 * 11;  // the 11 reducible arrays are contiguous at the head of accum_block
    std::vector<char> host(bytes);
    CN_CUDA_CHECK(cudaMemcpyAsync(host.data(), env->accum_block, bytes, cudaMemcpyDeviceToHost, s));
    CN_CUDA_CHECK(cudaStreamSynchronize(s));
    const int64_t *iv = (const int64_t *)host.data();
    const double *dv = (const double *)(host.data() + 6 * 8 * E);
    int64_t isum[6] = {0, 0, 0, 0, 0, 0};
    double dsum[5] = {0, 0, 0, 0, 0};
    for (int k = 0; k < 6; ++k) for (size_t e = 0; e < E; ++e) isum[k] += iv[k * E + e];
    for (int k = 0; k < 5; ++k) for (size_t e = 0; e < E; ++e) dsum[k] += dv[k * E + e];
    out->episodes = isum[0]; out->success = isum[1]; out->collision = isum[2]; out->timeout = isum[3];
    out->steps = isum[4]; out->too_close = isum[5];
    out->sum_min_dist = dsum[0]; out->sum_success_time = dsum[1]; out->sum_collision_time = dsum[2];
    out->sum_timeout_time = dsum[3]; out->sum_return = dsum[4];
    if (reset) CN_CUDA_CHECK(cudaMemsetAsync(env->accum_block, 0, bytes, s));
    return CN_OK;
}

int cn_env_copy_outputs(cn_env *env, double *reward_dev, uint8_t *done_dev, uint8_t *info_dev, void *stream)
{
    CN_ENV_ENTER(env);
    const size_t E = env->p.d.E;
    if (reward_dev) CN_CUDA_CHECK(cudaMemcpyAsync(reward_dev, env->reward, sizeof(double) * E, cudaMemcpyDeviceToDevice, s));
    if (done_dev) CN_CUDA_CHECK(cudaMemcpyAsync(done_dev, env->done, E, cudaMemcpyDeviceToDevice, s));
    if (info_dev) CN_CUDA_CHECK(cudaMemcpyAsync(info_dev, env->info, E, cudaMemcpyDeviceToDevice, s));
    return CN_OK;
}

int64_t cn_env_episode_table_bytes(const cn_env *env) { return env ? (int64_t)env->p.d.E * 8 * 11 : 0; }

int cn_env_read_episode_table(cn_env *env, void *table_host, uint8_t *frozen_host, void *stream)
{
    CN_ENV_ENTER(env);
    const size_t E = env->p.d.E;
    if (table_host) CN_CUDA_CHECK(cudaMemcpyAsync(table_host, env->accum_block, E * 8 * 11, cudaMemcpyDeviceToHost, s));
    if (frozen_host) CN_CUDA_CHECK(cudaMemcpyAsync(frozen_host, env->frozen, E, cudaMemcpyDeviceToHost, s));
    CN_CUDA_CHECK(cudaStreamSynchronize(s));
    return CN_OK;
}

// ---------------------------------------------------------------------------------------------
// policy
// ---------------------------------------------------------------------------------------------

static int pad4i(int x) { return (x + 3) & ~3; }

int64_t cn_policy_param_count(const cn_sarl_cfg *c)
{
    if (!c) return 0;
    SarlWeightsDev w;        // only the destinations of the layer list, never written here
    int64_t n = 0;
    for (const LayerSpec &l : cn_layers(cn_dims_of(c, 0), w)) n += (int64_t)cn_layer_floats(l);
    return n;
}

// CADRL.build_action_space (cadrl.py:82-102); glibc exp/cos/sin like numpy on the host.  Holonomic: (vx, vy) over 16
// headings; otherwise ActionRot (v, r) with r in np.linspace(-pi/4, pi/4, R) (endpoint included, last sample = stop).
static int build_action_table(const cn_sarl_cfg *c, double *out)
{
    const double E_ = 2.718281828459045;
    int n = 0;
    out[0] = 0; out[1] = 0; n = 1;
    if (c->kinematics != CN_KIN_HOLONOMIC) {
        const double PI = 3.141592653589793, start = -PI / 4, stop = PI / 4;
        const int div = c->rotation_samples - 1;
        const double step = div > 0 ? (stop - start) / div : 0.0;
        for (int r = 0; r < c->rotation_samples; ++r) {
            double rotation = start + r * step;
            if (div > 0 && r == c->rotation_samples - 1) rotation = stop;
            for (int s = 0; s < c->speed_samples; ++s) {
                out[2 * n] = (exp((double)(s + 1) / c->speed_samples) - 1) / (E_ - 1) * c->v_pref;
                out[2 * n + 1] = rotation;
                ++n;
            }
        }
        return n;
    }
    const double step = (2 * 3.141592653589793 - 0) / c->rotation_samples;
    for (int r = 0; r < c->rotation_samples; ++r) {
        const double rotation = r * step;
        for (int s = 0; s < c->speed_samples; ++s) {
            const double speed = (exp((double)(s + 1) / c->speed_samples) - 1) / (E_ - 1) * c->v_pref;
            out[2 * n] = speed * cos(rotation);
            out[2 * n + 1] = speed * sin(rotation);
            ++n;
        }
    }
    return n;
}

int cn_policy_create(const cn_sarl_cfg *cfg, int device, cn_policy **out)
{
    if (!cfg || !out) { cn_set_error("null argument"); return CN_EINVAL; }
    const int A = cfg->speed_samples * cfg->rotation_samples + 1;
    int om_dim = 0;
    if (cfg->with_om) {
        if (cfg->cell_num < 1 || cfg->cell_num > 8 || cfg->om_channel_size < 1 || cfg->om_channel_size > 3 || !(cfg->cell_size > 0)) {
            cn_set_error("with_om needs 1 <= cell_num <= 8, om_channel_size in {1, 2, 3} and cell_size > 0");
            return CN_EINVAL;
        }
        if (cfg->network == CN_NET_CADRL) { cn_set_error("CADRL has no occupancy maps (cadrl.py:60-62)"); return CN_EINVAL; }
        if (cfg->precision != CN_PREC_F32 && cfg->network != CN_NET_SARL) {
            cn_set_error("occupancy maps on the tensor-core path are built for SARL only; use CN_PREC_F32"); return CN_EUNSUPPORTED;
        }
        om_dim = cfg->cell_num * cfg->cell_num * cfg->om_channel_size;
    }
    if (cfg->input_dim != 13 + om_dim || cfg->self_state_dim < 1 || cfg->self_state_dim > 13) {
        cn_set_error("input_dim must be 13 + cell_num^2 * om_channel_size (13 without maps) and 1 <= self_state_dim <= 13");
        return CN_EUNSUPPORTED;
    }
    if (cfg->attn_dims[2] != 1 || cfg->mlp3_dims[3] != 1) { cn_set_error("attention and mlp3 must end in 1 unit"); return CN_EINVAL; }
    if (cfg->network != CN_NET_SARL && cfg->network != CN_NET_CADRL && cfg->network != CN_NET_LSTM_RL) {
        cn_set_error("unknown value network %d", cfg->network); return CN_EINVAL;
    }
    if (cfg->without_global_state && cfg->network != CN_NET_SARL) {
        cn_set_error("without_global_state is a [sarl] option; CADRL and LSTM-RL have no global state"); return CN_EINVAL;
    }
    if (cfg->network == CN_NET_LSTM_RL) {
        if (cfg->lstm_hidden < 1 || cfg->lstm_hidden > 64) { cn_set_error("1 <= lstm_hidden <= 64 required"); return CN_EINVAL; }
        if (cfg->lstm_mlp1_dims[0] > 0)
            for (int i = 0; i < 4; ++i)
                if (cfg->lstm_mlp1_dims[i] < 1 || cfg->lstm_mlp1_dims[i] > 256) { cn_set_error("layer widths must be in [1, 256]"); return CN_EINVAL; }
    }
    if (A < 1 || A > CN_MAX_ACTIONS) { cn_set_error("1 <= speed_samples*rotation_samples+1 <= %d required", CN_MAX_ACTIONS); return CN_EINVAL; }
    const int dims[] = {cfg->mlp1_dims[0], cfg->mlp1_dims[1], cfg->mlp2_dims[0], cfg->mlp2_dims[1], cfg->attn_dims[0],
                        cfg->attn_dims[1], cfg->mlp3_dims[0], cfg->mlp3_dims[1], cfg->mlp3_dims[2]};
    for (int v : dims) if (v < 1 || v > 256) { cn_set_error("layer widths must be in [1, 256]"); return CN_EINVAL; }
    if (cfg->precision != CN_PREC_F32 && cfg->precision != CN_PREC_F16_TC) { cn_set_error("unknown precision"); return CN_EINVAL; }
    int rc = use_device(device);
    if (rc) return rc;
    if ((rc = cn_f32_configure_device())) return rc;

    cn_policy *p = new cn_policy();
    memset(p, 0, sizeof(*p));
    p->device = device; p->cfg = *cfg;
    p->d = cn_dims_of(cfg, om_dim);
    SarlDims &d = p->d;
    d.A = build_action_table(cfg, p->action_host);
    p->n_params = cn_policy_param_count(cfg);

    // transposed/padded block: per layer in * pad4(out) + pad4(out) (the LSTM block: for W_ih and for W_hh)
    size_t tsize = 0;
    for (const LayerSpec &l : cn_layers(d, p->w))
        tsize += (size_t)(l.in + 1) * pad4i(l.out) + (l.dst_hh ? (size_t)(l.out / 4 + 1) * pad4i(l.out) : 0);
    cudaError_t e1 = cudaMalloc((void **)&p->action_dev, sizeof(double) * 2 * d.A);
    cudaError_t e2 = cudaMalloc((void **)&p->w_raw, sizeof(float) * p->n_params);
    cudaError_t e3 = cudaMalloc((void **)&p->w_t, sizeof(float) * tsize);
    cudaError_t e4 = cudaMalloc((void **)&p->bad_flag, 2 * sizeof(int32_t));
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess || e4 != cudaSuccess) {
        cn_set_error("cudaMalloc failed in cn_policy_create");
        cn_policy_destroy(p);
        return CN_ENOMEM;
    }
    cudaMemset(p->bad_flag, 0, 2 * sizeof(int32_t));
    CN_CUDA_CHECK(cudaMemcpy(p->action_dev, p->action_host, sizeof(double) * 2 * d.A, cudaMemcpyHostToDevice));
    if (cfg->precision == CN_PREC_F16_TC) {
        rc = cn_tc_init(p);
        if (rc) { cn_policy_destroy(p); return rc; }
    }
    *out = p;
    return CN_OK;
}

int cn_policy_destroy(cn_policy *p)
{
    if (!p) return CN_OK;
    cudaSetDevice(p->device);
    if (p->tc) cn_tc_destroy(p);
    void *ptrs[] = {p->action_dev, p->w_raw, p->w_t, p->bad_flag, p->values};
    for (void *q : ptrs) if (q) cudaFree(q);
    delete p;
    return CN_OK;
}

int cn_policy_load_weights(cn_policy *p, const float *flat, int64_t n, void *stream)
{
    if (!p || !flat) { cn_set_error("null argument"); return CN_EINVAL; }
    if (n != p->n_params) { cn_set_error("expected %lld parameters, got %lld", (long long)p->n_params, (long long)n); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    // host-side transpose to [in][pad4(out)] + bias, one contiguous block
    std::vector<float> t;
    auto put = [&](int in, int out, const float *w, const float *b, LinearDev *dst) {
        const int ld = pad4i(out);
        const size_t off = t.size();
        t.resize(off + (size_t)in * ld + ld, 0.0f);
        for (int o = 0; o < out; ++o)
            for (int k = 0; k < in; ++k) t[off + (size_t)k * ld + o] = w[(size_t)o * in + k];
        for (int o = 0; o < out; ++o) t[off + (size_t)in * ld + o] = b[o];
        dst->wt = p->w_t + off; dst->b = p->w_t + off + (size_t)in * ld;
        dst->in = in; dst->out = out; dst->ld = ld;
    };
    const float *src = flat;
    for (const LayerSpec &l : cn_layers(p->d, p->w)) {
        const float *w = src, *b = src + (size_t)l.in * l.out;
        if (l.dst_hh) {                                   // weight_ih_l0, weight_hh_l0, bias_ih_l0, bias_hh_l0
            const int h = l.out / 4;
            const float *w_hh = b;
            b = w_hh + (size_t)l.out * h;
            put(l.in, l.out, w, b, l.dst);
            put(h, l.out, w_hh, b + l.out, l.dst_hh);
        } else {
            put(l.in, l.out, w, b, l.dst);
        }
        src += cn_layer_floats(l);
    }
    CN_CUDA_CHECK(cudaMemcpyAsync(p->w_t, t.data(), sizeof(float) * t.size(), cudaMemcpyHostToDevice, s));
    CN_CUDA_CHECK(cudaMemcpyAsync(p->w_raw, flat, sizeof(float) * n, cudaMemcpyHostToDevice, s));
    CN_CUDA_CHECK(cudaStreamSynchronize(s));  // `t` and `flat` may go away after return
    if (p->cfg.precision == CN_PREC_F16_TC) {
        int rc = cn_tc_load_weights(p, flat, s);
        if (rc) return rc;
    }
    p->weights_loaded = 1;
    return CN_OK;
}

int cn_policy_action_table(cn_policy *p, double *out_xy_host, int32_t *n_actions)
{
    if (!p) { cn_set_error("null policy"); return CN_EINVAL; }
    if (out_xy_host) memcpy(out_xy_host, p->action_host, sizeof(double) * 2 * p->d.A);
    if (n_actions) *n_actions = p->d.A;
    return CN_OK;
}

static int check_pair(cn_policy *p, cn_env *env)
{
    if (!p || !env) { cn_set_error("null handle"); return CN_EINVAL; }
    if (p->device != env->device) { cn_set_error("policy and env live on different devices"); return CN_EINVAL; }
    if (!p->weights_loaded) { cn_set_error("cn_policy_load_weights has not been called"); return CN_EINVAL; }
    if (p->cfg.kinematics != env->p.kinematics) {
        cn_set_error("policy kinematics (%d) and env robot_kinematics (%d) differ", p->cfg.kinematics, env->p.kinematics);
        return CN_EINVAL;
    }
    return CN_OK;
}

// the lookahead of the policy's precision; tail: see cn_lookahead_tc (the FP32 lookahead runs on s alone)
static int lookahead(cn_policy *p, cn_env *env, int query_env, double epsilon, cudaStream_t s, cudaStream_t tail = nullptr)
{
    if (p->cfg.precision == CN_PREC_F16_TC) return cn_lookahead_tc(p, env, query_env, epsilon, s, tail);
    return cn_lookahead_f32(p, env, query_env, epsilon, s);
}

// waits for s, then refuses the last lookahead when some env had no finite value (multi_human_rl.py:57-58)
static int sync_and_check_values(cn_policy *p, cudaStream_t s)
{
    int32_t bad = 0;
    CN_CUDA_CHECK(cudaMemcpyAsync(&bad, p->bad_flag, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CN_CUDA_CHECK(cudaStreamSynchronize(s));
    if (bad) { cn_set_error("Value network is not well trained. "); return CN_EVALUE; }
    return CN_OK;
}

int cn_policy_lookahead(cn_policy *p, cn_env *env, int query_env, double epsilon, void *stream)
{
    int rc = check_pair(p, env);
    if (rc) return rc;
    CN_CUDA_CHECK(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    if (query_env && !env->orca_valid) {
        cn_set_error("query_env lookahead needs cn_env_orca for the current state");
        return CN_EINVAL;
    }
    return lookahead(p, env, query_env, epsilon, s);
}

int cn_policy_read(cn_policy *p, cn_env *env, int32_t *best_idx, double *values, void *stream)
{
    int rc = check_pair(p, env);
    if (rc) return rc;
    CN_CUDA_CHECK(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    const size_t E = env->p.d.E;
    if (best_idx) CN_CUDA_CHECK(cudaMemcpyAsync(best_idx, env->action_idx, sizeof(int32_t) * E, cudaMemcpyDeviceToHost, s));
    if (values) {
        if (!p->values) { cn_set_error("no lookahead has been run"); return CN_EINVAL; }
        CN_CUDA_CHECK(cudaMemcpyAsync(values, p->values, sizeof(double) * E * p->d.A, cudaMemcpyDeviceToHost, s));
    }
    return sync_and_check_values(p, s);
}

int cn_policy_bad_count(cn_policy *p, int64_t *count, int reset, void *stream)
{
    if (!p || !count) { cn_set_error("null argument"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    int32_t n = 0;
    CN_CUDA_CHECK(cudaMemcpyAsync(&n, p->bad_flag + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (reset) CN_CUDA_CHECK(cudaMemsetAsync(p->bad_flag + 1, 0, sizeof(int32_t), s));
    CN_CUDA_CHECK(cudaStreamSynchronize(s));
    *count = n;
    return CN_OK;
}

int cn_policy_transform(cn_policy *p, cn_env *env, float *out_dev, void *stream)
{
    if (!p || !env || !out_dev) { cn_set_error("null argument"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(p->device));
    return cn_transform_f32(p, env, out_dev, 0, (cudaStream_t)stream);
}

int cn_policy_last_state(cn_policy *p, cn_env *env, float *out_dev, void *stream)
{
    if (!p || !env || !out_dev) { cn_set_error("null argument"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(p->device));
    return cn_transform_f32(p, env, out_dev, p->cfg.network == CN_NET_LSTM_RL ? 1 : 0, (cudaStream_t)stream);
}

int cn_policy_forward(cn_policy *p, const float *x_dev, int32_t batch, int32_t human_num, float *out_dev, void *stream)
{
    if (!p || !x_dev || !out_dev) { cn_set_error("null argument"); return CN_EINVAL; }
    if (!p->weights_loaded) { cn_set_error("cn_policy_load_weights has not been called"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(p->device));
    return cn_forward_f32(p, x_dev, batch, human_num, out_dev, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------
// fused hot path
// ---------------------------------------------------------------------------------------------

// tail: stream that takes over after the row kernel (nullptr = stay on s); on return *cur is the stream the step ended on
static int rollout_step_impl(cn_policy *p, cn_env *env, int query_env, double epsilon, cudaStream_t s, cudaStream_t tail,
                             cudaStream_t *cur);

int cn_rollout_step(cn_policy *p, cn_env *env, int query_env, double epsilon, void *stream)
{
    int rc = check_pair(p, env);
    if (rc) return rc;
    CN_CUDA_CHECK(cudaSetDevice(p->device));
    cudaStream_t cur;
    return rollout_step_impl(p, env, query_env, epsilon, (cudaStream_t)stream, nullptr, &cur);
}

static int ensure_tail_stream(cn_env *env)
{
    if (env->tail_stream) return CN_OK;
    int lo = 0, hi = 0;
    CN_CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    CN_CUDA_CHECK(cudaStreamCreateWithPriority(&env->tail_stream, cudaStreamNonBlocking, hi));
    CN_CUDA_CHECK(cudaEventCreateWithFlags(&env->ev_rows, cudaEventDisableTiming));
    CN_CUDA_CHECK(cudaEventCreateWithFlags(&env->ev_tail, cudaEventDisableTiming));
    return CN_OK;
}

int cn_rollout_step_sharded(cn_policy *p, cn_env *env, int query_env, double epsilon, void *stream)
{
    int rc = check_pair(p, env);
    if (rc) return rc;
    CN_CUDA_CHECK(cudaSetDevice(p->device));
    if ((rc = ensure_tail_stream(env))) return rc;
    cudaStream_t s0 = (cudaStream_t)stream, cur = s0;
    if ((rc = rollout_step_impl(p, env, query_env, epsilon, s0, env->tail_stream, &cur))) return rc;
    if (cur != s0) {
        CN_CUDA_CHECK(cudaEventRecord(env->ev_tail, cur));
        CN_CUDA_CHECK(cudaStreamWaitEvent(s0, env->ev_tail, 0));
    }
    return CN_OK;
}

static int rollout_step_impl(cn_policy *p, cn_env *env, int query_env, double epsilon, cudaStream_t s, cudaStream_t tail,
                             cudaStream_t *cur)
{
    int rc = CN_OK;
    if (p->cfg.precision != CN_PREC_F16_TC) tail = nullptr;
    // query_env = 0: the lookahead propagates humans with their current velocity (cadrl.py:107-109) and never reads
    // the ORCA result, so ORCA (a latency-bound 16 us kernel) runs on a forked stream beside the lookahead and joins
    // before the env step.  Event fork/join keeps the whole step capturable in a CUDA graph.
    const bool fork = !query_env;
    cn_trace_mark("orca", s);
    if (fork) {
        if (!env->side_stream) {
            CN_CUDA_CHECK(cudaStreamCreateWithFlags(&env->side_stream, cudaStreamNonBlocking));
            CN_CUDA_CHECK(cudaEventCreateWithFlags(&env->ev_fork, cudaEventDisableTiming));
            CN_CUDA_CHECK(cudaEventCreateWithFlags(&env->ev_join, cudaEventDisableTiming));
        }
        CN_CUDA_CHECK(cudaEventRecord(env->ev_fork, s));
        CN_CUDA_CHECK(cudaStreamWaitEvent(env->side_stream, env->ev_fork, 0));
        if ((rc = cn_launch_orca(env, env->side_stream))) return rc;
        CN_CUDA_CHECK(cudaEventRecord(env->ev_join, env->side_stream));
    } else if ((rc = cn_launch_orca(env, s))) return rc;
    if ((rc = lookahead(p, env, query_env, epsilon, s, tail))) return rc;
    if (tail) s = tail;
    *cur = s;
    if (fork) CN_CUDA_CHECK(cudaStreamWaitEvent(s, env->ev_join, 0));
    cn_trace_mark("step", s);
    if ((rc = cn_launch_step(env, nullptr, 1, s, env->p.auto_reset ? 1 : 0))) return rc;     // auto-reset fused into the step
    cn_trace_mark("step_done", s);
    return rc;
}

// ---------------------------------------------------------------------------------------------
// whole episodes: the explorer's loop (explorer.py:53-69) enqueued natively
// ---------------------------------------------------------------------------------------------

static __global__ void count_active_kernel(int E, const uint8_t *__restrict__ frozen, int32_t *__restrict__ out)
{
    __shared__ int total;
    if (threadIdx.x == 0) total = 0;
    __syncthreads();
    int n = 0;
    for (int e = threadIdx.x; e < E; e += blockDim.x) n += frozen[e] ? 0 : 1;
    for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
    if ((threadIdx.x & 31) == 0 && n) atomicAdd(&total, n);
    __syncthreads();
    if (threadIdx.x == 0) *out = total;
}

int cn_rollout_episodes(cn_policy *p, cn_env *env, cn_world *world, int robot_mode, double safety_space, int query_env,
                        double epsilon, int32_t max_steps, int32_t check_every, const cn_rollout_record *rec,
                        int32_t *steps_run, void *stream)
{
    if (!env || !steps_run) { cn_set_error("null argument"); return CN_EINVAL; }
    if (robot_mode < CN_ROBOT_POLICY || robot_mode > CN_ROBOT_KEEP) { cn_set_error("robot_mode %d", robot_mode); return CN_EINVAL; }
    if (max_steps < 0 || check_every < 1) { cn_set_error("max_steps >= 0 and check_every >= 1"); return CN_EINVAL; }
    if (env->p.auto_reset) {
        cn_set_error("cn_rollout_episodes runs ONE episode per env: create the env with auto_reset = 0");
        return CN_EINVAL;
    }
    int rc;
    if (robot_mode == CN_ROBOT_POLICY) {
        if ((rc = check_pair(p, env))) return rc;
    }
    cn_policy *tp = rec ? rec->transform_policy : nullptr;
    if (rec && (!tp || !rec->states_dev || !rec->reward_dev || !rec->done_dev)) {
        cn_set_error("cn_rollout_record needs transform_policy, states_dev, reward_dev and done_dev");
        return CN_EINVAL;
    }
    if (tp && tp->device != env->device) { cn_set_error("transform policy and env live on different devices"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(env->device));
    cudaStream_t s = (cudaStream_t)stream;
    if (!env->active_dev) {
        CN_CUDA_CHECK(cudaMalloc(&env->active_dev, 2 * sizeof(int32_t)));
        CN_CUDA_CHECK(cudaMallocHost(&env->active_host, 2 * sizeof(int32_t)));
        for (cudaEvent_t &ev : env->ev_active) CN_CUDA_CHECK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    }
    const size_t E = env->p.d.E;
    const size_t state_floats = tp ? E * (size_t)env->p.d.H * (size_t)tp->cfg.input_dim : 0;
    int slot = 0, pending = -1;
    *steps_run = 0;
    for (int step = 0; step < max_steps; ++step) {
        if (tp) {
            // policy.last_state = transform(state) (multi_human_rl.py:60-61) / target_policy.transform(state) (explorer.py:163)
            const int sorted = rec->last_state && tp->cfg.network == CN_NET_LSTM_RL;
            if ((rc = cn_transform_f32(tp, env, rec->states_dev + (size_t)step * state_floats, sorted, s))) return rc;
        }
        if (robot_mode == CN_ROBOT_POLICY && !world) {
            cudaStream_t cur;
            if ((rc = rollout_step_impl(p, env, query_env, epsilon, s, nullptr, &cur))) return rc;
        } else {
            if (world) rc = cn_world_predict(world, env, s);
            else rc = cn_launch_orca(env, s);
            if (rc) return rc;
            if (robot_mode == CN_ROBOT_POLICY)
                rc = lookahead(p, env, query_env, epsilon, s);
            else if (robot_mode == CN_ROBOT_ORCA) rc = cn_launch_robot_orca(env, safety_space, s);
            if (rc) return rc;
            if ((rc = cn_launch_step(env, nullptr, 1, s, 0))) return rc;
        }
        if (rec) {
            CN_CUDA_CHECK(cudaMemcpyAsync(rec->reward_dev + (size_t)step * E, env->reward, sizeof(double) * E, cudaMemcpyDeviceToDevice, s));
            CN_CUDA_CHECK(cudaMemcpyAsync(rec->done_dev + (size_t)step * E, env->done, E, cudaMemcpyDeviceToDevice, s));
        }
        *steps_run = step + 1;
        if ((step + 1) % check_every == 0) {
            // the count enqueued one interval ago has (all but certainly) arrived: waiting for it does not drain the stream
            if (pending >= 0) {
                CN_CUDA_CHECK(cudaEventSynchronize(env->ev_active[pending]));
                if (env->active_host[pending] == 0) break;
            }
            count_active_kernel<<<1, 256, 0, s>>>((int)E, env->frozen, env->active_dev + slot);
            CN_CUDA_CHECK(cudaGetLastError());
            g_cn_launches.fetch_add(1);
            CN_CUDA_CHECK(cudaMemcpyAsync(env->active_host + slot, env->active_dev + slot, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
            CN_CUDA_CHECK(cudaEventRecord(env->ev_active[slot], s));
            pending = slot;
            slot ^= 1;
        }
    }
    return CN_OK;
}

int cn_rollout_step_host(cn_policy *p, cn_env *env, int query_env, double epsilon, const double *agents_in,
                         const double *times_in, double *agents_out, double *times_out, double *reward, uint8_t *done,
                         uint8_t *info, int32_t *action_idx, void *stream)
{
    int rc = check_pair(p, env);
    if (rc) return rc;
    CN_CUDA_CHECK(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    const size_t E = env->p.d.E, A1 = env->p.d.A1;
    if (agents_in) {
        CN_CUDA_CHECK(cudaMemcpyAsync(env->stage, agents_in, sizeof(double) * E * A1 * F_COUNT, cudaMemcpyHostToDevice, s));
        // unlike cn_env_set_state this keeps the per-episode accumulators: it is one step of a running episode
        if ((rc = cn_launch_pack_keep(env, s))) return rc;
    }
    if (times_in) CN_CUDA_CHECK(cudaMemcpyAsync(env->time, times_in, sizeof(double) * E, cudaMemcpyHostToDevice, s));
    if ((rc = cn_rollout_step(p, env, query_env, epsilon, s))) return rc;
    if (agents_out) {
        if ((rc = cn_launch_pack(env, 0, s))) return rc;
        CN_CUDA_CHECK(cudaMemcpyAsync(agents_out, env->stage, sizeof(double) * E * A1 * F_COUNT, cudaMemcpyDeviceToHost, s));
    }
    if (times_out) CN_CUDA_CHECK(cudaMemcpyAsync(times_out, env->time, sizeof(double) * E, cudaMemcpyDeviceToHost, s));
    if (reward) CN_CUDA_CHECK(cudaMemcpyAsync(reward, env->reward, sizeof(double) * E, cudaMemcpyDeviceToHost, s));
    if (done) CN_CUDA_CHECK(cudaMemcpyAsync(done, env->done, E, cudaMemcpyDeviceToHost, s));
    if (info) CN_CUDA_CHECK(cudaMemcpyAsync(info, env->info, E, cudaMemcpyDeviceToHost, s));
    if (action_idx) CN_CUDA_CHECK(cudaMemcpyAsync(action_idx, env->action_idx, sizeof(int32_t) * E, cudaMemcpyDeviceToHost, s));
    return sync_and_check_values(p, s);
}

int64_t cn_host_step_bytes(const cn_env *env, int out)
{
    if (!env) return 0;
    const int64_t E = env->p.d.E, A1 = env->p.d.A1;
    const int64_t in = 8 * (E * A1 * F_COUNT + E);
    return out ? in + 8 * E + 4 * E + E + E : in;
}

static int rollout_step_host_packed(cn_policy *p, cn_env *env, int query_env, double epsilon, const void *host_in,
                                    void *host_out, void *stream, bool sync)
{
    int rc = check_pair(p, env);
    if (rc) return rc;
    if (!host_in || !host_out) { cn_set_error("host_in / host_out must not be null"); return CN_EINVAL; }
    CN_CUDA_CHECK(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    if (!env->io_block) CN_CUDA_CHECK(cudaMalloc((void **)&env->io_block, (size_t)cn_host_step_bytes(env, 1) + 16));
    cn_trace_mark("h2d", s);
    CN_CUDA_CHECK(cudaMemcpyAsync(env->io_block, host_in, (size_t)cn_host_step_bytes(env, 0), cudaMemcpyHostToDevice, s));
    cn_trace_mark("unpack", s);
    if ((rc = cn_launch_io(env, env->io_block, 1, s))) return rc;          // keeps the per-episode accumulators
    cudaStream_t tail = nullptr;
    if (!sync) {
        // non-blocking form = one shard of a pipelined host loop: everything after the row kernel runs at high priority
        if ((rc = ensure_tail_stream(env))) return rc;
        tail = env->tail_stream;
    }
    cudaStream_t s0 = s;
    if ((rc = rollout_step_impl(p, env, query_env, epsilon, s, tail, &s))) return rc;
    if ((rc = cn_launch_io(env, env->io_block, 0, s))) return rc;
    cn_trace_mark("d2h", s);
    CN_CUDA_CHECK(cudaMemcpyAsync(host_out, env->io_block, (size_t)cn_host_step_bytes(env, 1), cudaMemcpyDeviceToHost, s));
    cn_trace_mark("d2h_done", s);
    if (s != s0) {                       // the caller's stream stays the one handle on the whole step
        CN_CUDA_CHECK(cudaEventRecord(env->ev_tail, s));
        CN_CUDA_CHECK(cudaStreamWaitEvent(s0, env->ev_tail, 0));
        s = s0;
    }
    return sync ? sync_and_check_values(p, s) : CN_OK;
}

int cn_rollout_step_host_packed(cn_policy *p, cn_env *env, int query_env, double epsilon, const void *host_in, void *host_out,
                                void *stream)
{
    return rollout_step_host_packed(p, env, query_env, epsilon, host_in, host_out, stream, true);
}

int cn_rollout_step_host_packed_async(cn_policy *p, cn_env *env, int query_env, double epsilon, const void *host_in,
                                      void *host_out, void *stream)
{
    return rollout_step_host_packed(p, env, query_env, epsilon, host_in, host_out, stream, false);
}

int cn_stream_sync(int device, void *stream)
{
    CN_CUDA_CHECK(cudaSetDevice(device));
    CN_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
    return CN_OK;
}

}  // extern "C"
