// lookahead_tc.cu -- SARL one-step lookahead on tcgen05 tensor cores (CN_PREC_F16_TC): host side (weight images,
// launch sequence) of the three kernels in tc_rows_pair.cuh / tc_mlp3_pair.cuh, plus the UMMA self-tests.
//
// fp16 operands, fp32 accumulation in TMEM, cta_group::2 UMMAs (M = 256 over the two SMs of a CTA pair):
//
//  tc_features_kernel   rows = (env, action, human): propagate + reward + rotate -> X tiles (13 features, split hi+lo
//       fp16 so layer 1 sees ~22-bit inputs), lookahead rewards, self-state chunks of the joint state J
//  tc_rows_pair_kernel  per 128-row tile, all on chip:
//       mlp1.0 -> mlp1.2 -> {mlp2.0 -> mlp2.2 ; attention.0 on [mlp1_out | group mean] (or on mlp1_out alone without the
//       global state) -> attention.2}
//       attention.4 (fp32 dot) -> masked softmax over the humans of a group -> weighted feature
//       -> joint state J (fp16, 160 B per (env, action)) to HBM, already in UMMA operand order
//  tc_mlp3_pair_kernel  rows = (env, action).  mlp3.0 -> .2 -> .4 on tensor cores, .6 as an fp32 dot,
//       value = reward + gamma_bar * V  -> values[E][A]; the shared argmax kernel follows.
//
// Biases ride inside the GEMMs: every activation tile carries two constant-one columns and the weight
// images hold bias_hi / bias_lo (fp16 split) in the matching K rows, so epilogues are pure
// tcgen05.ld -> cvt.rn.relu.f16x2 -> st.shared / tcgen05.st.
//
// Reference (file:line relative to the reference root): see lookahead_f32.cu; the network is
// crowd_nav/policy/sarl.py:28-65 with the default [sarl] dims of crowd_nav/configs/policy.config:41-49.
#include "env_math.cuh"
#include "umma.cuh"

#include <cuda_fp16.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

int cn_lookahead_prepare(cn_policy *p, cn_env *env, cudaStream_t s);
int cn_lookahead_argmax(cn_policy *p, cn_env *env, double epsilon, cudaStream_t s, bool pdl);

namespace {

using namespace umma;

// ---- padded GEMM shapes (default SARL dims) ---------------------------------------------------------
constexpr int K_X = 32;     // 13 hi | 1 1 0 | 13 lo | 0 0 0
constexpr int N_H1 = 160;   // 150 + ones(150,151)
constexpr int N_M1 = 112;   // 100 + ones(100,101)
constexpr int N_F = 64;     // 50
constexpr int K_A1 = 224;   // [mlp1_out 112 | group mean 112]
constexpr int K_J = 80;     // 50 weighted | 6 pad | 6 self_hi 1 1 | 6 self_lo 0 0 | 8 pad
constexpr int ROWS = 128;

__host__ __device__ constexpr uint32_t bytes_of(int rows, int K) { return (uint32_t)rows * K * 2; }
// full (unsplit) weight image of the row network; split_rows() cuts it into the two per-CTA halves
constexpr uint32_t OFF_W1 = 0;
constexpr uint32_t OFF_W2 = OFF_W1 + bytes_of(N_H1, K_X);
constexpr uint32_t OFF_W3 = OFF_W2 + bytes_of(N_M1, N_H1);
constexpr uint32_t OFF_W4 = OFF_W3 + bytes_of(N_M1, N_M1);
constexpr uint32_t OFF_WA1 = OFF_W4 + bytes_of(N_F, N_M1);
constexpr uint32_t OFF_WA2 = OFF_WA1 + bytes_of(N_M1, K_A1);
constexpr uint32_t IMG_A_BYTES = OFF_WA2 + bytes_of(N_M1, N_M1);
constexpr uint32_t TAIL_BYTES = 416;   // fp32 tail of a 100 -> 1 layer: weight[100], bias, 3 pad
// full weight image of mlp3
constexpr uint32_t OFF_M1 = 0;
constexpr uint32_t OFF_M2 = OFF_M1 + bytes_of(N_H1, K_J);
constexpr uint32_t OFF_M3 = OFF_M2 + bytes_of(N_M1, N_H1);
constexpr uint32_t IMG_B_BYTES = OFF_M3 + bytes_of(N_M1, N_M1);

constexpr uint32_t J_TILE_BYTES = bytes_of(ROWS, K_J);

struct TcState {
    uint8_t *img_pair;        // two half images of the row network for tc_rows_pair_kernel (rank 0 | rank 1)
    long long *dbg;           // optional phase timestamps of CTA 0 (cn_debug_tc_timing)
    uint8_t *X;               // layer-1 operand tiles of the CTA-pair path (tc_features_kernel -> tc_rows_pair_kernel)
    size_t cap_xtiles;
    uint8_t *J;               // joint-state tiles, zero-initialised (the mlp3 kernel reads whole rounds of tiles)
    size_t cap_jtiles;
    double *rew;              // NG rewards
    size_t cap_rew;
    int num_sms;
    float tail_a[104];        // attention.4 weight[100] + bias (kernel parameter of tc_rows_pair_kernel)
    float tail_b[104];        // mlp3.6 weight[100] + bias (kernel parameter of tc_mlp3_pair_kernel)
    uint8_t *img_pair_b;      // two half images of mlp3 for tc_mlp3_pair_kernel
    float *rowv;              // CADRL: one value per (env, action, human) row (tc_mlp3_pair_kernel<1> -> cadrl_min_kernel)
    size_t cap_rowv;
    uint8_t *img_lstm;        // LSTM-RL: two half images [W_ih | W_hh] of tc_lstm_pair_kernel
    uint8_t *XL;              // LSTM-RL: X_t operand tiles, (tile, step) major
    size_t cap_xl;
    int32_t *ord;             // LSTM-RL: predict()'s human order per env
    size_t cap_ord;
    float *omP;               // with_om: mlp1.0's occupancy-map product per (env, human), N_H1 floats each (tc_om_bias_kernel)
    size_t cap_om;
    int ktime_on;             // cn_debug_kernel_ms: CUDA events around each kernel of the lookahead, on the launching stream
    cudaEvent_t kev[5];       // before features | before the middle stage | before scoring | before argmax | after argmax
};

__device__ __forceinline__ void copy_image_to_smem(uint8_t *dst, const uint8_t *__restrict__ src, uint32_t bytes)
{
    for (uint32_t i = threadIdx.x * 16; i < bytes; i += blockDim.x * 16)
        *reinterpret_cast<uint4 *>(dst + i) = __ldg(reinterpret_cast<const uint4 *>(src + i));
}

__device__ __forceinline__ uint32_t h2(float lo, float hi) { return pack_f16x2(lo, hi); }

// split x into fp16 hi + fp16 lo (x ~ hi + lo to ~22 bits)
__device__ __forceinline__ void split_hl(float x, float &hi, float &lo)
{
    hi = __half2float(__float2half_rn(x));
    lo = x - hi;
}

#include "tc_rows_pair.cuh"
#include "tc_mlp3_pair.cuh"
#include "tc_lstm_pair.cuh"

// tc_rows_pair_kernel<HT, OM, GS> as kRowsKernels[!GS][OM][HT = 0, 5, 10]
using RowsKernel = decltype(&tc_rows_pair_kernel<0, false, true>);
constexpr RowsKernel kRowsKernels[2][2][3] = {
    {{tc_rows_pair_kernel<0, false, true>, tc_rows_pair_kernel<5, false, true>, tc_rows_pair_kernel<10, false, true>},
     {tc_rows_pair_kernel<0, true, true>, tc_rows_pair_kernel<5, true, true>, tc_rows_pair_kernel<10, true, true>}},
    {{tc_rows_pair_kernel<0, false, false>, tc_rows_pair_kernel<5, false, false>, tc_rows_pair_kernel<10, false, false>},
     {tc_rows_pair_kernel<0, true, false>, tc_rows_pair_kernel<5, true, false>, tc_rows_pair_kernel<10, true, false>}}};

// =====================================================================================================
// self-test kernel: D[128 x N] = A[128 x K] * B[N x K]^T
// =====================================================================================================
__global__ void __launch_bounds__(128, 1)
umma_selftest_kernel(const uint8_t *__restrict__ a_img, const uint8_t *__restrict__ b_img, float *__restrict__ d,
                     int N, int K, int mode /*0 SS, 1 SS with MN-major B, 2 TS (A in TMEM)*/)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5;
    const uint32_t a_bytes = bytes_of(ROWS, K), b_bytes = mode == 1 ? bytes_of(ROWS, N) : bytes_of(N, K);
    uint8_t *sa = smem, *sb = smem + a_bytes;
    uint8_t *misc = smem + ((a_bytes + b_bytes + 15) & ~15u);
    const uint32_t mbar = smem_u32(misc);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(misc + 8);
    copy_image_to_smem(sa, a_img, a_bytes);
    copy_image_to_smem(sb, b_img, b_bytes);
    if (tid == 0) { mbar_init(mbar, 1); fence_mbar_init(); }
    if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 512);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tlane = tmem + ((uint32_t)(warp * 32) << 16);
    constexpr uint32_t T_A = 256;          // TS mode: the packed fp16 A operand lives at TMEM column 256
    if (mode == 2) {
        // row `tid` of A: K/2 packed words, 8 per tcgen05.st
        for (int c8 = 0; c8 < K / 16; ++c8) {
            uint32_t w[8];
            for (int j = 0; j < 8; ++j) {
                const int k = c8 * 16 + 2 * j;   // element k lives in chunk k/8 at position k%8
                const __half2 h = *reinterpret_cast<const __half2 *>(sa + chunk_off(ROWS, tid, k >> 3) + (k & 7) * 2);
                w[j] = *reinterpret_cast<const uint32_t *>(&h);
            }
            st8(tlane + T_A + c8 * 8, w);
        }
        wait_st();
        fence_before_sync();
        __syncthreads();
        fence_after_sync();
    }
    if (tid == 0) {
        if (mode == 1) mma_layer_bmn(tmem, smem_u32(sa), ROWS, smem_u32(sb), K, N, false);
        else if (mode == 2) mma_layer_ts(tmem, tmem + T_A, smem_u32(sb), N, K, N, false);
        else mma_layer(tmem, smem_u32(sa), ROWS, smem_u32(sb), N, K, N, false);
        commit(mbar);
    }
    mbar_wait(mbar, 0);
    fence_after_sync();
    for (int c0 = 0; c0 < N; c0 += 16) {
        uint32_t v[16];
        ld16(tlane + c0, v);
        wait_ld();
        for (int k = 0; k < 16; ++k) d[(size_t)tid * N + c0 + k] = __uint_as_float(v[k]);
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

// CADRL scoring (cadrl.py:166-168): value = reward + gamma_bar * min over the humans of the group of the per-row network outputs
__global__ void cadrl_min_kernel(EnvParams p, const double *__restrict__ st, const float *__restrict__ rowv,
                                 const double *__restrict__ rew, int A, int NG, int G, int H, double gamma, double gamma_bar_host,
                                 double v_pref_host, double *__restrict__ values)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= NG) return;
    const size_t r0 = (size_t)(g / G) * ROWS + (size_t)(g % G) * H;
    float m = rowv[r0];
    for (int h = 1; h < H; ++h) m = fminf(m, rowv[r0 + h]);
    const double vp = st[st_idx(p.d, F_VPREF, 0, g / A)];
    const double gamma_bar = (vp == v_pref_host) ? gamma_bar_host : pow(gamma, p.time_step * vp);
    values[g] = rew[g] + gamma_bar * (double)m;
}

// ---- host-side weight images ------------------------------------------------------------------------
struct HostLinear { const float *w, *b; int in, out; };

inline void put(std::vector<uint8_t> &img, uint32_t base, int R, int r, int k, float v)
{
    const __half h = __float2half_rn(v);
    memcpy(&img[base + chunk_off(R, r, k >> 3) + (k & 7) * 2], &h, 2);
}
inline float f16r(float v) { return __half2float(__float2half_rn(v)); }

// generic layer: rows n < out get W[n][k] at K index kmap(k), bias hi/lo at kb/kb+1; ones columns at
// output rows (ones_n, ones_n+1) fed from K index kb (which holds 1.0 in the activation tile)
void fill_layer(std::vector<uint8_t> &img, uint32_t base, int R, const HostLinear &L, int k_in0, int n_in, int k_dst0,
                int kb, int ones_n)
{
    for (int n = 0; n < L.out; ++n) {
        for (int k = 0; k < n_in; ++k) put(img, base, R, n, k_dst0 + k, L.w[(size_t)n * L.in + k_in0 + k]);
        if (kb >= 0) {
            const float bh = f16r(L.b[n]);
            put(img, base, R, n, kb, bh);
            put(img, base, R, n, kb + 1, L.b[n] - bh);
        }
    }
    if (ones_n >= 0 && kb >= 0) { put(img, base, R, ones_n, kb, 1.0f); put(img, base, R, ones_n + 1, kb, 1.0f); }
}

// rows [rank N/2, (rank+1) N/2) of a chunked K-major [N x K] image -> chunked K-major [N/2 x K]
void split_rows(uint8_t *dst, const uint8_t *src, int N, int K, int rank)
{
    const int hn = N / 2;
    for (int c = 0; c < K / 8; ++c)
        memcpy(dst + (size_t)c * hn * 16, src + (size_t)c * N * 16 + (size_t)rank * hn * 16, (size_t)hn * 16);
}

// fp32 tail of a 100 -> 1 output layer (kernel parameter TailW): weight[100], bias at [100]
void fill_tail(const HostLinear &L, float *tail)
{
    memset(tail, 0, TAIL_BYTES);
    for (int k = 0; k < 100; ++k) tail[k] = L.w[k];
    tail[100] = L.b[0];
}

// The row network (mlp1, mlp2, attention: L[0..6]) as the two half images of tc_rows_pair_kernel (CTA `rank` holds output
// rows [rank N/2, (rank+1) N/2) of every layer); attention.4 goes to `tail`.  gs = false: attention.0 has only the 100
// mlp1_out columns (sarl.py:40-47) and the group-mean half H_WB stays empty (tc_rows_pair_kernel<.., .., false> never reads it).
std::vector<uint8_t> rows_image(const HostLinear *L, bool gs, float *tail)
{
    std::vector<uint8_t> a(IMG_A_BYTES, 0);
    // mlp1.0: K = [x_hi(13) 1 1 0 | x_lo(13) 0 0 0]; bias at k = 13,14; ones -> n = 150,151
    fill_layer(a, OFF_W1, N_H1, L[0], 0, 13, 0, 13, 150);
    fill_layer(a, OFF_W1, N_H1, L[0], 0, 13, 16, -1, -1);
    fill_layer(a, OFF_W2, N_M1, L[1], 0, 150, 0, 150, 100);          // mlp1.2
    fill_layer(a, OFF_W3, N_M1, L[2], 0, 100, 0, 100, 100);          // mlp2.0
    fill_layer(a, OFF_W4, N_F, L[3], 0, 100, 0, 100, -1);            // mlp2.2 (no ones needed downstream)
    fill_layer(a, OFF_WA1, N_M1, L[4], 0, 100, 0, 100, 100);         // attention.0, mlp1_out half
    if (gs) fill_layer(a, OFF_WA1, N_M1, L[4], 100, 100, N_M1, -1, -1);   //          group-mean half
    fill_layer(a, OFF_WA2, N_M1, L[5], 0, 100, 0, 100, -1);          // attention.2
    fill_tail(L[6], tail);
    std::vector<uint8_t> hp(2 * IMG_H_BYTES, 0);
    for (int rank = 0; rank < 2; ++rank) {
        uint8_t *h = hp.data() + (size_t)rank * IMG_H_BYTES;
        split_rows(h + H_W1, a.data() + OFF_W1, N_H1, K_X, rank);
        split_rows(h + H_W2, a.data() + OFF_W2, N_M1, N_H1, rank);
        // stage 2 is ONE N = 224 UMMA: rank 0's half = attention.0 (mlp1_out half of K) -> D [0,112), rank 1's = mlp2.0 -> [112,224)
        memcpy(h + H_W3A, rank == 0 ? a.data() + OFF_WA1 : a.data() + OFF_W3, bytes_of(N_M1, N_M1));
        if (gs) split_rows(h + H_WB, a.data() + OFF_WA1 + bytes_of(N_M1, N_M1), N_M1, N_M1, rank);   // group-mean half of K
        split_rows(h + H_W4, a.data() + OFF_W4, N_F, N_M1, rank);
        split_rows(h + H_WA2, a.data() + OFF_WA2, N_M1, N_M1, rank);
        memcpy(h + H_TAIL, tail, TAIL_BYTES);      // copied to shared memory by the kernel, which reads the TailW parameter
    }
    return hp;
}

// A 150, 100, 100, 1 mlp (M[0..3]) as the two half images of tc_mlp3_pair_kernel; the last layer goes to `tail`.  Stage 0 reads
// the X tiles (x_input: CADRL's value network on every row) or the joint-state tiles J (SARL's mlp3, LSTM-RL's mlp).
std::vector<uint8_t> mlp3_image(const HostLinear *M, bool x_input, float *tail)
{
    std::vector<uint8_t> b(IMG_B_BYTES, 0);
    if (x_input) {
        // X = [x_hi(13) 1 1 0 | x_lo(13) 0 0 0]: bias at k = 13, 14; ones -> n = 150, 151
        fill_layer(b, OFF_M1, N_H1, M[0], 0, 13, 0, 13, 150);
        fill_layer(b, OFF_M1, N_H1, M[0], 0, 13, 16, -1, -1);
    } else {
        // J = [weighted or h_n(50) pad6 | self_hi(6) 1 1 | self_lo(6) 0 0 | pad8]; torch input = [self(6), weighted or h_n(50)]
        fill_layer(b, OFF_M1, N_H1, M[0], 6, 50, 0, -1, -1);
        fill_layer(b, OFF_M1, N_H1, M[0], 0, 6, 56, 62, 150);
        fill_layer(b, OFF_M1, N_H1, M[0], 0, 6, 64, -1, -1);
    }
    fill_layer(b, OFF_M2, N_M1, M[1], 0, 150, 0, 150, 100);
    fill_layer(b, OFF_M3, N_M1, M[2], 0, 100, 0, 100, -1);
    fill_tail(M[3], tail);
    std::vector<uint8_t> hb(2 * IMG_HM_BYTES, 0);
    for (int rank = 0; rank < 2; ++rank) {
        uint8_t *h = hb.data() + (size_t)rank * IMG_HM_BYTES;
        split_rows(h + HM_M1, b.data() + OFF_M1, N_H1, K_J, rank);
        split_rows(h + HM_M2, b.data() + OFF_M2, N_M1, N_H1, rank);
        split_rows(h + HM_M3, b.data() + OFF_M3, N_M1, N_M1, rank);
    }
    return hb;
}

// LSTM-RL's LSTM block (lstm_rl.py:9-16: weight_ih_l0 [200][13], weight_hh_l0 [200][50], bias_ih_l0, bias_hh_l0 from src) as
// the two half images [W_ih | W_hh] of tc_lstm_pair_kernel
std::vector<uint8_t> lstm_image(const float *src)
{
    const int G4 = 4 * L_HIDDEN;
    const float *w_ih = src, *w_hh = w_ih + (size_t)G4 * 13, *b_ih = w_hh + (size_t)G4 * L_HIDDEN, *b_hh = b_ih + G4;
    // gate column n of the pair = half * 128 + gate * 32 + cl  <-  torch row gate * 50 + cell, cell = cl (half 0, cl < 24)
    // or 24 + cl (half 1, cl < 26); the other columns keep zero weights and bias (their cells stay at c = h = 0)
    std::vector<float> wi((size_t)N_LG * 13, 0.0f), wh((size_t)N_LG * L_HIDDEN, 0.0f), bb(N_LG, 0.0f);
    for (int n = 0; n < N_LG; ++n) {
        const int half = n / 128, gate = (n % 128) / 32, cl = n % 32;
        const int ncell = half ? L_HIDDEN - L_CELLS0 : L_CELLS0;
        if (cl >= ncell) continue;
        const int r = gate * L_HIDDEN + (half ? L_CELLS0 + cl : cl);
        memcpy(&wi[(size_t)n * 13], w_ih + (size_t)r * 13, sizeof(float) * 13);
        memcpy(&wh[(size_t)n * L_HIDDEN], w_hh + (size_t)r * L_HIDDEN, sizeof(float) * L_HIDDEN);
        bb[n] = b_ih[r] + b_hh[r];
    }
    const HostLinear Li = {wi.data(), bb.data(), 13, N_LG}, Lh = {wh.data(), bb.data(), L_HIDDEN, N_LG};
    std::vector<uint8_t> li(bytes_of(N_LG, K_X), 0), lh(bytes_of(N_LG, K_LH), 0);
    // X_t = [x_hi(13) 1 1 0 | x_lo(13) 0 0 0]: bias (b_ih + b_hh, hi / lo) at k = 13, 14
    fill_layer(li, 0, N_LG, Li, 0, 13, 0, 13, -1);
    fill_layer(li, 0, N_LG, Li, 0, 13, 16, -1, -1);
    // h = [h_hi(50) pad6 | h_lo(50) pad6]
    fill_layer(lh, 0, N_LG, Lh, 0, L_HIDDEN, 0, -1, -1);
    fill_layer(lh, 0, N_LG, Lh, 0, L_HIDDEN, 56, -1, -1);
    std::vector<uint8_t> hl(2 * IMG_HL_BYTES, 0);
    for (int rank = 0; rank < 2; ++rank) {
        uint8_t *h = hl.data() + (size_t)rank * IMG_HL_BYTES;
        split_rows(h + HL_WIH, li.data(), N_LG, K_X, rank);
        split_rows(h + HL_WHH, lh.data(), N_LG, K_LH, rank);
    }
    return hl;
}

// CTA-pair grid over ntiles tiles: every (cluster, rank, context) slot runs the same number of rounds; tiles past the end
// (up to `tiles`) are all padding
struct PairGrid {
    int clusters, rounds;
    size_t tiles;
};
PairGrid pair_grid(int num_sms, int ntiles)
{
    int clusters = num_sms / 2;
    const int slots_needed = (ntiles + 3) / 4;
    if (clusters > slots_needed) clusters = slots_needed;
    const int rounds = (ntiles + 4 * clusters - 1) / (4 * clusters);
    return {clusters, rounds, (size_t)rounds * 4 * clusters};
}

// developer timeline mark (nullptr: none) and, with cn_debug_kernel_ms on, the timing event kev[i], on stream s
int stamp(TcState *t, int i, const char *name, cudaStream_t s)
{
    if (name) cn_trace_mark(name, s);
    if (t->ktime_on) CN_CUDA_CHECK(cudaEventRecord(t->kev[i], s));
    return CN_OK;
}

}  // namespace

// with_om: P[e][h][n] = sum_k W_mlp1.0[n][13 + k] * om[e][h][k]  (fp32), om = the occupancy map of human h built from the
// NEXT human states of env e (multi_human_rl.py:47-49,109-163).  The map does not depend on the robot's action, so it enters
// mlp1.0 as a per-row bias in the E0 epilogue of tc_rows_pair_kernel<.., true> instead of 48 more K columns on 81 x the rows.
// A block serves kOmItems (env, human) pairs: one thread per (pair, other human) finds that human's cell and rotated velocity
// (float64 like the reference), one thread per (pair, cell) sums them in list order (one fp32 rounding), then one thread per
// output unit n applies the [om_dim x 150] weight block to all pairs (coalesced over n).
constexpr int kOmItems = 8;
__global__ void __launch_bounds__(N_H1)
tc_om_bias_kernel(EnvParams p, SarlDims d, LinearDev m10, const double *__restrict__ st, const double *__restrict__ human_v,
                  int query_env, float *__restrict__ P)
{
    __shared__ float om[kOmItems][8 * 8 * 3];
    __shared__ int cell_of[kOmItems][CN_MAX_HUMANS];
    __shared__ double vrot_of[kOmItems][CN_MAX_HUMANS][2];
    const EnvDims ed = p.d;
    const int H = ed.H, cells = d.cell_num * d.cell_num;
    const long long item0 = (long long)blockIdx.x * kOmItems, n_items = (long long)ed.E * H;
    const double dt = p.time_step;
    // (pair, other human j): j's cell in the human's grid and its velocity in the human's frame
    for (int idx = threadIdx.x; idx < kOmItems * H; idx += blockDim.x) {
        const int it = idx / H, j = idx - it * H;
        const long long item = item0 + it;
        int cell = -1;
        double vxr = 0.0, vyr = 0.0;
        if (item < n_items) {
            const int e = (int)(item / H), i = (int)(item - (long long)e * H);
            // next human states: query_env -> the cached ORCA velocity (agent.py:63-74), else constant velocity (cadrl.py:107-109)
            auto get = [&](int k, int f) -> double {
                const double vx = query_env ? human_v[(size_t)(0 * H + k) * ed.E + e] : st[st_idx(ed, F_VX, k + 1, e)];
                const double vy = query_env ? human_v[(size_t)(1 * H + k) * ed.E + e] : st[st_idx(ed, F_VY, k + 1, e)];
                if (f == 0) return st[st_idx(ed, F_PX, k + 1, e)] + vx * dt;
                if (f == 1) return st[st_idx(ed, F_PY, k + 1, e)] + vy * dt;
                return f == 2 ? vx : vy;
            };
            if (j != i) cell = occupancy_map_pair(d, i, j, get, vxr, vyr);
        }
        cell_of[it][j] = cell;
        vrot_of[it][j][0] = vxr; vrot_of[it][j][1] = vyr;
    }
    __syncthreads();
    // (pair, cell): sums over the others in list order (the reference's summation order)
    for (int idx = threadIdx.x; idx < kOmItems * cells; idx += blockDim.x) {
        const int it = idx / cells, c = idx - it * cells;
        double cnt = 0.0, sx = 0.0, sy = 0.0;
        for (int j = 0; j < H; ++j)
            if (cell_of[it][j] == c) { cnt += 1.0; sx += vrot_of[it][j][0]; sy += vrot_of[it][j][1]; }
        occupancy_map_store(d.om_ch, c, cnt, sx, sy, om[it]);
    }
    __syncthreads();
    const int n = threadIdx.x;
    float acc[kOmItems];
#pragma unroll
    for (int it = 0; it < kOmItems; ++it) acc[it] = 0.0f;
    if (n < m10.out)
        for (int k = 0; k < d.om_dim; ++k) {
            const float w = m10.wt[(size_t)(13 + k) * m10.ld + n];
#pragma unroll
            for (int it = 0; it < kOmItems; ++it) acc[it] = fmaf(om[it][k], w, acc[it]);
        }
#pragma unroll
    for (int it = 0; it < kOmItems; ++it)
        if (item0 + it < n_items) P[(size_t)(item0 + it) * N_H1 + n] = acc[it];
}

int cn_tc_init(cn_policy *p)
{
    const SarlDims &d = p->d;
    if (d.net == CN_NET_CADRL) {
        // CADRL's value network = the three tensor-core stages of the mlp3 kernel (tc_mlp3_pair_kernel<1>)
        if (!(d.in == 13 && d.m3[0] == 150 && d.m3[1] == 100 && d.m3[2] == 100 && d.m3[3] == 1)) {
            cn_set_error("CN_PREC_F16_TC is specialised for the default [cadrl] mlp_dims (150, 100, 100, 1); use CN_PREC_F32 "
                         "for other shapes");
            return CN_EUNSUPPORTED;
        }
    } else if (d.net == CN_NET_LSTM_RL) {
        // ValueNetwork1 (lstm_rl.py:9-34): LSTM(13 -> 50) on tc_lstm_pair_kernel, mlp(56 -> 150, 100, 100, 1) on the mlp3 kernel
        if (!(d.in == 13 && d.self_dim == 6 && d.lstm_h == L_HIDDEN && d.lm1[0] == 0 && d.om_dim == 0 && d.m3[0] == 150 &&
              d.m3[1] == 100 && d.m3[2] == 100 && d.m3[3] == 1)) {
            cn_set_error("CN_PREC_F16_TC runs LSTM-RL's default shape only (no interaction module, no occupancy maps, "
                         "global_state_dim 50, mlp2_dims 150,100,100,1); use CN_PREC_F32 for other shapes");
            return CN_EUNSUPPORTED;
        }
    } else {
        const bool ok = d.net == CN_NET_SARL && d.in == 13 + d.om_dim && d.self_dim == 6 && d.m1[0] == 150 && d.m1[1] == 100 &&
                        d.m2[0] == 100 && d.m2[1] == 50 && d.at[0] == 100 && d.at[1] == 100 && d.at[2] == 1 &&
                        d.m3[0] == 150 && d.m3[1] == 100 && d.m3[2] == 100 && d.m3[3] == 1;
        if (!ok) {
            cn_set_error("CN_PREC_F16_TC is specialised for the default [sarl] dims (150,100 / 100,50 / 100,100,1 / "
                         "150,100,100,1) and the default [cadrl] mlp_dims; use CN_PREC_F32 for other shapes / networks");
            return CN_EUNSUPPORTED;
        }
    }
    TcState *t = new TcState();
    memset(t, 0, sizeof(*t));
    p->tc = t;                 // from here on a failure leaves everything allocated to cn_policy_destroy
    cudaDeviceProp prop;
    CN_CUDA_CHECK(cudaGetDeviceProperties(&prop, p->device));
    t->num_sms = prop.multiProcessorCount;
    for (const auto &by_om : kRowsKernels)
        for (const auto &by_ht : by_om)
            for (RowsKernel k : by_ht) CN_CUDA_CHECK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Q_SMEM));
    CN_CUDA_CHECK(cudaFuncSetAttribute(tc_mlp3_pair_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)M_SMEM));
    CN_CUDA_CHECK(cudaFuncSetAttribute(tc_mlp3_pair_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)M_SMEM));
    CN_CUDA_CHECK(cudaFuncSetAttribute(tc_lstm_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L_SMEM));
    if (cudaMalloc((void **)&t->img_pair, 2 * IMG_H_BYTES) != cudaSuccess ||
        cudaMalloc((void **)&t->img_lstm, 2 * IMG_HL_BYTES) != cudaSuccess ||
        cudaMalloc((void **)&t->img_pair_b, 2 * IMG_HM_BYTES) != cudaSuccess) {
        cn_set_error("cudaMalloc failed for the tensor-core weight images");
        return CN_ENOMEM;
    }
    return CN_OK;
}

void cn_tc_destroy(cn_policy *p)
{
    TcState *t = (TcState *)p->tc;
    if (!t) return;
    if (t->img_pair) cudaFree(t->img_pair);
    if (t->img_pair_b) cudaFree(t->img_pair_b);
    if (t->J) cudaFree(t->J);
    if (t->X) cudaFree(t->X);
    if (t->rew) cudaFree(t->rew);
    if (t->rowv) cudaFree(t->rowv);
    if (t->omP) cudaFree(t->omP);
    if (t->img_lstm) cudaFree(t->img_lstm);
    if (t->XL) cudaFree(t->XL);
    if (t->ord) cudaFree(t->ord);
    if (t->dbg) cudaFree(t->dbg);
    if (t->kev[0]) for (int i = 0; i < 5; ++i) cudaEventDestroy(t->kev[i]);
    delete t;
    p->tc = nullptr;
}

int cn_tc_load_weights(cn_policy *p, const float *flat, cudaStream_t s)
{
    TcState *t = (TcState *)p->tc;
    const SarlDims &d = p->d;
    std::vector<HostLinear> L;           // the Linear layers in state-dict order
    const float *lstm = nullptr, *src = flat;
    for (const LayerSpec &l : cn_layers(d, p->w)) {
        if (l.dst_hh) lstm = src;
        else L.push_back({src, src + (size_t)l.in * l.out, l.in, l.out});
        src += cn_layer_floats(l);
    }
    // the last four Linears: SARL's mlp3, CADRL's value_network (cadrl.py:22-26), LSTM-RL's mlp (lstm_rl.py:9-16)
    const std::vector<uint8_t> hb = mlp3_image(&L[L.size() - 4], d.net == CN_NET_CADRL, t->tail_b);
    std::vector<uint8_t> hp, hl;
    CN_CUDA_CHECK(cudaMemcpyAsync(t->img_pair_b, hb.data(), hb.size(), cudaMemcpyHostToDevice, s));
    if (d.net == CN_NET_SARL) {
        hp = rows_image(L.data(), !d.no_gs, t->tail_a);
        CN_CUDA_CHECK(cudaMemcpyAsync(t->img_pair, hp.data(), hp.size(), cudaMemcpyHostToDevice, s));
    } else if (d.net == CN_NET_LSTM_RL) {
        hl = lstm_image(lstm);
        CN_CUDA_CHECK(cudaMemcpyAsync(t->img_lstm, hl.data(), hl.size(), cudaMemcpyHostToDevice, s));
    }
    CN_CUDA_CHECK(cudaStreamSynchronize(s));
    return CN_OK;
}

// One lookahead of every network: feature kernel, the network's middle stage, the hand-over to `tail`, the scoring stage,
// argmax.  Middle stage: SARL [tc_om_bias_kernel] tc_rows_pair_kernel; CADRL tc_mlp3_pair_kernel<1> (its whole network on
// the X tiles, one value per row); LSTM-RL lstm_order_kernel, tc_features_lstm_kernel, tc_lstm_pair_kernel.  Scoring stage:
// tc_mlp3_pair_kernel<0> on the joint-state tiles (SARL, LSTM-RL) or cadrl_min_kernel (CADRL: minimum over each group's humans).
int cn_lookahead_tc(cn_policy *p, cn_env *env, int query_env, double epsilon, cudaStream_t s, cudaStream_t tail)
{
    TcState *t = (TcState *)p->tc;
    const EnvDims ed = env->p.d;
    if (ed.H > CN_MAX_HUMANS) { cn_set_error("human_num too large"); return CN_EUNSUPPORTED; }
    int rc = cn_lookahead_prepare(p, env, s);
    if (rc) return rc;
    // programmatic dependent launches only when this handle has the GPU to itself: with several env shards in flight
    // (PipelinedHostRollout: tail stream set) a row kernel that becomes resident early and waits keeps another shard's kernels
    // off the SMs (measured: end to end 1.18e7 -> 1.14e7 env-steps/s)
    const bool pipelined = tail && tail != s;
    const int net = p->d.net, A = p->d.A;
    const bool om = p->d.om_dim > 0;
    const size_t NG = (size_t)ed.E * A;
    int G = ROWS / ed.H;
    if (G > 64) G = 64;                      // H = 1: two rows of padding per group keep the group loops within 64 items
    const PairGrid ga = pair_grid(t->num_sms, (int)((NG + G - 1) / G));       // tiles of (env, action, human) rows
    const PairGrid gb = pair_grid(t->num_sms, (int)((NG + ROWS - 1) / ROWS));  // tiles of (env, action) rows
    // the CTA-pair mlp3 kernel reads whole rounds of tiles: pad with up to one round of (zero) tiles
    if ((rc = cn_grow(t->J, t->cap_jtiles, (NG + ROWS - 1) / ROWS + 4 * (size_t)(t->num_sms / 2), J_TILE_BYTES, true, s))) return rc;
    if ((rc = cn_grow(t->rew, t->cap_rew, NG, sizeof(double)))) return rc;
    if ((rc = cn_grow(t->X, t->cap_xtiles, ga.tiles, X_TILE_BYTES))) return rc;
    const double gamma_bar = pow(p->cfg.gamma, env->p.time_step * p->cfg.v_pref);
    TailW twa, twb;
    memcpy(twa.w, t->tail_a, sizeof(twa.w));
    memcpy(twb.w, t->tail_b, sizeof(twb.w));
    const int ht = (ed.H == 5 && G == ROWS / 5) ? 5 : ((ed.H == 10 && G == ROWS / 10) ? 10 : 0);
    auto feat = ht == 5 ? tc_features_kernel<5> : (ht == 10 ? tc_features_kernel<10> : tc_features_kernel<0>);

    if ((rc = stamp(t, 0, "features", s))) return rc;
    feat<<<(unsigned)ga.tiles, ROWS, 0, s>>>(env->p, env->state, env->time, env->human_v, p->action_dev, A, query_env, (int)NG, G,
                                             env->theta, t->X, t->J, t->rew);
    CN_LAUNCH_CHECK();
    if ((rc = stamp(t, 1, "rows", s))) return rc;
    if (net == CN_NET_LSTM_RL) {
        // one sequence per (env, action) group over the humans in predict()'s order; h_n lands in the joint-state tiles
        // (the feature kernel above left their self-state chunks and the rewards)
        if ((rc = cn_grow(t->XL, t->cap_xl, gb.tiles * ed.H, X_TILE_BYTES))) return rc;
        if ((rc = cn_grow(t->ord, t->cap_ord, (size_t)ed.E * ed.H, sizeof(int32_t)))) return rc;
        lstm_order_kernel<<<(ed.E + 127) / 128, 128, 0, s>>>(env->p, env->state, query_env, t->ord);
        CN_LAUNCH_CHECK();
        tc_features_lstm_kernel<<<(unsigned)(gb.tiles * ed.H), ROWS, 0, s>>>(env->p, env->state, env->time, env->human_v, p->action_dev,
                                                                           A, query_env, (int)NG, env->theta, t->ord, t->XL);
        CN_LAUNCH_CHECK();
        tc_lstm_pair_kernel<<<2 * gb.clusters, kThreadsL, L_SMEM, s>>>(t->img_lstm, t->XL, t->J, ed.H, gb.rounds);
        CN_LAUNCH_CHECK();
    } else if (net == CN_NET_CADRL) {
        if ((rc = cn_grow(t->rowv, t->cap_rowv, ga.tiles * ROWS, sizeof(float)))) return rc;
        if ((rc = cn_launch(tc_mlp3_pair_kernel<1>, 2 * ga.clusters, kThreadsM3, M_SMEM, s, false, env->p, env->state, t->img_pair_b,
                            t->X, t->rew, A, (int)NG, p->cfg.gamma, gamma_bar, p->cfg.v_pref, p->values, ga.rounds, twb, t->rowv)))
            return rc;
    } else {
        if (om) {
            // occupancy maps of the NEXT human states (multi_human_rl.py:47-49), folded into one row bias of mlp1.0 per human
            const size_t items = (size_t)ed.E * ed.H;
            if ((rc = cn_grow(t->omP, t->cap_om, items, sizeof(float) * N_H1))) return rc;
            tc_om_bias_kernel<<<(unsigned)((items + kOmItems - 1) / kOmItems), N_H1, 0, s>>>(env->p, p->d, p->w.m1[0], env->state,
                                                                                          env->human_v, query_env, t->omP);
            CN_LAUNCH_CHECK();
        }
        const RowsKernel rows = kRowsKernels[p->d.no_gs ? 1 : 0][om ? 1 : 0][ht == 5 ? 1 : (ht == 10 ? 2 : 0)];
        // PDL: the CTAs' prologue runs under the feature kernel's tail (pdl_wait() in the kernel); with om the bias kernel
        // sits between the two -> plain launch
        if ((rc = cn_launch(rows, 2 * ga.clusters, kThreadsPair, Q_SMEM, s, !om && !pipelined, env->p, t->img_pair, t->X, t->J, (int)NG,
                            G, ga.rounds, twa, t->dbg, t->omP, A)))
            return rc;
    }
    if (pipelined) {
        // pipelined host steps: the rest of this shard's step runs on a HIGH-priority stream, so that when the middle stage
        // exits the scoring kernel is placed before the other shard's (already queued, lower-priority) row kernel takes every SM
        CN_CUDA_CHECK(cudaEventRecord(env->ev_rows, s));
        CN_CUDA_CHECK(cudaStreamWaitEvent(tail, env->ev_rows, 0));
        s = tail;
    }
    if ((rc = stamp(t, 2, "mlp3", s))) return rc;
    if (net == CN_NET_CADRL) {
        cadrl_min_kernel<<<(unsigned)((NG + 255) / 256), 256, 0, s>>>(env->p, env->state, t->rowv, t->rew, A, (int)NG, G, ed.H,
                                                                      p->cfg.gamma, gamma_bar, p->cfg.v_pref, p->values);
        CN_LAUNCH_CHECK();
    } else if ((rc = cn_launch(tc_mlp3_pair_kernel<0>, 2 * gb.clusters, kThreadsM3, M_SMEM, s, net != CN_NET_LSTM_RL, env->p,
                                 env->state, t->img_pair_b, t->J, t->rew, A, (int)NG, p->cfg.gamma, gamma_bar, p->cfg.v_pref,
                                 p->values, gb.rounds, twb, nullptr))) {
        return rc;
    }
    if ((rc = stamp(t, 3, "argmax", s))) return rc;
    if ((rc = cn_lookahead_argmax(p, env, epsilon, s, !pipelined))) return rc;
    return stamp(t, 4, nullptr, s);
}

static int selftest_impl(int32_t N, int32_t K, const float *a_host, const float *b_host, float *d_host, int device, int mode)
{
    const int bmn = mode == 1;
    if (N < 16 || N > 256 || N % 16 || K < 16 || K % 16 || K > 256 || (bmn && K > ROWS)) {
        cn_set_error("N in [16,256] step 16, K in [16,256] step 16 (K <= 128 for the MN-major variant)");
        return CN_EINVAL;
    }
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); cn_set_error("no CUDA device available; no CPU fallback"); return CN_ECUDA; }
    CN_CUDA_CHECK(cudaSetDevice(device));
    std::vector<uint8_t> ai(bytes_of(ROWS, K), 0), bi(bmn ? bytes_of(ROWS, N) : bytes_of(N, K), 0);
    for (int r = 0; r < ROWS; ++r) for (int k = 0; k < K; ++k) put(ai, 0, ROWS, r, k, a_host[(size_t)r * K + k]);
    for (int r = 0; r < N; ++r)
        for (int k = 0; k < K; ++k) {
            if (bmn) put(bi, 0, ROWS, k, r, b_host[(size_t)r * K + k]);   // activation-style image: rows = k, columns = n
            else put(bi, 0, N, r, k, b_host[(size_t)r * K + k]);
        }
    uint8_t *da = nullptr, *db = nullptr;
    float *dd = nullptr;
    CN_CUDA_CHECK(cudaMalloc((void **)&da, ai.size()));
    CN_CUDA_CHECK(cudaMalloc((void **)&db, bi.size()));
    CN_CUDA_CHECK(cudaMalloc((void **)&dd, sizeof(float) * ROWS * N));
    CN_CUDA_CHECK(cudaMemcpy(da, ai.data(), ai.size(), cudaMemcpyHostToDevice));
    CN_CUDA_CHECK(cudaMemcpy(db, bi.data(), bi.size(), cudaMemcpyHostToDevice));
    const size_t smem = ai.size() + bi.size() + 64;
    CN_CUDA_CHECK(cudaFuncSetAttribute(umma_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    umma_selftest_kernel<<<1, 128, smem>>>(da, db, dd, N, K, mode);
    CN_LAUNCH_CHECK();
    CN_CUDA_CHECK(cudaDeviceSynchronize());
    CN_CUDA_CHECK(cudaMemcpy(d_host, dd, sizeof(float) * ROWS * N, cudaMemcpyDeviceToHost));
    cudaFree(da); cudaFree(db); cudaFree(dd);
    return CN_OK;
}

/* D[128 x N] = A[128 x K] * B[N x K]^T with one cta_group::1 UMMA chain; the three operand modes the kernels use */
extern "C" int cn_selftest_umma(int32_t N, int32_t K, const float *a_host, const float *b_host, float *d_host, int device)
{
    return selftest_impl(N, K, a_host, b_host, d_host, device, 0);
}

extern "C" int cn_selftest_umma_bmn(int32_t N, int32_t K, const float *a_host, const float *b_host, float *d_host, int device)
{
    return selftest_impl(N, K, a_host, b_host, d_host, device, 1);
}

extern "C" int cn_selftest_umma_ts(int32_t N, int32_t K, const float *a_host, const float *b_host, float *d_host, int device)
{
    return selftest_impl(N, K, a_host, b_host, d_host, device, 2);
}

// CTA-pair building block: D[256 x N] = A[256 x K] * B[N x K]^T with one cta_group::2 UMMA chain (N % 16 == 0)
extern "C" int cn_selftest_umma_pair(int32_t N, int32_t K, const float *a_host, const float *b_host, float *d_host,
                                     int32_t reps, long long *cycles_host, int device)
{
    if (N < 32 || N > 256 || N % 16 || K < 16 || K % 16 || K > 256 || reps < 1) {
        cn_set_error("N in [32,256] step 16, K in [16,256] step 16, reps >= 1");
        return CN_EINVAL;
    }
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); cn_set_error("no CUDA device available; no CPU fallback"); return CN_ECUDA; }
    CN_CUDA_CHECK(cudaSetDevice(device));
    const size_t a_bytes = bytes_of(ROWS, K), b_bytes = bytes_of(N / 2, K);
    std::vector<uint8_t> ai(2 * a_bytes, 0), bi(2 * b_bytes, 0);
    for (int r = 0; r < 2 * ROWS; ++r)
        for (int k = 0; k < K; ++k) put(ai, (uint32_t)((r / ROWS) * a_bytes), ROWS, r % ROWS, k, a_host[(size_t)r * K + k]);
    for (int r = 0; r < N; ++r)
        for (int k = 0; k < K; ++k) put(bi, (uint32_t)((r / (N / 2)) * b_bytes), N / 2, r % (N / 2), k, b_host[(size_t)r * K + k]);
    uint8_t *da = nullptr, *db = nullptr;
    float *dd = nullptr;
    long long *dc = nullptr;
    CN_CUDA_CHECK(cudaMalloc((void **)&da, ai.size()));
    CN_CUDA_CHECK(cudaMalloc((void **)&db, bi.size()));
    CN_CUDA_CHECK(cudaMalloc((void **)&dd, sizeof(float) * 2 * ROWS * N));
    CN_CUDA_CHECK(cudaMalloc((void **)&dc, sizeof(long long)));
    CN_CUDA_CHECK(cudaMemcpy(da, ai.data(), ai.size(), cudaMemcpyHostToDevice));
    CN_CUDA_CHECK(cudaMemcpy(db, bi.data(), bi.size(), cudaMemcpyHostToDevice));
    const size_t smem = a_bytes + b_bytes + 64;
    CN_CUDA_CHECK(cudaFuncSetAttribute(umma_pair_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    umma_pair_selftest_kernel<<<2, 160, smem>>>(da, db, dd, N, K, reps, dc);
    CN_LAUNCH_CHECK();
    CN_CUDA_CHECK(cudaDeviceSynchronize());
    CN_CUDA_CHECK(cudaMemcpy(d_host, dd, sizeof(float) * 2 * ROWS * N, cudaMemcpyDeviceToHost));
    if (cycles_host) CN_CUDA_CHECK(cudaMemcpy(cycles_host, dc, sizeof(long long), cudaMemcpyDeviceToHost));
    cudaFree(da); cudaFree(db); cudaFree(dd); cudaFree(dc);
    return CN_OK;
}

// Developer diagnostic (not part of the reference surface): clock64() at the phase boundaries of one tile of
// tc_rows_pair_kernel's first cluster (QPROBE slots).  First call arms the probes; later calls return the last recorded timestamps.
extern "C" int cn_debug_tc_timing(cn_policy *p, long long *out16)
{
    if (!p || !p->tc) { cn_set_error("policy has no tensor-core state"); return CN_EINVAL; }
    TcState *t = (TcState *)p->tc;
    CN_CUDA_CHECK(cudaSetDevice(p->device));
    if (!t->dbg) {
        CN_CUDA_CHECK(cudaMalloc((void **)&t->dbg, 256 * sizeof(long long)));
        CN_CUDA_CHECK(cudaMemset(t->dbg, 0, 256 * sizeof(long long)));
    }
    CN_CUDA_CHECK(cudaDeviceSynchronize());
    CN_CUDA_CHECK(cudaMemcpy(out16, t->dbg, 256 * sizeof(long long), cudaMemcpyDeviceToHost));
    return CN_OK;
}

// Measurement hook of bench.py (the `roofline` object needs the duration of the dominant KERNEL, measured live with CUDA
// events on the stream the kernel is launched on -- torch.cuda.Event only sees torch's current stream around the whole C
// call).  on = 1: every later cn_policy_lookahead / cn_rollout_step records events around its kernels; out4 (optional)
// receives the durations of the LAST lookahead in ms: tc_features_kernel, tc_rows_pair_kernel, tc_mlp3_pair_kernel,
// argmax_kernel (blocking: synchronises on the last event).  Not meaningful for the pipelined (tail-stream) calls.
extern "C" int cn_debug_kernel_ms(cn_policy *p, int on, float *out4)
{
    if (!p || !p->tc) { cn_set_error("policy has no tensor-core state"); return CN_EINVAL; }
    TcState *t = (TcState *)p->tc;
    CN_CUDA_CHECK(cudaSetDevice(p->device));
    if (out4) {
        if (!t->kev[0]) { cn_set_error("kernel timing was never enabled"); return CN_EINVAL; }
        CN_CUDA_CHECK(cudaEventSynchronize(t->kev[4]));
        for (int i = 0; i < 4; ++i) CN_CUDA_CHECK(cudaEventElapsedTime(&out4[i], t->kev[i], t->kev[i + 1]));
    }
    if (on && !t->kev[0]) for (int i = 0; i < 5; ++i) CN_CUDA_CHECK(cudaEventCreate(&t->kev[i]));
    t->ktime_on = on ? 1 : 0;
    return CN_OK;
}
