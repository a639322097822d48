// dense_f32.cuh -- FP32 CUDA-core building blocks of the small dense layers that run OUTSIDE the tensor-core lookahead
// (the fused trainer, trainer_nets.cu, and the world models, world_model.cu): activations in shared memory, weights streamed
// from L2 as a transposed [in][out] block, one CTA of kThreads threads.
#pragma once
#include <stdint.h>

namespace dense_f32 {

constexpr int kThreads = 256;

__host__ __device__ __forceinline__ int pad4(int x) { return (x + 3) & ~3; }

// Y[r][o] = act(b[o] + sum_k X[r * ldx + k] * Wt[k * O + o]),  r < R, o < O.   Wt is [K][O] in global memory (coalesced over
// o); X lives in shared memory.  One thread = kRowsPerItem rows x 1 output: with R <= 8 every weight is fetched ONCE per CTA.
// K is walked 16 at a time with the 16 weight loads issued before any FMA: the loop is bound by the L2 latency of those loads
// (a CTA has 256 threads and no other work to hide it), so loads in flight per thread are what sets the speed.
constexpr int kRowsPerItem = 8;
template <bool W_IN_SMEM>
__device__ __forceinline__ float ldw(const float *p) { return W_IN_SMEM ? *p : __ldg(p); }

// gate: optional ReLU-backward mask applied to the result (see the epilogue).
// W_IN_SMEM: the weight block (and bias) was staged into shared memory (trainer_nets.cu prefetches the next op's block with
// cp.async while this one computes); otherwise it is streamed from L2.
template <bool W_IN_SMEM>
__device__ __forceinline__ void dense_t(const float *__restrict__ X, int ldx, int R, int K, const float *__restrict__ Wt,
                                        const float *__restrict__ b, int O, float *__restrict__ Y, int ldy, bool relu, bool accumulate,
                                        const float *__restrict__ gate = nullptr, int ldg = 0)
{
    const int groups = (R + kRowsPerItem - 1) / kRowsPerItem;
    for (int idx = threadIdx.x; idx < O * groups; idx += kThreads) {
        const int o = idx % O, r0 = (idx / O) * kRowsPerItem;
        float acc[kRowsPerItem];
        const float bias = b ? b[o] : 0.0f;
#pragma unroll
        for (int i = 0; i < kRowsPerItem; ++i) acc[i] = bias;
        const float *x0 = X + (size_t)r0 * ldx;
        const int nr = min(kRowsPerItem, R - r0);
        const float *wp = Wt + o;
        int k = 0;
        for (; k + 16 <= K; k += 16) {                   // 16 independent L2 loads in flight per thread
            float w[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) w[j] = ldw<W_IN_SMEM>(wp + (size_t)(k + j) * O);
#pragma unroll
            for (int i = 0; i < kRowsPerItem; ++i) {
                if (i < nr) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float4 x = *reinterpret_cast<const float4 *>(x0 + (size_t)i * ldx + k + 4 * q);
                        acc[i] = fmaf(x.x, w[4 * q], acc[i]); acc[i] = fmaf(x.y, w[4 * q + 1], acc[i]);
                        acc[i] = fmaf(x.z, w[4 * q + 2], acc[i]); acc[i] = fmaf(x.w, w[4 * q + 3], acc[i]);
                    }
                }
            }
        }
        for (; k + 4 <= K; k += 4) {
            float w[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) w[j] = ldw<W_IN_SMEM>(wp + (size_t)(k + j) * O);
#pragma unroll
            for (int i = 0; i < kRowsPerItem; ++i) {
                if (i < nr) {
                    const float4 x = *reinterpret_cast<const float4 *>(x0 + (size_t)i * ldx + k);
                    acc[i] = fmaf(x.x, w[0], acc[i]); acc[i] = fmaf(x.y, w[1], acc[i]);
                    acc[i] = fmaf(x.z, w[2], acc[i]); acc[i] = fmaf(x.w, w[3], acc[i]);
                }
            }
        }
        for (; k < K; ++k) {
            const float w = ldw<W_IN_SMEM>(wp + (size_t)k * O);
#pragma unroll
            for (int i = 0; i < kRowsPerItem; ++i) if (i < nr) acc[i] = fmaf(x0[(size_t)i * ldx + k], w, acc[i]);
        }
#pragma unroll
        for (int i = 0; i < kRowsPerItem; ++i) {
            if (i < nr) {
                float v = acc[i];
                if (accumulate) v += Y[(size_t)(r0 + i) * ldy + o];
                // gate = the post-ReLU activation this gradient flows back through: dA *= (act > 0), fused ReLU backward
                if (gate && !(gate[(size_t)(r0 + i) * ldg + o] > 0.0f)) v = 0.0f;
                Y[(size_t)(r0 + i) * ldy + o] = relu ? fmaxf(v, 0.0f) : v;
            }
        }
    }
}

// Weight staging (the fused trainers): cp.async copies of a 16-byte aligned block of n floats (n a multiple of 4) from
// global into shared memory, issued by the whole CTA as one commit group; cp_async_wait<N> leaves N groups in flight.
__device__ __forceinline__ void cp_async16(float *dst_smem, const float *src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }
__device__ __forceinline__ void stage_async(float *dst, const float *src, int n)
{
#pragma unroll 4
    for (int i = threadIdx.x * 4; i < n; i += kThreads * 4) cp_async16(dst + i, src + i);
    cp_async_commit();
}

__device__ __forceinline__ void dense(const float *__restrict__ X, int ldx, int R, int K, const float *__restrict__ Wt,
                                      const float *__restrict__ b, int O, float *__restrict__ Y, int ldy, bool relu, bool accumulate)
{
    dense_t<false>(X, ldx, R, K, Wt, b, O, Y, ldy, relu, accumulate);
}

// dW[o][k] = sum_r dY[r][o] * Xin[r][k] and db[o] = sum_r dY[r][o] -> this CTA's partial gradient block (global memory).
// One thread = 2 outputs x 4 inputs; consecutive threads walk k (conflict-free LDS.128 of Xin, broadcast dY).
__device__ __forceinline__ void weight_grad(const float *__restrict__ dY, int ldy, const float *__restrict__ Xin, int ldx, int R,
                                            int O, int K, float *__restrict__ gW /*[O][K]*/, float *__restrict__ gb /*[O]*/)
{
    const int k4n = (K + 3) >> 2, o2n = (O + 1) >> 1;
    for (int idx = threadIdx.x; idx < o2n * k4n; idx += kThreads) {
        const int k = (idx % k4n) * 4, o = (idx / k4n) * 2;
        const bool o1 = o + 1 < O;
        float a0[4] = {0, 0, 0, 0}, a1[4] = {0, 0, 0, 0};
        if (k + 4 <= K) {
            for (int r = 0; r < R; ++r) {
                const float4 x = *reinterpret_cast<const float4 *>(Xin + (size_t)r * ldx + k);
                const float d0 = dY[(size_t)r * ldy + o], d1 = o1 ? dY[(size_t)r * ldy + o + 1] : 0.0f;
                a0[0] = fmaf(d0, x.x, a0[0]); a0[1] = fmaf(d0, x.y, a0[1]); a0[2] = fmaf(d0, x.z, a0[2]); a0[3] = fmaf(d0, x.w, a0[3]);
                a1[0] = fmaf(d1, x.x, a1[0]); a1[1] = fmaf(d1, x.y, a1[1]); a1[2] = fmaf(d1, x.z, a1[2]); a1[3] = fmaf(d1, x.w, a1[3]);
            }
        } else {
            for (int r = 0; r < R; ++r) {
                const float d0 = dY[(size_t)r * ldy + o], d1 = o1 ? dY[(size_t)r * ldy + o + 1] : 0.0f;
                for (int j = 0; k + j < K; ++j) {
                    const float x = Xin[(size_t)r * ldx + k + j];
                    a0[j] = fmaf(d0, x, a0[j]); a1[j] = fmaf(d1, x, a1[j]);
                }
            }
        }
        for (int j = 0; j < 4 && k + j < K; ++j) {
            gW[(size_t)o * K + k + j] = a0[j];
            if (o1) gW[(size_t)(o + 1) * K + k + j] = a1[j];
        }
    }
    for (int o = threadIdx.x; o < O; o += kThreads) {
        float s = 0.0f;
        for (int r = 0; r < R; ++r) s += dY[(size_t)r * ldy + o];
        gb[o] = s;
    }
}

}  // namespace dense_f32
