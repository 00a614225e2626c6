// Sinkhorn "EMD" of the reference (metrics.py:94-158, `earth_mover_distance_gpu`) on the GPU.
//
// The reference materialises the [n, m] cost matrix per pair (16.8 MB at 2048 x 2048) and runs dense
// logsumexp passes over it; here the cost is recomputed from the two normalised clouds on the fly (the
// same direct-difference tile as the Chamfer kernels), so a half-iteration touches 64 KB per pair:
//   cmax   = max_{b,i,j} |x_bi - y_bj|                      (ONE maximum over the whole batch, metrics.py:124)
//   alpha_i = eps * (log(mu + 1e-10) - LSE_j(-C_ij / eps + beta_j)),  C = |x_i - y_j| / cmax   (:142)
//   beta_j  = eps * (log(nu + 1e-10) - LSE_i(-C_ij / eps + alpha_i))  (uses the NEW alpha, :145)
//   emd    = sum_ij exp(-C_ij / eps + alpha_i + beta_j) * C_ij                                  (:154-157)
// LSE is an online (running max) log-sum-exp in base 2, 4 targets per rescale.  The host loop reads the two
// max-abs dual changes back after every iteration, exactly like the reference's `if err < thresh` (:148-151).
#include <cstdint>
#include <cuda_runtime.h>

namespace pcd {

constexpr int kEmdTile = 1024;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

__device__ __forceinline__ float block_max_128(float v, float* red) {
    for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    v = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
    __syncthreads();
    return v;
}

// max pairwise distance of every pair of the batch -> one scalar (float bits, values >= 0)
template <int R>
__global__ void __launch_bounds__(128) emd_cmax_kernel(const float4* __restrict__ X, const float4* __restrict__ Y, int N, int M,
                                                       unsigned* __restrict__ cmax_bits) {
    __shared__ float4 st[kEmdTile];
    __shared__ float red[4];
    const int pair = blockIdx.y;
    const float4* x = X + static_cast<long long>(pair) * N;
    const float4* y = Y + static_cast<long long>(pair) * M;
    float qx[R], qy[R], qz[R], best[R];
    int nan_d = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = blockIdx.x * (128 * R) + r * 128 + threadIdx.x;
        const float4 v = x[i < N ? i : N - 1];     // duplicates of a real row never change a maximum
        qx[r] = v.x; qy[r] = v.y; qz[r] = v.z; best[r] = 0.f;
    }
    for (int t0 = 0; t0 < M; t0 += kEmdTile) {
        const int cnt = min(kEmdTile, M - t0);
        __syncthreads();
        for (int i = threadIdx.x; i < cnt; i += 128) st[i] = y[t0 + i];
        __syncthreads();
#pragma unroll 4
        for (int j = 0; j < cnt; ++j) {
            const float4 tv = st[j];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const float dx = qx[r] - tv.x, dy = qy[r] - tv.y, dz = qz[r] - tv.z;
                const float d2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
                nan_d |= d2 != d2;
                best[r] = fmaxf(best[r], d2);
            }
        }
    }
    float m = best[0];
#pragma unroll
    for (int r = 1; r < R; ++r) m = fmaxf(m, best[r]);
    m = block_max_128(m, red);
    // torch's C.max() (metrics.py:124) propagates NaN, fmaxf drops it: a NaN distance (a poisoned cloud) makes the batch maximum,
    // hence every pair's cost, NaN.  Under the unsigned atomicMax the NaN bits 0x7fc00000 beat every finite value and inf.
    nan_d = __syncthreads_or(nan_d);
    if (threadIdx.x == 0) atomicMax(cmax_bits, nan_d ? 0x7fc00000u : __float_as_uint(sqrtf(m)));
}

// One Sinkhorn half-step for the duals of the QUERY cloud:
//   dual_q[i] = eps * (log_marg - LSE_j(-lambda * |q_i - t_j| / cmax + dual_t[j]))
// and the max-abs change of dual_q over the whole batch -> err_bits (float bits, pre-zeroed).
template <int R>
__global__ void __launch_bounds__(128) sinkhorn_half_kernel(const float4* __restrict__ Q, const float4* __restrict__ T,
                                                            const float* __restrict__ dual_t, float* __restrict__ dual_q, int Nq,
                                                            int Nt, const unsigned* __restrict__ cmax_bits, float lambda, float eps,
                                                            float log_marg, unsigned* __restrict__ err_bits) {
    __shared__ float4 st[kEmdTile];     // (x, y, z, dual_t * log2e)
    __shared__ float red[4];
    const int pair = blockIdx.y;
    const float4* q = Q + static_cast<long long>(pair) * Nq;
    const float4* t = T + static_cast<long long>(pair) * Nt;
    const float* dt = dual_t + static_cast<long long>(pair) * Nt;
    const float s2 = -lambda / __uint_as_float(*cmax_bits) * kLog2e;   // exponent scale in base 2
    float qx[R], qy[R], qz[R], mx[R], sum[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = blockIdx.x * (128 * R) + r * 128 + threadIdx.x;
        const float4 v = q[i < Nq ? i : Nq - 1];
        qx[r] = v.x; qy[r] = v.y; qz[r] = v.z;
        mx[r] = -INFINITY; sum[r] = 0.f;
    }
    for (int t0 = 0; t0 < Nt; t0 += kEmdTile) {
        const int cnt = min(kEmdTile, Nt - t0);
        __syncthreads();
        for (int i = threadIdx.x; i < kEmdTile; i += 128) {
            float4 v = make_float4(0.f, 0.f, 0.f, -INFINITY);     // padding: exp2(-inf) = 0, contributes nothing
            if (i < cnt) { v = t[t0 + i]; v.w = dt[t0 + i] * kLog2e; }
            st[i] = v;
        }
        __syncthreads();
        const int cnt4 = (cnt + 3) & ~3;
        for (int j = 0; j < cnt4; j += 4) {
            const float4 a = st[j], b = st[j + 1], c = st[j + 2], d = st[j + 3];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                float v0, v1, v2, v3;
                {
                    const float dx = qx[r] - a.x, dy = qy[r] - a.y, dz = qz[r] - a.z;
                    v0 = fmaf(sqrtf(fmaf(dz, dz, fmaf(dy, dy, dx * dx))), s2, a.w);
                }
                {
                    const float dx = qx[r] - b.x, dy = qy[r] - b.y, dz = qz[r] - b.z;
                    v1 = fmaf(sqrtf(fmaf(dz, dz, fmaf(dy, dy, dx * dx))), s2, b.w);
                }
                {
                    const float dx = qx[r] - c.x, dy = qy[r] - c.y, dz = qz[r] - c.z;
                    v2 = fmaf(sqrtf(fmaf(dz, dz, fmaf(dy, dy, dx * dx))), s2, c.w);
                }
                {
                    const float dx = qx[r] - d.x, dy = qy[r] - d.y, dz = qz[r] - d.z;
                    v3 = fmaf(sqrtf(fmaf(dz, dz, fmaf(dy, dy, dx * dx))), s2, d.w);
                }
                const float mn = fmaxf(fmaxf(mx[r], fmaxf(v0, v1)), fmaxf(v2, v3));   // finite: group 0 holds a real target
                sum[r] = sum[r] * exp2f(mx[r] - mn) + ((exp2f(v0 - mn) + exp2f(v1 - mn)) + (exp2f(v2 - mn) + exp2f(v3 - mn)));
                mx[r] = mn;
            }
        }
    }
    float err = 0.f;
    int nan_change = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = blockIdx.x * (128 * R) + r * 128 + threadIdx.x;
        if (i < Nq) {
            const float lse = (mx[r] + log2f(sum[r])) * kLn2;
            const float nv = eps * (log_marg - lse);
            float* dst = dual_q + static_cast<long long>(pair) * Nq + i;
            const float change = fabsf(nv - *dst);
            nan_change |= change != change;
            err = fmaxf(err, change);
            *dst = nv;
        }
    }
    err = block_max_128(err, red);
    // torch's max-abs change propagates NaN (a NaN dual, or inf - inf), fmaxf drops it: publish NaN, so that `err < thresh` never
    // holds and the loop runs max_iter iterations like the reference's (:148-151)
    nan_change = __syncthreads_or(nan_change);
    if (threadIdx.x == 0) atomicMax(err_bits, nan_change ? 0x7fc00000u : __float_as_uint(err));
}

// rowsum[pair][block] = sum over the block's rows i and all j of exp(-lambda*C_ij + alpha_i + beta_j) * C_ij (fixed order)
template <int R>
__global__ void __launch_bounds__(128) sinkhorn_cost_kernel(const float4* __restrict__ Q, const float4* __restrict__ T,
                                                            const float* __restrict__ alpha, const float* __restrict__ beta, int Nq,
                                                            int Nt, const unsigned* __restrict__ cmax_bits, float lambda,
                                                            float* __restrict__ partial) {
    __shared__ float4 st[kEmdTile];
    __shared__ float red[128];
    const int pair = blockIdx.y;
    const float4* q = Q + static_cast<long long>(pair) * Nq;
    const float4* t = T + static_cast<long long>(pair) * Nt;
    const float inv_cmax = 1.0f / __uint_as_float(*cmax_bits);
    const float s2 = -lambda * kLog2e;
    float qx[R], qy[R], qz[R], qa[R], acc[R];
    bool ok[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = blockIdx.x * (128 * R) + r * 128 + threadIdx.x;
        ok[r] = i < Nq;
        const float4 v = q[ok[r] ? i : Nq - 1];
        qx[r] = v.x; qy[r] = v.y; qz[r] = v.z;
        qa[r] = ok[r] ? alpha[static_cast<long long>(pair) * Nq + i] * kLog2e : -INFINITY;
        acc[r] = 0.f;
    }
    for (int t0 = 0; t0 < Nt; t0 += kEmdTile) {
        const int cnt = min(kEmdTile, Nt - t0);
        __syncthreads();
        for (int i = threadIdx.x; i < cnt; i += 128) {
            float4 v = t[t0 + i];
            v.w = beta[static_cast<long long>(pair) * Nt + t0 + i] * kLog2e;
            st[i] = v;
        }
        __syncthreads();
        // Two-level row sum: 32 targets into `sub`, then `sub` into the row total.  One fp32 accumulator over a whole row rounds
        // the long tail of small terms away against the large total: the result came out low by ~6e-10 relative per target
        // (-2.7e-6 at 4100 targets, against fp64).  With 32-target chunks the error stays near 2e-8.
        for (int j0 = 0; j0 < cnt; j0 += 32) {
            const int j1 = min(cnt, j0 + 32);
            float sub[R];
#pragma unroll
            for (int r = 0; r < R; ++r) sub[r] = 0.f;
#pragma unroll 2
            for (int j = j0; j < j1; ++j) {
                const float4 tv = st[j];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const float dx = qx[r] - tv.x, dy = qy[r] - tv.y, dz = qz[r] - tv.z;
                    const float c = sqrtf(fmaf(dz, dz, fmaf(dy, dy, dx * dx))) * inv_cmax;
                    sub[r] = fmaf(exp2f(fmaf(c, s2, qa[r] + tv.w)), c, sub[r]);
                }
            }
#pragma unroll
            for (int r = 0; r < R; ++r) acc[r] += sub[r];
        }
    }
    float tot = 0.f;
#pragma unroll
    for (int r = 0; r < R; ++r) tot += ok[r] ? acc[r] : 0.f;
    red[threadIdx.x] = tot;
    __syncthreads();
    for (int s = 64; s; s >>= 1) {
        if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[static_cast<long long>(pair) * gridDim.x + blockIdx.x] = red[0];
}

__global__ void emd_finish_kernel(const float* __restrict__ partial, int nblk, float scaling, float* __restrict__ emd) {
    const int pair = blockIdx.x;
    float s = 0.f;
    for (int b = 0; b < nblk; ++b) s += partial[static_cast<long long>(pair) * nblk + b];
    emd[pair] = s * scaling;
}

constexpr int kEmdR = 2;   // rows per thread: 256-row blocks -> 8 blocks per 2048-point cloud

int emd_row_blocks(int n) { return (n + 128 * kEmdR - 1) / (128 * kEmdR); }

cudaError_t launch_emd_cmax(const float4* X, const float4* Y, int pairs, int N, int M, unsigned* cmax_bits, cudaStream_t s) {
    emd_cmax_kernel<kEmdR><<<dim3(emd_row_blocks(N), pairs), 128, 0, s>>>(X, Y, N, M, cmax_bits);
    return cudaGetLastError();
}

cudaError_t launch_sinkhorn_half(const float4* Q, const float4* T, const float* dual_t, float* dual_q, int pairs, int Nq, int Nt,
                                 const unsigned* cmax_bits, float lambda, float eps, float log_marg, unsigned* err_bits,
                                 cudaStream_t s) {
    sinkhorn_half_kernel<kEmdR><<<dim3(emd_row_blocks(Nq), pairs), 128, 0, s>>>(Q, T, dual_t, dual_q, Nq, Nt, cmax_bits, lambda, eps,
                                                                               log_marg, err_bits);
    return cudaGetLastError();
}

cudaError_t launch_sinkhorn_cost(const float4* Q, const float4* T, const float* alpha, const float* beta, int pairs, int Nq, int Nt,
                                 const unsigned* cmax_bits, float lambda, float scaling, float* partial, float* emd, cudaStream_t s) {
    const int nblk = emd_row_blocks(Nq);
    sinkhorn_cost_kernel<kEmdR><<<dim3(nblk, pairs), 128, 0, s>>>(Q, T, alpha, beta, Nq, Nt, cmax_bits, lambda, partial);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    emd_finish_kernel<<<pairs, 1, 0, s>>>(partial, nblk, scaling, emd);
    return cudaGetLastError();
}

}  // namespace pcd
