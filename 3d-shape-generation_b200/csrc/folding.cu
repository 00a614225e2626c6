// FoldingDecoder (reference networks.py:386-412, 1449-1509; PointNetVAE.decode :1579-1589): small kernels
// around the tcgen05 GEMM of gemm_tc.cu.  Rows are (sample, grid point) pairs, 1024 grid points per sample.
//
// Algebra done at load time (api_latent.cu): a FoldingLayer is conv-ReLU-conv with NO activation after it, so the
// second conv of one layer and the first conv of the next compose into one matrix; the latent columns of the first
// conv of a fold multiply a per-sample constant and become a per-sample bias.  One fold is therefore
//   h1 = relu(bias_z[b] + Wg * in[row])        in = grid point (K = 2) or fold1's output (K = 3)   (fold_first_kernel)
//   h3 = relu(W_ab * h1 + b_ab)                512 x 512 GEMM      (tcgen05 split precision, gemm_tc.cu NP = 3)
//   h5 = relu(W_bc * h3 + b_bc)                3 x 512 GEMM        (fold_tail16_kernel)
//   out = W_c2 * h5 + b_c2                     3 x 3               (fold_tail16_kernel)
// h1 and h3 are fp16 hi + lo planes ([2 * rows][512], lo plane `rows` rows below; x = hi + lo to ~22 mantissa
// bits) and the 512 x 512 GEMM runs D += hi*hi + hi*lo + lo*hi with fp32 accumulation: fp32-class results (measured 2e-6 relative
// against the reference) at tensor-core rate.  96 % of the decoder's FLOPs.
#include <cstdint>
#include <cuda_runtime.h>

#include "pcd_types.h"

namespace pcd {

// out[row][c] = relu(bias[b][c] + sum_k W[c][k] * in[row_in][k]),  c < 512, 8 rows per CTA, 4 channels per thread.
// in_mod > 0: row_in = row % in_mod (the shared 32 x 32 grid), otherwise row_in = row.
// out16: fp16 hi / lo planes (lo plane `plane_rows` rows below)
template <int KIN>
__global__ void __launch_bounds__(128) fold_first_kernel(const float* __restrict__ in, int in_mod, const float* __restrict__ W,
                                                         const float* __restrict__ bias, int rows_per_sample,
                                                         uint16_t* __restrict__ out16, long long plane_rows) {
    const int c0 = threadIdx.x * 4;
    float w[4][KIN];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int k = 0; k < KIN; ++k) w[j][k] = W[(c0 + j) * KIN + k];
    const long long row0 = static_cast<long long>(blockIdx.x) * 8;
    uint16_t* __restrict__ lo16 = out16 + plane_rows * 512;
    const int b = static_cast<int>(row0 / rows_per_sample);          // 8 | rows_per_sample: one sample per CTA
    const float4 bz = *reinterpret_cast<const float4*>(bias + static_cast<long long>(b) * 512 + c0);
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const long long row = row0 + r;
        const long long ri = in_mod > 0 ? row % in_mod : row;
        float x[KIN];
#pragma unroll
        for (int k = 0; k < KIN; ++k) x[k] = in[ri * KIN + k];
        float v[4] = {bz.x, bz.y, bz.z, bz.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
            for (int k = 0; k < KIN; ++k) v[j] = fmaf(w[j][k], x[k], v[j]);
            v[j] = fmaxf(v[j], 0.f);
        }
        const uint32_t h0 = pack16x2(v[0], v[1], 1), h1 = pack16x2(v[2], v[3], 1);
        const float2 r0 = unpack16x2(h0, 1), r1 = unpack16x2(h1, 1);
        *reinterpret_cast<uint2*>(out16 + row * 512 + c0) = make_uint2(h0, h1);
        *reinterpret_cast<uint2*>(lo16 + row * 512 + c0) =
            make_uint2(pack16x2(v[0] - r0.x, v[1] - r0.y, 1), pack16x2(v[2] - r1.x, v[3] - r1.y, 1));
    }
}

// Tail of a fold: h3 arrives as fp16 hi / lo planes; h5 = relu(W_bc (hi + lo) + b_bc) (3 x 512, fp32
// FMAs), out = W_c2 h5 + b_c2 (3 x 3).  One warp per row: a lane owns 16 of the 512 channels, shuffle reduction.
__global__ void __launch_bounds__(256) fold_tail16_kernel(const uint16_t* __restrict__ h3, long long plane_rows, const float* __restrict__ Wbc,
                                                          const float* __restrict__ bbc, const float* __restrict__ Wc2,
                                                          const float* __restrict__ bc2, long long rows, int rows_per_sample,
                                                          int channel_major, float* __restrict__ out) {
    const long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    float acc[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int k0 = half * 256 + lane * 8;
        const uint4 hv = *reinterpret_cast<const uint4*>(h3 + row * 512 + k0);
        const uint4 lv = *reinterpret_cast<const uint4*>(h3 + (row + plane_rows) * 512 + k0);
        const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w}, lw[4] = {lv.x, lv.y, lv.z, lv.w};
        float x[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float2 a = unpack16x2(hw[j], 1), b = unpack16x2(lw[j], 1);
            x[2 * j] = a.x + b.x; x[2 * j + 1] = a.y + b.y;
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float4 w0 = *reinterpret_cast<const float4*>(Wbc + c * 512 + k0), w1 = *reinterpret_cast<const float4*>(Wbc + c * 512 + k0 + 4);
            acc[c] = fmaf(w0.x, x[0], fmaf(w0.y, x[1], fmaf(w0.z, x[2], fmaf(w0.w, x[3], acc[c]))));
            acc[c] = fmaf(w1.x, x[4], fmaf(w1.y, x[5], fmaf(w1.z, x[6], fmaf(w1.w, x[7], acc[c]))));
        }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c)
        for (int o = 16; o; o >>= 1) acc[c] += __shfl_xor_sync(0xffffffffu, acc[c], o);
    if (lane != 0) return;
    const float x0 = fmaxf(acc[0] + bbc[0], 0.f), x1 = fmaxf(acc[1] + bbc[1], 0.f), x2 = fmaxf(acc[2] + bbc[2], 0.f);
    float v[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) v[c] = fmaf(Wc2[c * 3 + 2], x2, fmaf(Wc2[c * 3 + 1], x1, fmaf(Wc2[c * 3], x0, bc2[c])));
    if (channel_major) {
        const long long b = row / rows_per_sample, n = row - b * rows_per_sample;
#pragma unroll
        for (int c = 0; c < 3; ++c) out[(b * 3 + c) * rows_per_sample + n] = v[c];
    } else {
#pragma unroll
        for (int c = 0; c < 3; ++c) out[row * 3 + c] = v[c];
    }
}

// U [B*3][P] (channel-major) -> out [B][P][3]
__global__ void __launch_bounds__(256) fold_transpose_kernel(const float* __restrict__ U, int B, int P, float* __restrict__ out) {
    const long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;     // over B * P
    if (i >= static_cast<long long>(B) * P) return;
    const long long b = i / P, p = i - b * P;
#pragma unroll
    for (int c = 0; c < 3; ++c) out[i * 3 + c] = U[(b * 3 + c) * P + p];
}

cudaError_t launch_fold_first(int kin, const float* in, int in_mod, const float* W, const float* bias, long long rows,
                              int rows_per_sample, void* out16, cudaStream_t s) {
    const int grid = static_cast<int>(rows / 8);
    uint16_t* o16 = static_cast<uint16_t*>(out16);
    if (kin == 2) fold_first_kernel<2><<<grid, 128, 0, s>>>(in, in_mod, W, bias, rows_per_sample, o16, rows);
    else if (kin == 3) fold_first_kernel<3><<<grid, 128, 0, s>>>(in, in_mod, W, bias, rows_per_sample, o16, rows);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}
cudaError_t launch_fold_tail16(const void* h3, const float* Wbc, const float* bbc, const float* Wc2, const float* bc2, long long rows,
                               int rows_per_sample, int channel_major, float* out, cudaStream_t s) {
    fold_tail16_kernel<<<static_cast<unsigned>((rows + 7) / 8), 256, 0, s>>>(static_cast<const uint16_t*>(h3), rows, Wbc, bbc, Wc2, bc2, rows,
                                                                            rows_per_sample, channel_major, out);
    return cudaGetLastError();
}
cudaError_t launch_fold_transpose(const float* U, int B, int P, float* out, cudaStream_t s) {
    const long long n = static_cast<long long>(B) * P;
    fold_transpose_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, s>>>(U, B, P, out);
    return cudaGetLastError();
}

}  // namespace pcd
