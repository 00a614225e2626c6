// Voxel-VAE decoder helpers (VAE3DLarge.decode, networks.py:2247-2264, 2327-2339) and the voxel -> point-cloud glue
// (utils.py:511-539).  The 3-D (transposed) convolutions themselves run on the tcgen05 GEMM of gemm_tc.cu as implicit GEMMs
// (ConvGeom in pcd_types.h); this file holds what is not a GEMM:
//   vae3d_final_conv_kernel   decoder.12 (Conv3d 32 -> 1, k = 3, padding 1) + Sigmoid on the channels-last 16-bit grid
//   vae3d_first_conv_kernel   encoder.0 (Conv3d 1 -> 32, k = 3, padding 1) + ReLU of VAE3DLarge.encode
//   voxel_count_kernel        per sample: number of voxels above the threshold
//   voxel_points_kernel       per sample: ordered stream compaction of those voxels into (x, y, z) in [-1, 1]
#include "pcd_launch.h"
#include "pcd_types.h"

namespace pcd {

// One thread per output voxel.  The grid is [planes][batch][D][H][W][ldc] 16-bit (hi plane, then the rounding-residual plane
// `plane_elems` elements further); weights w[27][cin] fp32 (tap-major) and the bias sit in shared memory.
template <int F16>
__global__ void __launch_bounds__(256)
vae3d_final_conv_kernel(const uint16_t* __restrict__ x, long long plane_elems, int planes, int ldc, int cin, int D, int H, int W,
                        long long nvox_total, const float* __restrict__ w, const float* __restrict__ bias, float* __restrict__ out) {
    extern __shared__ float sw[];            // [27 * cin + 1]
    for (int i = threadIdx.x; i < 27 * cin; i += blockDim.x) sw[i] = w[i];
    if (threadIdx.x == 0) sw[27 * cin] = bias[0];
    __syncthreads();
    const long long v = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (v >= nvox_total) return;
    const int xw = static_cast<int>(v % W), yh = static_cast<int>((v / W) % H), zd = static_cast<int>((v / (1LL * W * H)) % D);
    float acc = 0.f;
    for (int kd = 0; kd < 3; ++kd) {
        const int z2 = zd + kd - 1;
        if (z2 < 0 || z2 >= D) continue;
        for (int kh = 0; kh < 3; ++kh) {
            const int y2 = yh + kh - 1;
            if (y2 < 0 || y2 >= H) continue;
            for (int kw = 0; kw < 3; ++kw) {
                const int x2 = xw + kw - 1;
                if (x2 < 0 || x2 >= W) continue;
                const long long nb = v + (static_cast<long long>(kd - 1) * H + (kh - 1)) * W + (kw - 1);
                const uint4* ph = reinterpret_cast<const uint4*>(x + nb * ldc);
                const uint4* pl = reinterpret_cast<const uint4*>(x + plane_elems + nb * ldc);
                const float* wt = sw + ((kd * 3 + kh) * 3 + kw) * cin;
                for (int c8 = 0; c8 < cin / 8; ++c8) {
                    const uint4 a = ph[c8];
                    const uint32_t u[4] = {a.x, a.y, a.z, a.w};
                    float f[8];
#pragma unroll
                    for (int j = 0; j < 4; ++j) { const float2 t = unpack16x2(u[j], F16); f[2 * j] = t.x; f[2 * j + 1] = t.y; }
                    if (planes == 2) {
                        const uint4 b = pl[c8];
                        const uint32_t ul[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
                        for (int j = 0; j < 4; ++j) { const float2 t = unpack16x2(ul[j], F16); f[2 * j] += t.x; f[2 * j + 1] += t.y; }
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc = fmaf(wt[c8 * 8 + j], f[j], acc);
                }
            }
        }
    }
    acc += sw[27 * cin];
    out[v] = 1.f / (1.f + expf(-acc));       // nn.Sigmoid (networks.py:2263)
}

cudaError_t launch_vae3d_final_conv(const void* x, long long plane_elems, int planes, int f16, int ldc, int cin, int D, int H, int W,
                                    long long nvox_total, const float* w, const float* bias, float* out, cudaStream_t s) {
    if (cin % 8 != 0 || ldc % 8 != 0) return cudaErrorInvalidValue;
    const int grid = static_cast<int>((nvox_total + 255) / 256);
    const size_t smem = sizeof(float) * (27 * cin + 1);
    if (f16) vae3d_final_conv_kernel<1><<<grid, 256, smem, s>>>(static_cast<const uint16_t*>(x), plane_elems, planes, ldc, cin, D, H, W, nvox_total, w, bias, out);
    else     vae3d_final_conv_kernel<0><<<grid, 256, smem, s>>>(static_cast<const uint16_t*>(x), plane_elems, planes, ldc, cin, D, H, W, nvox_total, w, bias, out);
    return cudaGetLastError();
}

// encoder.0 of VAE3DLarge.encode: Conv3d(1 -> 32, k = 3, padding 1) + ReLU on the fp32 occupancy grid [B][32^3], one thread per
// voxel, written as the dense 32-channel 16-bit rows ([plane][Bpad][32^3][32], hi then rounding-residual plane) that encoder.2
// reads.  Weights w[27][32] (tap-major) and the bias sit in shared memory.
template <int F16>
__global__ void __launch_bounds__(256)
vae3d_first_conv_kernel(const float* __restrict__ vox, long long nvox_total, const float* __restrict__ w, const float* __restrict__ bias,
                        uint16_t* __restrict__ hi, uint16_t* __restrict__ lo) {
    constexpr int G = 32, C = 32;
    __shared__ float sw[27 * C + C];
    for (int i = threadIdx.x; i < 27 * C; i += blockDim.x) sw[i] = w[i];
    if (threadIdx.x < C) sw[27 * C + threadIdx.x] = bias[threadIdx.x];
    __syncthreads();
    const long long v = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (v >= nvox_total) return;
    const int xw = static_cast<int>(v % G), yh = static_cast<int>((v / G) % G), zd = static_cast<int>((v / (G * G)) % G);
    float acc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = sw[27 * C + c];
    for (int kd = 0; kd < 3; ++kd) {
        const int z2 = zd + kd - 1;
        if (z2 < 0 || z2 >= G) continue;
        for (int kh = 0; kh < 3; ++kh) {
            const int y2 = yh + kh - 1;
            if (y2 < 0 || y2 >= G) continue;
            for (int kw = 0; kw < 3; ++kw) {
                const int x2 = xw + kw - 1;
                if (x2 < 0 || x2 >= G) continue;
                const float x = __ldg(vox + v + ((kd - 1) * G + (kh - 1)) * G + (kw - 1));
                const float* wt = sw + ((kd * 3 + kh) * 3 + kw) * C;
#pragma unroll
                for (int c = 0; c < C; ++c) acc[c] = fmaf(wt[c], x, acc[c]);
            }
        }
    }
    uint4* ph = reinterpret_cast<uint4*>(hi + v * C);
    uint4* pl = lo ? reinterpret_cast<uint4*>(lo + v * C) : nullptr;
#pragma unroll
    for (int c8 = 0; c8 < C / 8; ++c8) {
        float f[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = fmaxf(acc[c8 * 8 + j], 0.f);
        const uint32_t h0 = pack16x2(f[0], f[1], F16), h1 = pack16x2(f[2], f[3], F16);
        const uint32_t h2 = pack16x2(f[4], f[5], F16), h3 = pack16x2(f[6], f[7], F16);
        ph[c8] = make_uint4(h0, h1, h2, h3);
        if (pl) {
            const float2 r0 = unpack16x2(h0, F16), r1 = unpack16x2(h1, F16), r2 = unpack16x2(h2, F16), r3 = unpack16x2(h3, F16);
            pl[c8] = make_uint4(pack16x2(f[0] - r0.x, f[1] - r0.y, F16), pack16x2(f[2] - r1.x, f[3] - r1.y, F16),
                                pack16x2(f[4] - r2.x, f[5] - r2.y, F16), pack16x2(f[6] - r3.x, f[7] - r3.y, F16));
        }
    }
}

cudaError_t launch_vae3d_first_conv(const float* vox, long long nvox_total, const float* w, const float* bias, void* hi, void* lo,
                                    int f16, cudaStream_t s) {
    const int grid = static_cast<int>((nvox_total + 255) / 256);
    if (f16) vae3d_first_conv_kernel<1><<<grid, 256, 0, s>>>(vox, nvox_total, w, bias, static_cast<uint16_t*>(hi), static_cast<uint16_t*>(lo));
    else     vae3d_first_conv_kernel<0><<<grid, 256, 0, s>>>(vox, nvox_total, w, bias, static_cast<uint16_t*>(hi), static_cast<uint16_t*>(lo));
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------------
// voxel_tensor_to_point_clouds (utils.py:511-539): per sample, the voxels with value > threshold in torch.where order
// (z, then y, then x ascending = ascending linear index), as points (x, y, z) mapped to [-1, 1] by 2 * p / (dim - 1) - 1.
// One CTA per sample; thread t owns the `chunk` consecutive voxels [t * chunk, (t + 1) * chunk).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kVoxThreads = 1024;

__device__ __forceinline__ int block_exclusive_scan(int v, int* total) {
    __shared__ int warp_sums[kVoxThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int s = warp_sums[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += n;
        }
        warp_sums[lane] = s;
    }
    __syncthreads();
    *total = warp_sums[kVoxThreads / 32 - 1];
    return incl - v + (warp > 0 ? warp_sums[warp - 1] : 0);
}

__global__ void __launch_bounds__(kVoxThreads)
voxel_count_kernel(const float* __restrict__ vox, int nvox, float threshold, int* __restrict__ counts) {
    const float* v = vox + static_cast<long long>(blockIdx.x) * nvox;
    const int chunk = (nvox + kVoxThreads - 1) / kVoxThreads;
    const int lo = threadIdx.x * chunk, hi = min(lo + chunk, nvox);
    int c = 0;
    for (int i = lo; i < hi; ++i) c += v[i] > threshold ? 1 : 0;
    int total;
    block_exclusive_scan(c, &total);
    if (threadIdx.x == 0) counts[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kVoxThreads)
voxel_points_kernel(const float* __restrict__ vox, int D, int H, int W, float threshold, const long long* __restrict__ offsets,
                    float* __restrict__ pts) {
    const int nvox = D * H * W;
    const float* v = vox + static_cast<long long>(blockIdx.x) * nvox;
    const int chunk = (nvox + kVoxThreads - 1) / kVoxThreads;
    const int lo = threadIdx.x * chunk, hi = min(lo + chunk, nvox);
    int c = 0;
    for (int i = lo; i < hi; ++i) c += v[i] > threshold ? 1 : 0;
    int total;
    long long o = offsets[blockIdx.x] + block_exclusive_scan(c, &total);
    // utils.py:533: 2 * points / tensor([W - 1, H - 1, D - 1]) - 1 in fp32, in that order
    const float fw = static_cast<float>(W - 1), fh = static_cast<float>(H - 1), fd = static_cast<float>(D - 1);
    for (int i = lo; i < hi; ++i) {
        if (!(v[i] > threshold)) continue;
        const int x = i % W, y = (i / W) % H, z = i / (W * H);
        pts[o * 3 + 0] = __fsub_rn(__fdiv_rn(__fmul_rn(2.f, static_cast<float>(x)), fw), 1.f);
        pts[o * 3 + 1] = __fsub_rn(__fdiv_rn(__fmul_rn(2.f, static_cast<float>(y)), fh), 1.f);
        pts[o * 3 + 2] = __fsub_rn(__fdiv_rn(__fmul_rn(2.f, static_cast<float>(z)), fd), 1.f);
        ++o;
    }
}

cudaError_t launch_voxel_count(const float* vox, int B, int nvox, float threshold, int* counts, cudaStream_t s) {
    voxel_count_kernel<<<B, kVoxThreads, 0, s>>>(vox, nvox, threshold, counts);
    return cudaGetLastError();
}
cudaError_t launch_voxel_points(const float* vox, int B, int D, int H, int W, float threshold, const long long* offsets, float* pts,
                                cudaStream_t s) {
    voxel_points_kernel<<<B, kVoxThreads, 0, s>>>(vox, D, H, W, threshold, offsets, pts);
    return cudaGetLastError();
}

// fp32 channels-last [rows][c_src] -> 16-bit [rows][c_dst] hi (+ lo) planes, zero-padding channels c_src..c_dst-1
// (decoder_input output -> first activation grid)
__global__ void f32_rows_to_16_kernel(const float* __restrict__ in, int c_src, uint16_t* __restrict__ hi, uint16_t* __restrict__ lo,
                                      int c_dst, long long rows, int f16) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= rows * c_dst) return;
    const long long r = i / c_dst; const int c = static_cast<int>(i - r * c_dst);
    const float v = c < c_src ? in[r * c_src + c] : 0.f;
    const uint16_t h = pack16(v, f16);
    hi[i] = h;
    if (lo) lo[i] = pack16(v - unpack16(h, f16), f16);
}
cudaError_t launch_f32_rows_to_16(const float* in, int c_src, void* hi, void* lo, int c_dst, long long rows, int f16, cudaStream_t s) {
    const long long n = rows * c_dst;
    f32_rows_to_16_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, s>>>(in, c_src, static_cast<uint16_t*>(hi), static_cast<uint16_t*>(lo), c_dst, rows, f16);
    return cudaGetLastError();
}

// 16-bit [rows][c_src_ld] (hi + optional lo) -> fp32 [rows][c_keep]   (debug taps)
__global__ void rows16_to_f32_kernel(const uint16_t* __restrict__ hi, const uint16_t* __restrict__ lo, int ld, float* __restrict__ out,
                                     int c_keep, long long rows, int f16) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= rows * c_keep) return;
    const long long r = i / c_keep; const int c = static_cast<int>(i - r * c_keep);
    out[i] = unpack16(hi[r * ld + c], f16) + (lo ? unpack16(lo[r * ld + c], f16) : 0.f);
}
cudaError_t launch_rows16_to_f32(const void* hi, const void* lo, int ld, float* out, int c_keep, long long rows, int f16, cudaStream_t s) {
    const long long n = rows * c_keep;
    rows16_to_f32_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, s>>>(static_cast<const uint16_t*>(hi), static_cast<const uint16_t*>(lo), ld, out, c_keep, rows, f16);
    return cudaGetLastError();
}

}  // namespace pcd
