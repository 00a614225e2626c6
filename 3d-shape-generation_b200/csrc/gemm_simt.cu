// CUDA-core fp32 kernels: the 'fp32' precision mode of the per-point layers (parity at 1e-5,
// separates algorithm bugs from tensor-core bugs), the per-sample side GEMMs (time MLP,
// hoisted time/global-feature biases: networks.py:737-741,796-797,808,811), the K=3 first
// layer, the unfused final layer of fp32 mode, and small utilities.
#include "pcd_launch.h"
#include "pcd_sampler.cuh"
#include "pcd_ptx.cuh"
#include "pcd_types.h"

namespace pcd {

// ------------------------------------------------------------------------------------------
// 64x64x16 register-tiled fp32 GEMM, 256 threads, 4x4 outputs per thread.
// ------------------------------------------------------------------------------------------
template <int EPI>
__global__ void __launch_bounds__(256) gemm_simt_kernel(const SimtGemmParams p) {
    __shared__ float As[2][16][64 + 4];
    __shared__ float Ws[2][16][64 + 4];
    pdl_launch(); pdl_wait();
    const int tid = threadIdx.x;
    const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
    const int lr = tid >> 2, lk = (tid & 3) * 4;   // loader: row 0..63, k offset 0,4,8,12
    const int ty = tid >> 4, tx = tid & 15;        // compute: 16x16 threads
    float acc[4][4] = {};
    const int K = p.K0 + p.K1;
    // split-K: blockIdx.z owns the k range [kbeg, kend); partial sums go to p.partial (fixed-order reduce later)
    const int nsplit = gridDim.z;
    const int kper = K / nsplit;
    const int kbeg = blockIdx.z * kper, kend = kbeg + kper;
    const int ar = m0 + lr, wr = n0 + lr;
    auto load_tile = [&](int k0, float4& a, float4& w) {
        a = make_float4(0.f, 0.f, 0.f, 0.f); w = a;
        if (ar < p.M) {
            const int k = k0 + lk;
            a = (k < p.K0) ? *reinterpret_cast<const float4*>(p.A0 + static_cast<long long>(ar) * p.lda0 + k)
                           : *reinterpret_cast<const float4*>(p.A1 + static_cast<long long>(ar) * p.lda1 + (k - p.K0));
        }
        if (wr < p.Nout) w = *reinterpret_cast<const float4*>(p.W + static_cast<long long>(wr) * p.ldw + k0 + lk);
    };
    float4 a, w;
    load_tile(kbeg, a, w);
    int buf = 0;
    for (int k0 = kbeg; k0 < kend; k0 += 16) {
        As[buf][lk + 0][lr] = a.x; As[buf][lk + 1][lr] = a.y; As[buf][lk + 2][lr] = a.z; As[buf][lk + 3][lr] = a.w;
        Ws[buf][lk + 0][lr] = w.x; Ws[buf][lk + 1][lr] = w.y; Ws[buf][lk + 2][lr] = w.z; Ws[buf][lk + 3][lr] = w.w;
        __syncthreads();
        if (k0 + 16 < kend) load_tile(k0 + 16, a, w);   // register prefetch overlaps the FMAs below
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const float4 av = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
            const float4 wv = *reinterpret_cast<const float4*>(&Ws[buf][k][tx * 4]);
            const float ar4[4] = {av.x, av.y, av.z, av.w}, wr4[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar4[i], wr4[j], acc[i][j]);
        }
        buf ^= 1;   // two buffers: the store of iteration i+1 cannot race with the reads of iteration i-1 (one barrier apart)
    }
    if (nsplit > 1) {
        float* part = p.partial + static_cast<long long>(blockIdx.z) * p.M * p.Nout;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = m0 + ty * 4 + i;
            if (r >= p.M) continue;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = n0 + tx * 4 + j;
                if (c < p.Nout) part[static_cast<long long>(r) * p.Nout + c] = acc[i][j];
            }
        }
        return;
    }
    if constexpr (EPI == EPI_STORE) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = m0 + ty * 4 + i;
            if (r >= p.M) continue;
            const int sample = r / p.rows_per_sample;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = n0 + tx * 4 + j;
                if (c >= p.Nout) continue;
                float v = acc[i][j];
                if (p.bias) v += p.bias[static_cast<long long>(sample) * p.bias_sample_stride + c];
                if (p.relu) v = fmaxf(v, 0.f);
                p.out[static_cast<long long>(r) * p.ldo + c] = v;
            }
        }
    } else {  // EPI_MAXPOOL: rows = points (a 64-row tile never straddles clouds: 64 | Npad)
        const int sample = m0 / p.rows_per_sample;
        const int nbase = m0 - sample * p.rows_per_sample + ty * 4;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = n0 + tx * 4 + j;
            if (c >= p.Nout) continue;
            float mx = -3.0e38f;
            bool any = false;
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (nbase + i < p.n_valid && m0 + ty * 4 + i < p.M) { mx = fmaxf(mx, acc[i][j]); any = true; }
            if (any) atomic_max_nonneg(&p.gmax[static_cast<long long>(sample) * p.ld_g + c], fmaxf(mx + p.bias[c], 0.f));
        }
    }
}

// out[r][c] = act(bias[c] + sum_s partial[s][r][c]) in a fixed order (deterministic split-K)
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ partial, int nsplit, const float* __restrict__ bias,
                                                            float* __restrict__ out, int M, int Nout, int relu) {
    pdl_launch(); pdl_wait();
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long n = static_cast<long long>(M) * Nout;
    if (i >= n) return;
    float v = bias ? bias[i % Nout] : 0.f;
    for (int s = 0; s < nsplit; ++s) v += partial[s * n + i];
    out[i] = relu ? fmaxf(v, 0.f) : v;
}
cudaError_t launch_splitk_reduce(const float* partial, int nsplit, const float* bias, float* out, int M, int Nout, int relu,
                                 cudaStream_t stream) {
    const long long n = static_cast<long long>(M) * Nout;
    return launch_pdl(splitk_reduce_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, stream, partial, nsplit, bias, out, M, Nout, relu);
}

// Skinny split-K GEMM for M <= 8 rows (dec4's per-sample bias at small batch: [B, 4096] x [4096, 1024]): the 64-row tiles of
// gemm_simt_kernel are 94 % padding there and every k-step is a shared-memory tile hand-over (21 us at batch 4 for 17 MB of
// weights).  One CTA per (32 output columns, k split): the W slab [32][kper] is read with one coalesced 512-byte row segment per
// warp load into padded shared memory, then thread (row r = warp, column c = lane) runs the SAME accumulation as gemm_simt_kernel
// -- ONE fmaf chain from 0 over the split's k range in ascending order -- so the partial sums, and after splitk_reduce_kernel the
// result, are bit-identical to the tiled kernel's: a sample does not change with the batch size it is generated in.
__global__ void __launch_bounds__(256) skinny_splitk_kernel(const float* __restrict__ A, int lda, const float* __restrict__ W, int ldw,
                                                            int M, int Nout, int kper, float* __restrict__ partial) {
    __shared__ float Ws[32][129];
    __shared__ __align__(16) float As[8][128];
    pdl_launch(); pdl_wait();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c0 = blockIdx.x * 32, split = blockIdx.y;
    float acc = 0.f;
    for (int kc = 0; kc < kper; kc += 128) {
        const long long kb = static_cast<long long>(split) * kper + kc;
        if (kc) __syncthreads();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int row = warp * 4 + i;
            const float4 v = __ldg(reinterpret_cast<const float4*>(W + static_cast<long long>(c0 + row) * ldw + kb) + lane);
            Ws[row][4 * lane] = v.x; Ws[row][4 * lane + 1] = v.y; Ws[row][4 * lane + 2] = v.z; Ws[row][4 * lane + 3] = v.w;
        }
        if (warp < M)
            *reinterpret_cast<float4*>(&As[warp][4 * lane]) = __ldg(reinterpret_cast<const float4*>(A + static_cast<long long>(warp) * lda + kb) + lane);
        __syncthreads();
        if (warp < M) {
#pragma unroll 16
            for (int k = 0; k < 128; ++k) acc = fmaf(As[warp][k], Ws[lane][k], acc);
        }
    }
    if (warp < M) partial[(static_cast<long long>(split) * M + warp) * Nout + c0 + lane] = acc;
}

bool skinny_splitk_ok(const SimtGemmParams& p) {
    return p.partial != nullptr && p.splits > 1 && p.M <= 8 && p.K1 == 0 && (p.Nout & 31) == 0 && p.K0 % p.splits == 0 &&
           (p.K0 / p.splits) % 128 == 0 && (p.lda0 & 3) == 0 && (p.ldw & 3) == 0;
}

// partial sums only: the caller runs launch_splitk_reduce afterwards, exactly as after launch_gemm_simt with splits > 1
cudaError_t launch_skinny_splitk(const SimtGemmParams& p, cudaStream_t stream) {
    return launch_pdl(skinny_splitk_kernel, dim3(p.Nout / 32, p.splits), dim3(256), 0, stream, p.A0, p.lda0, p.W, p.ldw, p.M, p.Nout,
                      p.K0 / p.splits, p.partial);
}

// number of k-splits that fills the GPU for a skinny problem (M small): power of two, K/splits a multiple of 64
int simt_pick_splits(int M, int Nout, int K, int num_sms) {
    const int ctas = ((M + 63) / 64) * ((Nout + 63) / 64);
    int s = 1;
    while (ctas * s < 2 * num_sms && K % (s * 2 * 64) == 0 && s < 32) s *= 2;
    return s;
}

cudaError_t launch_gemm_simt(int epi, const SimtGemmParams& p, cudaStream_t stream) {
    const int splits = (p.partial != nullptr && p.splits > 1 && epi == EPI_STORE) ? p.splits : 1;
    dim3 grid((p.Nout + 63) / 64, (p.M + 63) / 64, splits);
    if (epi == EPI_STORE) return launch_pdl(gemm_simt_kernel<EPI_STORE>, grid, dim3(256), 0, stream, p);
    if (epi == EPI_MAXPOOL) return launch_pdl(gemm_simt_kernel<EPI_MAXPOOL>, grid, dim3(256), 0, stream, p);
    return cudaErrorInvalidValue;
}

// ------------------------------------------------------------------------------------------
// Per-sample time path (networks.py:791-792, 820-838) + hoisted enc1.conv1 time bias:
//   temb = W2 * silu(W1 * [sin(t f), cos(t f)] + b1) + b2
//   bias1[b][c] = scale1[c]*(Wt[c,:] . temb + b_conv[c] - mu[c]) + beta[c]   (pre-folded: Wt', b')
// One CTA (256 threads) per sample row.  W1/W2/Wt are stored TRANSPOSED ([in][out]).
// ------------------------------------------------------------------------------------------
// One dense stage of the time path on a 256-thread CTA: out[o] = act(b[o] + sum_k W[k][o] * in[k]), o < NO, k < K, W stored
// transposed ([K][NO]: a warp's loads are coalesced).  Warp w owns a K slice and every lane carries 8 independent accumulators
// (outputs lane + 32 j), so 8 loads are in flight per k instead of one dependent chain of K loads per thread -- this kernel runs
// on B CTAs only and sits on the critical path of every reverse step (41 us of a 378 us step at batch 4 before this form).
template <int ACT>   // 0 none, 1 SiLU
__device__ __forceinline__ void tb_stage(const float* __restrict__ W, const float* __restrict__ b, const float* in, float* out,
                                         float (*red)[256], int K, int NO) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int kper = (K + 7) >> 3, k0 = warp * kper, k1 = min(K, k0 + kper);
    for (int ob = 0; ob < NO; ob += 256) {
        float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
        for (int k = k0; k < k1; ++k) {
            const float x = in[k];
            const float* w = W + static_cast<size_t>(k) * NO + ob + lane;
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (ob + lane + 32 * j < NO) acc[j] = fmaf(__ldg(w + 32 * j), x, acc[j]);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) red[warp][lane + 32 * j] = acc[j];
        __syncthreads();
        if (ob + tid < NO) {
            float s = b[ob + tid];
#pragma unroll
            for (int w8 = 0; w8 < 8; ++w8) s += red[w8][tid];      // fixed order: deterministic
            out[ob + tid] = ACT == 1 ? s / (1.f + expf(-s)) : s;
        }
        __syncthreads();
    }
}

// per_step != 0 (sampler calls): one CTA per reverse STEP, t = that step's schedule entry -- the whole loop's time path in one
// launch before the loop; per_step == 0 (forward hook): one CTA per sample, t = t_in[sample].
__global__ void __launch_bounds__(256) time_bias_kernel(const CallArgs* __restrict__ ca, int T, int per_step,
                                                        const float* __restrict__ freqs,  // [T / 2]
                                                        const float* __restrict__ W1, const float* __restrict__ b1,
                                                        const float* __restrict__ W2, const float* __restrict__ b2,
                                                        const float* __restrict__ Wt,  // [T][64] folded, transposed
                                                        const float* __restrict__ bt,  // [64] folded
                                                        float* __restrict__ temb_out,  // [rows][T] (debug tap)
                                                        float* __restrict__ bias1_out /* [rows][64] */) {
    extern __shared__ float tb_smem[];           // e | h | o, T floats each (T = dim = time_dim; 256 in the reference defaults)
    __shared__ float red[8][256];
    float* e = tb_smem; float* h = e + T; float* o = h + T;
    pdl_launch(); pdl_wait();
    const int b = blockIdx.x, tid = threadIdx.x, half = T >> 1;
    // every sample of a step shares t, also with per-sample schedule rows ('linear'): row 0 of the step
    const float t = per_step ? ca->s.sched[static_cast<long long>(b) * ca->s.sched_rows * kSchedRow + 5] : ca->t_in[b];
    for (int i = tid; i < T; i += 256) {
        // networks.py:834-837: [sin(t f) | cos(t f)], an odd embedding_dim is zero padded
        const int j = i < half ? i : i - half;
        const float a = t * freqs[j < half ? j : 0];
        e[i] = i < half ? sinf(a) : (i < 2 * half ? cosf(a) : 0.f);
    }
    __syncthreads();
    tb_stage<1>(W1, b1, e, h, red, T, T);            // Linear -> SiLU      (networks.py:737-741)
    tb_stage<0>(W2, b2, h, o, red, T, T);            // Linear = temb
    for (int i = tid; i < T; i += 256) temb_out[static_cast<long long>(b) * T + i] = o[i];
    tb_stage<0>(Wt, bt, o, bias1_out + b * 64, red, T, 64);   // hoisted temb columns of enc1.conv1 (+ folded BN bias)
}

cudaError_t launch_time_bias(int rows, int T, int per_step, const CallArgs* ca, const float* freqs,
                             const float* W1, const float* b1, const float* W2, const float* b2, const float* Wt,
                             const float* bt, float* temb_out, float* bias1_out, cudaStream_t stream) {
    return launch_pdl(time_bias_kernel, dim3(rows), dim3(256), 3 * sizeof(float) * T, stream, ca, T, per_step, freqs, W1, b1, W2, b2, Wt, bt,
                      temb_out, bias1_out);
}

// ------------------------------------------------------------------------------------------
// enc1.conv1 with the time channels hoisted (K = 3): h[row][c] = relu(Wx[c,:] . x[row] + bias1[b][c])
// 128 padded rows per CTA (one sample per CTA: 128 | Npad), 64 outputs per row, written as 16-bit planes or fp32.
// 16-bit form: eight threads share a row and own eight channels each, so a warp stores 4 rows x 128 contiguous bytes per
// instruction (one row per thread scattered every 16-byte store over 32 lines: 0.19 ms for 0.27 GB at batch 512).
// ------------------------------------------------------------------------------------------
template <typename OutT>
__global__ void __launch_bounds__(128) enc1_first_kernel(const CallArgs* __restrict__ ca, const float* __restrict__ Wx /*[64][3]*/,
                                                         const float* __restrict__ bias1, long long bias_stride,
                                                         OutT* __restrict__ out, OutT* __restrict__ out_lo, int B, int N, int Npad,
                                                         int f16) {
    __shared__ float sw[64 * 3];
    __shared__ float sb[64];
    __shared__ float sx[128 * 3];
    pdl_launch(); pdl_wait();
    const long long row0 = static_cast<long long>(blockIdx.x) * 128;
    const int b = static_cast<int>(row0 / Npad);  // 128 | Npad: uniform per CTA
    for (int i = threadIdx.x; i < 192; i += 128) sw[i] = Wx[i];
    if (threadIdx.x < 64)      // sampler calls: this step's row of the per-call table; forward hook: the sample's row
        sb[threadIdx.x] = ca->bias1_steps ? ca->bias1_steps[static_cast<long long>(*ca->s.step_ptr) * 64 + threadIdx.x]
                                          : bias1[b * bias_stride + threadIdx.x];
    {
        const int n = static_cast<int>(row0 - static_cast<long long>(b) * Npad) + threadIdx.x;
        float x0 = 0.f, x1 = 0.f, x2 = 0.f;
        if (n < N) {
            const float* xp = ca->s.x + (static_cast<long long>(b) * N + n) * 3;
            x0 = xp[0]; x1 = xp[1]; x2 = xp[2];
        }
        sx[threadIdx.x * 3] = x0; sx[threadIdx.x * 3 + 1] = x1; sx[threadIdx.x * 3 + 2] = x2;
    }
    __syncthreads();
    if constexpr (sizeof(OutT) == 2) {
        const int c8 = threadIdx.x & 7;                 // channels 8 c8 .. 8 c8 + 7
#pragma unroll 4
        for (int it = 0; it < 8; ++it) {
            const int r = it * 16 + (threadIdx.x >> 3);
            const float x0 = sx[r * 3], x1 = sx[r * 3 + 1], x2 = sx[r * 3 + 2];
            uint32_t pk[4], pl[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = c8 * 8 + 2 * j;
                float a = fmaf(sw[c * 3 + 2], x2, fmaf(sw[c * 3 + 1], x1, fmaf(sw[c * 3], x0, sb[c])));
                float d = fmaf(sw[c * 3 + 5], x2, fmaf(sw[c * 3 + 4], x1, fmaf(sw[c * 3 + 3], x0, sb[c + 1])));
                a = fmaxf(a, 0.f); d = fmaxf(d, 0.f);
                pk[j] = pack16x2(a, d, f16);
                const float2 back = unpack16x2(pk[j], f16);
                pl[j] = pack16x2(a - back.x, d - back.y, f16);
            }
            const long long row = row0 + r;
            reinterpret_cast<uint4*>(out + row * 64)[c8] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            if (out_lo) reinterpret_cast<uint4*>(out_lo + row * 64)[c8] = make_uint4(pl[0], pl[1], pl[2], pl[3]);
        }
    } else {
        const float x0 = sx[threadIdx.x * 3], x1 = sx[threadIdx.x * 3 + 1], x2 = sx[threadIdx.x * 3 + 2];
        OutT* orow = out + (row0 + threadIdx.x) * 64;
#pragma unroll
        for (int c4 = 0; c4 < 16; ++c4) {
            float v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = c4 * 4 + j;
                v[j] = fmaxf(fmaf(sw[c * 3 + 2], x2, fmaf(sw[c * 3 + 1], x1, fmaf(sw[c * 3], x0, sb[c]))), 0.f);
            }
            reinterpret_cast<float4*>(orow)[c4] = make_float4(v[0], v[1], v[2], v[3]);
        }
    }
}

cudaError_t launch_enc1_first(int elt_bytes, int f16, const CallArgs* x, const float* Wx, const float* bias1, long long bias_stride,
                              void* out, void* out_lo, int B, int N, int Npad, cudaStream_t stream) {
    const int grid = static_cast<int>((static_cast<long long>(B) * Npad) / 128);
    if (elt_bytes == 2)
        return launch_pdl(enc1_first_kernel<uint16_t>, dim3(grid), dim3(128), 0, stream, x, Wx, bias1, bias_stride, static_cast<uint16_t*>(out),
                          static_cast<uint16_t*>(out_lo), B, N, Npad, f16);
    return launch_pdl(enc1_first_kernel<float>, dim3(grid), dim3(128), 0, stream, x, Wx, bias1, bias_stride, static_cast<float*>(out),
                      static_cast<float*>(nullptr), B, N, Npad, 0);
}

// ------------------------------------------------------------------------------------------
// fp32 mode tail: output.3 (64 -> 3) + sampler update from the fp32 [rows][64] activation.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) final_simt_kernel(const float* __restrict__ h, long long rows, const CallArgs* __restrict__ ca) {
    pdl_launch(); pdl_wait();
    const SamplerArgs& s = ca->s;
    __shared__ float sw3[195];
    for (int i = threadIdx.x; i < 192; i += 128) sw3[i] = s.w3[i];
    if (threadIdx.x < 3) sw3[192 + threadIdx.x] = s.b3[threadIdx.x];
    __syncthreads();
    const long long row = static_cast<long long>(blockIdx.x) * 128 + threadIdx.x;
    if (row >= rows) return;
    float e0 = sw3[192], e1 = sw3[193], e2 = sw3[194];
    const float4* hp = reinterpret_cast<const float4*>(h + row * 64);
#pragma unroll
    for (int j4 = 0; j4 < 16; ++j4) {
        const float4 v = hp[j4];
        const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            e0 = fmaf(sw3[j4 * 4 + j], vv[j], e0);
            e1 = fmaf(sw3[64 + j4 * 4 + j], vv[j], e1);
            e2 = fmaf(sw3[128 + j4 * 4 + j], vv[j], e2);
        }
    }
    sampler_apply(s, row, e0, e1, e2);
}

cudaError_t launch_final_simt(const float* h, long long rows, const CallArgs* ca, cudaStream_t stream) {
    return launch_pdl(final_simt_kernel, dim3(static_cast<unsigned>((rows + 127) / 128)), dim3(128), 0, stream, h, rows, ca);
}

// ------------------------------------------------------------------------------------------
// utilities
// ------------------------------------------------------------------------------------------
__global__ void advance_step_kernel(int* step) { pdl_launch(); pdl_wait(); *step += 1; }
__global__ void __launch_bounds__(256) zero_f32_kernel(float* __restrict__ p, long long n) {
    pdl_launch(); pdl_wait();
    const long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
    if (i < n) p[i] = 0.f;
}
cudaError_t launch_zero_f32(float* p, long long n, cudaStream_t stream) {
    return launch_pdl(zero_f32_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, stream, p, n);
}
cudaError_t launch_advance_step(int* step, cudaStream_t stream) {
    return launch_pdl(advance_step_kernel, dim3(1), dim3(1), 0, stream, step);
}

__global__ void philox_fill_kernel(float* out, unsigned long long seed, unsigned long long sample_offset, int step, int B,
                                   int N) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= static_cast<long long>(B) * N) return;
    const int b = static_cast<int>(i / N), n = static_cast<int>(i - static_cast<long long>(b) * N);
    float z0, z1, z2;
    philox_normal3(seed, sample_offset + b, static_cast<uint32_t>(step), static_cast<uint32_t>(n), z0, z1, z2);
    out[i * 3 + 0] = z0; out[i * 3 + 1] = z1; out[i * 3 + 2] = z2;
}
cudaError_t launch_philox_fill(float* out, unsigned long long seed, unsigned long long sample_offset, int step, int B, int N,
                               cudaStream_t stream) {
    const long long n = static_cast<long long>(B) * N;
    philox_fill_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, stream>>>(out, seed, sample_offset, step, B, N);
    return cudaGetLastError();
}

// fp32 <-> 16-bit (bf16 or fp16, `f16` selects) conversions; the split form writes v = hi + lo planes
__global__ void f32_to_16_kernel(const float* __restrict__ in, uint16_t* __restrict__ out, long long n, int f16) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) out[i] = pack16(in[i], f16);
}
__global__ void f16b_to_f32_kernel(const uint16_t* __restrict__ in, const uint16_t* __restrict__ in_lo, float* __restrict__ out,
                                   long long n, int f16) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) out[i] = unpack16(in[i], f16) + (in_lo ? unpack16(in_lo[i], f16) : 0.f);
}
__global__ void f32_split_16_kernel(const float* __restrict__ in, uint16_t* __restrict__ hi, uint16_t* __restrict__ lo, long long n,
                                    int f16) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint16_t h = pack16(in[i], f16);
    hi[i] = h;
    lo[i] = pack16(in[i] - unpack16(h, f16), f16);
}
// weights of an fp8-corrected layer: fp16 hi plane + the e5m2 byte plane, per 32 k-elements [32 x e5m2(W_hi / kC8ScaleLo) | 32 x
// e5m2(W_lo / kC8ScaleHi)] -- the B-role mirror of the activations' [lo8 | hi8] half rows (gemm_tc.cu, NP == 4); k % 64 == 0
__global__ void f32_split_c8_kernel(const float* __restrict__ in, uint16_t* __restrict__ hi, uint8_t* __restrict__ c8, long long n, int k) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long r = i / k;
    const int kk = static_cast<int>(i - r * k), g = kk >> 5, j = kk & 31;
    const uint16_t h = pack16(in[i], 1);
    const float hv = unpack16(h, 1);
    hi[i] = h;
    uint8_t* row = c8 + r * (2LL * k) + g * 64;
    row[j] = __nv_cvt_float_to_fp8(hv * (1.f / kC8ScaleLo), __NV_SATFINITE, __NV_E5M2);
    row[32 + j] = __nv_cvt_float_to_fp8((in[i] - hv) * (1.f / kC8ScaleHi), __NV_SATFINITE, __NV_E5M2);
}
cudaError_t launch_f32_split_c8(const float* in, void* hi, void* c8, long long rows, int k, cudaStream_t stream) {
    const long long n = rows * k;
    f32_split_c8_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, stream>>>(in, static_cast<uint16_t*>(hi), static_cast<uint8_t*>(c8), n, k);
    return cudaGetLastError();
}
// activations with a c8 second plane back to fp32 (taps): hi + residual byte / kC8ScaleLo
__global__ void f16c8_to_f32_kernel(const uint16_t* __restrict__ in, const uint8_t* __restrict__ c8, float* __restrict__ out, long long n, int k) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long r = i / k;
    const int kk = static_cast<int>(i - r * k), g = kk >> 5, j = kk & 31;
    const __half_raw lo = __nv_cvt_fp8_to_halfraw(c8[r * (2LL * k) + g * 64 + j], __NV_E5M2);
    out[i] = unpack16(in[i], 1) + __half2float(__half(lo)) * (1.f / kC8ScaleLo);
}
cudaError_t launch_16c8_to_f32(const void* in, const void* c8, float* out, long long rows, int k, cudaStream_t stream) {
    const long long n = rows * k;
    f16c8_to_f32_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, stream>>>(static_cast<const uint16_t*>(in), static_cast<const uint8_t*>(c8), out, n, k);
    return cudaGetLastError();
}
cudaError_t launch_f32_split_16(const float* in, void* hi, void* lo, long long n, int f16, cudaStream_t stream) {
    f32_split_16_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, stream>>>(in, static_cast<uint16_t*>(hi), static_cast<uint16_t*>(lo), n, f16);
    return cudaGetLastError();
}
cudaError_t launch_f32_to_16(const float* in, void* out, long long n, int f16, cudaStream_t stream) {
    f32_to_16_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, stream>>>(in, static_cast<uint16_t*>(out), n, f16);
    return cudaGetLastError();
}
cudaError_t launch_16_to_f32(const void* in, const void* in_lo, float* out, long long n, int f16, cudaStream_t stream) {
    f16b_to_f32_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, stream>>>(static_cast<const uint16_t*>(in),
                                                                           static_cast<const uint16_t*>(in_lo), out, n, f16);
    return cudaGetLastError();
}

}  // namespace pcd
