// Parameter blocks shared by the host plan (api.cu) and the kernels.
#pragma once
#include <cstdint>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>
#include <cuda.h>
#include <cuda_runtime.h>

namespace pcd {

constexpr int kSchedRow = 8;  // floats per schedule-table row: n, s, s_next, n_next, cz, t, -, -

// Sampler update fused behind the last layer (diffusion.py:154-168, 246-257, 283-287).
struct SamplerArgs {
    float* x;                      // [B, N, 3] fp32, updated in place (mode 1)
    float* eps_out;                // [B, N, 3] fp32 (mode 0: forward-only parity hook)
    const float* w3;               // output.3 weight [3][64] fp32
    const float* b3;               // output.3 bias [3]
    const float* sched;            // device table [S][sched_rows][kSchedRow]
    int sched_rows;                // rows per step: 1 = one schedule row shared by the batch, B = one row per sample
                                   // (the reference's 'linear' schedule cumprods over the batch axis, diffusion.py:202)
    const int* step_ptr;           // device step counter (advanced by a 1-thread kernel per step)
    const float* noise;            // injected noise [S-1][B][N][3] or nullptr
    long long noise_step_stride;   // B*N*3
    unsigned long long seed;       // Philox key (used when noise == nullptr and cz != 0)
    unsigned long long sample_offset;  // global index of sample 0 of this call (multi-GPU sharding)
    int N;                         // valid points per cloud
    int Npad;                      // rows per cloud in the activation layout (multiple of 128)
    int mode;                      // 0 = write eps, 1 = sampler update
};

// Everything that changes between API calls but not between graph replays is read through
// this device-resident block, so one captured step graph serves every call with the same (B, N).
struct CallArgs {
    SamplerArgs s;
    const float* t_in;   // per-sample t [B] (forward hook) or nullptr (sampler: t from the schedule table)
    const float* bias1_steps;   // sampler calls: enc1.conv1's hoisted time bias for EVERY step of the loop, [S][64], computed once per
                                // call (t depends on the step only, networks.py:791-797); nullptr in the forward hook
};

// latent path: per-call block (device resident, read by the graph's kernels)
struct LatentCall {
    float* z;                 // [B, D] fp32, updated in place (mode 1)
    float* eps_out;           // [B, D] (mode 0)
    const float* t_in;        // per-sample t or nullptr
    const float* sched;       // [S][sched_rows][kSchedRow]
    int sched_rows;           // rows per step: 1 = shared by the batch; B = one per sample ('linear' schedule: the reference cumprods
                              // over the batch axis, diffusion.py:553-569); 0 is read as 1
    const int* step_ptr;
    const float* noise;       // injected [S-1][B][D] or nullptr
    long long noise_step_stride;
    unsigned long long seed, sample_offset;
    int B, D, mode;
};

// latent persistent kernel (latent_mk.cu): one phase of the per-step "program" walked by every CTA
enum LtKind { LT_GEMM = 0, LT_NORM = 1, LT_EMB = 2, LT_TAIL = 3, LT_HEAD = 4 };
enum LtEpi { LT_PARTIAL = 0, LT_BIAS = 1, LT_BIAS_RELU = 2, LT_BIAS_SILU = 3, LT_FINAL = 4 };
struct LtOp {
    int kind;                // LtKind
    int rows_mode;           // 0: rows = samples (B); 1: rows = time rows (R = S in the samplers, B in the forward hook)
    // LT_GEMM: out = [A0 | A1] W^T over 128 x 64 tiles, K split `ks` ways
    const float* A0; int lda0; int K0;
    const float* A1; int lda1; int K1;
    const float* W; int kchunks;         // tile-major pre-swizzled weights [N / bn][kchunks][bn x 32], kchunks = (K0 + K1) / 32
    int N, ks, chunks_per_split;         // (K0 + K1) / 32 / ks
    int bn;                              // tile columns: 64, or 128 for the big split-K layers (LT_PARTIAL only)
    int epi;                             // LtEpi
    float* out; int ldo;                 // LT_PARTIAL: workspace [ks][rows][N]; otherwise the layer output (also LT_NORM / LT_EMB)
    const float* bias; int bias_mode; int bias_ld;   // 0: shared [N]; 1: one row per time row (forward: row = sample, else = step)
    // LT_NORM: out = relu(GroupNorm8(bias + sum_s partial[s])) (gamma == nullptr: bias + optional ReLU only)
    const float* partial; int nsplit;
    const float* gamma; const float* beta;
    int act, C;
    // LT_TAIL: dec1 + its GroupNorm + output.0 + ReLU + output.2 + the sampler update as ONE row-per-CTA phase on CUDA cores
    // (weights transposed [in][out]); A0 / A1 / W = dec1's inputs and composed weights, bias / gamma / beta its GroupNorm as in LT_NORM
    const float* W2; const float* b2;    // output.0  [128][128]^T
    const float* W3; const float* b3;    // output.2  [128][256]^T
    // LT_HEAD (the first two layers as ONE row-per-CTA phase on CUDA cores): W2 = enc1's z columns [256][128]^T with bias (one row
    // per time row) / gamma / beta / out as in LT_NORM; W3 / b3 = enc2 [128][256]^T with gamma2 / beta2 / out2
    const float* gamma2; const float* beta2; float* out2;
};
constexpr int kLtBarrierWords = 64 + 32 * 16;     // grid barrier: flag line, top counter line, up to 16 group counter lines
struct LtProgram {
    int n_pre, n_loop;       // ops [0, n_pre) run once; ops [n_pre, n_pre + n_loop) run every reverse step
    LtOp ops[40];
};

// Two fp32 values -> one packed pair of 16-bit floats (bf16 or fp16; fp16 saturates instead of overflowing to inf).
__device__ __forceinline__ uint32_t pack16x2(float a, float b, int f16) {
    if (f16) {
        a = fminf(fmaxf(a, -65504.f), 65504.f); b = fminf(fmaxf(b, -65504.f), 65504.f);
        __half2 h = __floats2half2_rn(a, b);
        return *reinterpret_cast<uint32_t*>(&h);
    }
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack16x2(uint32_t v, int f16) {
    if (f16) return __half22float2(*reinterpret_cast<__half2*>(&v));
    return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&v));
}
__device__ __forceinline__ uint16_t pack16(float a, int f16) { return static_cast<uint16_t>(pack16x2(a, 0.f, f16) & 0xffffu); }
__device__ __forceinline__ float unpack16(uint16_t v, int f16) { return unpack16x2(v, f16).x; }

// "c8" byte planes (fp8-corrected split layers, gemm_tc.cu NP == 4): per 32 channels, 32 residual bytes then 32 copy bytes.  e5m2 has fp16's exponent range and the residuals are 2^-11
// of their values, so both products are balanced with powers of two that cancel:  (lo * 2^6)(W_hi * 2^-6) + (hi * 2^-8)(W_lo * 2^8)
constexpr float kC8ScaleLo = 64.f;            // activation residual plane: e5m2(lo * 2^6);   weights' hi copy: e5m2(W_hi * 2^-6)
constexpr float kC8ScaleHi = 1.f / 256.f;     // activation hi copy:        e5m2(hi * 2^-8);  weights' residual: e5m2(W_lo * 2^8)

// four fp32 values -> four e5m2 bytes (round to nearest, saturating), element 0 in the low byte
__device__ __forceinline__ uint32_t pack_e5m2x4(float a, float b, float c, float d) {
    const uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(a, b), __NV_SATFINITE, __NV_E5M2);
    const uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(c, d), __NV_SATFINITE, __NV_E5M2);
    return lo | (hi << 16);
}

enum EpiKind { EPI_STORE = 0, EPI_MAXPOOL = 1, EPI_FINAL = 2 };

// Implicit-GEMM 3-D convolution on the tcgen05 GEMM (VAE3DLarge.decode, networks.py:2247-2264): the A-role operand is a
// channels-last activation grid [batch][D][H][W][C]; a 128-row tile is 128 consecutive voxels (a box of whole W rows), and
// k-block kb reads channel block kb % cin_kb of the box shifted by tap kb / cin_kb.  Out-of-range voxels are zero-filled by
// TMA = the convolution's zero padding.  ntaps == 0: plain 2-D GEMM.
struct ConvGeom {
    int ntaps;                        // taps read through A source 0 (27 for k=3; 8 for one output-parity class of the k=4 s=2
                                      // transposed conv); A source 1, if any, is read at offset (0,0,0) (residual shortcut)
    int cin_kb;                       // 64-channel k-blocks per tap
    int W, H, D;                      // input grid
    int batch_plane;                  // lo plane = batch index + batch_plane (5-D tensors keep planes on the batch axis)
    int store5d;                      // 1: the output tile is scattered through a strided 5-D map (transposed conv, one parity class)
    int stride;                       // 1, or 2 (Conv3d k=4 s=2 p=1): the rows are OUTPUT voxels, tap t reads input voxel
                                      // stride * o + (dd, dh, dw)[t] through a map that steps 2 input voxels per box element
    signed char dw[64], dh[64], dd[64];
};

// Tap-grouped implicit-GEMM 3-D convolution (conv3d_tc.cu): 64 output channels, a 128-voxel tile = bh whole w-lines (bw = W
// voxels each) of one d-slice; one A load per (group, 64-channel block) brings bh + nt - 1 lines and serves the group's nt taps,
// which differ only in their h offset (tap t = box rows [t * bw, t * bw + 128)).
struct Conv3dParams {
    int num_m_blocks;                 // 128-voxel tiles
    int W, H, D;                      // input grid (W == bw)
    int bw, bh;                       // tile: bh lines of bw voxels, bw * bh == 128
    int ngroups;                      // (dw, dd) tap groups read through A source 0
    int nt;                           // h-taps per group (1..3)
    int cin_kb;                       // 64-channel blocks per tap
    int res, res_t;                   // res: append res_kb shortcut stages from A source 1 (identity or 1x1 weights), read at
                                      // offset 0 = line res_t of a box loaded at h0 - res_t
    int res_kb;                       // 64-channel blocks of the shortcut source
    int stride;                       // 1, or 2: lines are output lines and the A map steps 2 input voxels per element (h0, d0
                                      // of a tile are multiplied by 2 before the group offset is added)
    int a_box_bytes;                  // bytes one A load deposits: (bh + nt - 1) * bw * 128
    int batch_plane;                  // lo plane of a grid = batch index + batch_plane
    int b_plane_rows;                 // lo plane of the weights = row + b_plane_rows
    int out_plane_rows;               // 2-D store: lo plane = row + out_plane_rows
    int store5d;                      // 1: scatter through a strided 5-D view of the output grid (transposed conv parity class)
    int relu;
    const float* bias;                // [64]
    signed char gdw[32], gdh0[32], gdd[32];   // per group: w offset, h offset of tap 0, d offset
};

// tcgen05 GEMM: D[128 x BN] = Arole[128 x K] * Brole[BN x K]^T, both operands K-major bf16.
struct TcGemmParams {
    ConvGeom conv;
    int num_m_blocks;   // A-role blocks of 128 rows
    int num_n_blocks;   // B-role blocks of BN rows
    int kb0, kb1;       // 64-wide k-blocks taken from A source 0 / source 1
    int a_plane_rows, b_plane_rows, out_plane_rows;   // bf16x3: row offset of the lo plane inside each 2-D tensor (0 otherwise)
    // EPI_STORE / EPI_FINAL: lanes = point rows, columns = output channels
    __nv_bfloat16* out;
    int ldo;
    const float* bias;              // bias + sample * bias_sample_stride + column
    long long bias_sample_stride;   // 0 = shared by all samples
    int rows_per_sample;            // Npad
    int relu;
    // EPI_MAXPOOL: lanes = output channels (weights are the A role), columns = points
    float* gmax;        // [B][ld_g], pre-zeroed; values are post-ReLU (>= 0)
    int ld_g;
    int n_valid;        // N
    int num_samples;    // B (guards point blocks past the last cloud)
    int epi_warps;      // EPI_STORE: 8 = two epilogue warps per TMEM lane quarter on 32-column sub-groups (tmOut box 32 x 32, SWIZZLE_64B;
                        // plain 2-D stores only); 0 / 4 = one warp per quarter on 64-column groups (tmOut box 64 x 32, SWIZZLE_128B)
    int tile_order;     // STORE / FINAL tile schedule: 0 = a cluster keeps its row block across the weight tiles, 1 = n fastest (gemm_tc.cu)
    int f16;            // 16-bit operand/activation format: 0 = bf16, 1 = fp16 (values saturate at +-65504); selects the kernel instantiation
    const CallArgs* call;   // EPI_FINAL: per-call arguments live in device memory (graph-invariant)
};

// Fused chain of narrow per-point layers (chain_tc.cu): layer l reads its input from the on-chip activation buffer (or, for a
// chain's first layer, streams it from one or two HBM tensors) and writes its output to that buffer and / or to HBM.
struct ChainLayer {
    int kb;                 // 64-wide k-blocks of the input
    int kb_ext0, kb_ext1;   // streamed input: k-blocks taken from external tensor 0, then 1 (both 0: the input is the activation buffer)
    int n;                  // output channels: 64, 128 or 256 (256: two 128-column chunks, HBM output only)
    int np;                 // MMA passes per k-step: 1, or 3 (hi*hi + hi*lo + lo*hi on two-plane operands)
    int to_act;             // the output is the next layer's input (at most 128 channels)
    int to_hbm;             // index of the 32 x 32 store map the output is also / only written through, or -1
    int final;              // output.0: the epilogue is output.3 + the sampler update (EPI_FINAL of gemm_tc.cu)
    const float* bias;
    long long bias_sample_stride;
};
struct ChainParams {
    int nlayers;
    ChainLayer L[8];
    int num_m_blocks;       // 128-row tiles
    int rows_per_sample;    // Npad
    int a_plane_rows;       // row offset of the second plane in every activation tensor (0 in the one-plane modes)
    int first_from_x;       // chain A: enc1.conv1's xyz columns are evaluated in the kernel from x_t
    const float* Wx;        // [64][3]
    const float* bias1;     // forward hook: per-sample hoisted time bias [B][64] (sampler calls read CallArgs::bias1_steps)
    const CallArgs* call;
};
struct ChainMaps {
    CUtensorMap w[8];       // per layer: weights [planes * cout][K], box 64 x min(128, cout), SWIZZLE_128B
    CUtensorMap ext[2];     // streamed inputs [planes * M][C], box 64 x 128
    CUtensorMap out[4];     // HBM outputs [planes * M][C], box 32 x 32, SWIZZLE_64B
};

// fp32 CUDA-core GEMM (precision 'fp32' and the small per-sample GEMMs):
// C[M x Nout] = [A0 | A1][M x (K0+K1)] * W[Nout x (K0+K1)]^T
struct SimtGemmParams {
    const float* A0; int lda0; int K0;
    const float* A1; int lda1; int K1;
    const float* W;  int ldw;
    int M, Nout;
    float* out; int ldo;
    const float* bias; long long bias_sample_stride; int rows_per_sample; int relu;
    float* gmax; int ld_g; int n_valid;   // EPI_MAXPOOL (lanes = points here)
    float* partial; int splits;           // split-K workspace [splits][M][Nout] (EPI_STORE only; nullptr/1 = off)
};

}  // namespace pcd
