// Launcher prototypes (defined in gemm_tc.cu, gemm_simt.cu, chamfer.cu, emd.cu, emd_exact.cu).
#pragma once
#include <cstdlib>
#include <utility>
#include <cuda.h>
#include <cuda_runtime.h>
#include "pcd_types.h"

namespace pcd {

// Programmatic dependent launch (see pcd_ptx.cuh)
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
cudaError_t launch_zero_f32(float* p, long long n, cudaStream_t stream);

cudaError_t launch_gemm_tc(int bn, int epi, int np, int out_planes, int cl, int two_sm, const CUtensorMap& a0, const CUtensorMap& a1,
                           const CUtensorMap& b, const CUtensorMap& out, const TcGemmParams& p, int num_sms, cudaStream_t stream);
cudaError_t configure_gemm_tc();
cudaError_t configure_chain_tc();
cudaError_t launch_chain_tc(int planes, int f16, const ChainMaps& maps, const ChainParams& p, int num_sms, cudaStream_t stream);
cudaError_t launch_conv3d_tc(int np, int cl, int f16, const CUtensorMap& a0, const CUtensorMap& a1, const CUtensorMap& b,
                             const CUtensorMap& out, const Conv3dParams& p, int num_sms, cudaStream_t stream);
cudaError_t configure_conv3d_tc();
cudaError_t launch_gemm_simt(int epi, const SimtGemmParams& p, cudaStream_t stream);
bool skinny_splitk_ok(const SimtGemmParams& p);
cudaError_t launch_skinny_splitk(const SimtGemmParams& p, cudaStream_t stream);
cudaError_t launch_splitk_reduce(const float* partial, int nsplit, const float* bias, float* out, int M, int Nout, int relu,
                                 cudaStream_t stream);
int simt_pick_splits(int M, int Nout, int K, int num_sms);
cudaError_t launch_time_bias(int rows, int T, int per_step, const CallArgs* ca, const float* freqs, const float* W1T, const float* b1,
                             const float* W2T, const float* b2, const float* WtT, const float* bt, float* temb_out,
                             float* bias1_out, cudaStream_t stream);
cudaError_t launch_enc1_first(int elt_bytes, int f16, const CallArgs* ca, const float* Wx, const float* bias1, long long bias_stride,
                              void* out, void* out_lo, int B, int N, int Npad, cudaStream_t stream);
cudaError_t launch_final_simt(const float* h, long long rows, const CallArgs* ca, cudaStream_t stream);
cudaError_t launch_advance_step(int* step, cudaStream_t stream);
cudaError_t launch_philox_fill(float* out, unsigned long long seed, unsigned long long sample_offset, int step, int B, int N,
                               cudaStream_t stream);
cudaError_t launch_f32_to_16(const float* in, void* out, long long n, int f16, cudaStream_t stream);
cudaError_t launch_16_to_f32(const void* in, const void* in_lo, float* out, long long n, int f16, cudaStream_t stream);
cudaError_t launch_f32_split_16(const float* in, void* hi, void* lo, long long n, int f16, cudaStream_t stream);
cudaError_t launch_f32_split_c8(const float* in, void* hi, void* c8, long long rows, int k, cudaStream_t stream);
cudaError_t launch_16c8_to_f32(const void* in, const void* c8, float* out, long long rows, int k, cudaStream_t stream);

cudaError_t launch_cloud_norm(const float* pts, int clouds, int N, float4* out, cudaStream_t stream);
cudaError_t launch_chamfer_dir(const float4* Q, const float4* T, int pairs, int Nq, int Nt, float* mind, int* idx,
                               cudaStream_t stream);
cudaError_t launch_chamfer_reduce(const float* dxy, const float* dyx, int pairs, int N, int M, float scaling, float* cd,
                                  cudaStream_t stream);
bool chamfer_fused_fits(int Na, int Nb);
cudaError_t launch_chamfer_fused(const float4* A, const float4* B, long long pairs, int nB, int Na, int Nb, float scaling,
                                 float* out, cudaStream_t stream);
cudaError_t launch_chamfer_matrix_self(const float4* G, int n, int N, float scaling, float* out, cudaStream_t stream);
cudaError_t launch_chamfer_matrix(const float4* G, int nG, const float4* R, int nR, int N, float scaling, float* out,
                                  cudaStream_t stream);

int emd_row_blocks(int n);
cudaError_t launch_emd_cmax(const float4* X, const float4* Y, int pairs, int N, int M, unsigned* cmax_bits, cudaStream_t s);
cudaError_t launch_sinkhorn_half(const float4* Q, const float4* T, const float* dual_t, float* dual_q, int pairs, int Nq, int Nt,
                                 const unsigned* cmax_bits, float lambda, float eps, float log_marg, unsigned* err_bits,
                                 cudaStream_t s);
cudaError_t launch_sinkhorn_cost(const float4* Q, const float4* T, const float* alpha, const float* beta, int pairs, int Nq, int Nt,
                                 const unsigned* cmax_bits, float lambda, float scaling, float* partial, float* emd, cudaStream_t s);

bool emd_exact_fits(int N, int M);
cudaError_t launch_emd_exact(const float4* X, const float4* Y, int pairs, int N, int M, float scaling, float* emd, int* assign_xy,
                             int* err, cudaStream_t s);

cudaError_t launch_fold_first(int kin, const float* in, int in_mod, const float* W, const float* bias, long long rows,
                              int rows_per_sample, void* out16, cudaStream_t s);
cudaError_t launch_fold_tail16(const void* h3, const float* Wbc, const float* bbc, const float* Wc2, const float* bc2, long long rows,
                               int rows_per_sample, int channel_major, float* out, cudaStream_t s);
cudaError_t launch_fold_transpose(const float* U, int B, int P, float* out, cudaStream_t s);

cudaError_t launch_groupnorm_relu(float* y, const float* partial, int nsplit, const float* bias, const float* gamma, const float* beta,
                                  int B, int C, cudaStream_t stream);
cudaError_t launch_latent_update(const float* eps, const LatentCall* ca, int B, int D, cudaStream_t stream);
cudaError_t launch_latent_philox_fill(float* out, unsigned long long seed, unsigned long long sample_offset, int step, int B,
                                      int D, cudaStream_t stream);
cudaError_t launch_latent_time(int B, const LatentCall* ca, const float* freqs, const float* W1T, const float* b1,
                               const float* W2T, const float* b2, float* temb_out, cudaStream_t stream);

cudaError_t launch_compose_refine(const float* Wd, int ldd, int col0, const float* Wr, int kr, const float* bd, const float* br,
                                  float* C, float* cbias, int cout, cudaStream_t s);
cudaError_t launch_tile_weights(const float* W, int ldw, int col0, int N, int K, int bn, float* out, cudaStream_t s);
cudaError_t latent_mk_grid(int num_sms, int* grid_out);
cudaError_t launch_latent_mk(const LtProgram* prog, const LatentCall* call, int S, int R, int forward, unsigned* bar, int grid,
                             cudaStream_t stream);

}  // namespace pcd
