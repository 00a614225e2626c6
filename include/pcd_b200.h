/* pcd_b200.h -- C ABI of the B200-native point-cloud diffusion sampling hot path.
 *
 * The reference (dhillon24/3d-shape-generation) is pure Python; its "operator API" for this
 * path is the Python class surface cited below.  Each entry point names the reference
 * interface it stands behind (file:line in the reference tree).  Plain pointers and sizes
 * only; no torch types.  All device pointers are BORROWED (never freed here); every call
 * takes the CUDA stream to enqueue on and performs no hidden device-wide synchronisation
 * unless stated.  A handle is not thread-safe; distinct handles are independent; one
 * handle per GPU.  Functions return 0 on success, non-zero on error; the message is
 * available from pcd_last_error() (thread-local).  The library never calls exit()/abort().
 */
#ifndef PCD_B200_H
#define PCD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCD_ABI_VERSION 1

/* precision of the per-point layers */
#define PCD_PRECISION_BF16 0 /* tcgen05 bf16 x bf16 -> fp32 accumulate (headline path)            */
#define PCD_PRECISION_FP32 1 /* CUDA-core fp32 (parity at 1e-5; also the debugging ground truth)   */
#define PCD_PRECISION_BF16X3 2 /* tcgen05, operands split into hi+lo bf16 planes, 3 MMAs per k-step:
                                 near-fp32 products at 1/3 tensor throughput (meets the 1e-3 bound)  */
#define PCD_PRECISION_F16 3 /* tcgen05 fp16 x fp16 -> fp32 accumulate: the speed of BF16 with 3 more mantissa
                               bits (eps error ~2.6e-3 instead of ~2.4e-2); activations saturate at 65504 */
#define PCD_PRECISION_F16MIX 4 /* fp16 hi+lo planes, 3 MMAs per k-step everywhere except the two layers that
                                  hold 67 % of the FLOPs (global_feat.0/.3), which run one fp16 pass:
                                  meets the 1e-3 bound at ~1.7x the cost of one pass instead of 3x        */

/* dtype codes for pcd_named_tensor */
#define PCD_DTYPE_F32 0
#define PCD_DTYPE_I64 1

/* One entry of the reference's state_dict (PointCloudDiffusion.state_dict(), keys such as
 * "model.enc1.conv1.weight" -- networks.py:737-777, PointNetLayer networks.py:29-34). Host memory. */
typedef struct pcd_named_tensor {
    const char* name;
    const void* data;
    int32_t dtype;
    int32_t ndim;
    int64_t shape[4];
} pcd_named_tensor;

typedef struct pcd_denoiser pcd_denoiser; /* opaque: folded/packed weights + workspaces on one GPU */

int pcd_abi_version(void);
const char* pcd_last_error(void);

/* Replaces: PointCloudDiffusion.__init__ + load_state_dict + .to(device)
 * (diffusion.py:15-38, test_point_ddpm.py:161-163).  Consumes the UNMODIFIED reference
 * state_dict; BatchNorm(eval) folding (networks.py:46-48), hoisting of the time-embedding
 * columns of enc1.conv1 (networks.py:796-797) and of the global-feature columns of dec4.conv1
 * (networks.py:808,811), and pre-composition of refineK into decK.conv1 (networks.py:811-814)
 * happen inside. */
int pcd_denoiser_create(const pcd_named_tensor* tensors, int32_t n_tensors, int32_t precision, int32_t device,
                        pcd_denoiser** out);
int pcd_denoiser_destroy(pcd_denoiser* h);

/* Replaces: UNetPointNetLarge.forward(x[B,N,3], t[B]) -> eps[B,N,3]  (networks.py:779-818;
 * call site diffusion.py:245,282,328).  Device pointers, fp32. */
int pcd_denoiser_forward(pcd_denoiser* h, const float* x, const float* t, float* eps, int32_t B, int32_t N,
                         void* stream);

/* Replaces the reverse loops PointCloudDiffusion.sample / sample2 / sample3
 * (diffusion.py:261-289, 225-259, 291-337).  The loop is table driven: `sched` (HOST pointer,
 * S rows of 8 floats: noise_rate n, signal_rate s, s_next, n_next, cz, t, 0, 0) holds the
 * reference's own fp32 schedule values for each step, so one entry point serves DDIM, DDPM
 * and DDIM-from-t.  Per step and per point, with eps = denoiser(x, t):
 *      x0 = (x - n*eps)/s ;  x <- s_next*x0 + n_next*eps + cz*z
 * The last row carries s_next=1, n_next=0, cz=0 so the call leaves the final x0 in `x`
 * (diffusion.py:257,289,336).  z (only where cz != 0, i.e. DDPM): taken from `noise`
 * (device, [S-1][B][N][3], the reference's randn_like draws in order, diffusion.py:254) when
 * non-NULL, otherwise Philox4x32-10 keyed by (seed, sample_offset + b, step, point).
 * `x` is updated in place ([B,N,3] fp32 device).  The whole step is one CUDA graph replayed S times. */
int pcd_sample(pcd_denoiser* h, const float* sched, int32_t S, float* x, const float* noise, uint64_t seed,
               uint64_t sample_offset, int32_t B, int32_t N, void* stream);

/* pcd_sample with ONE SCHEDULE ROW PER SAMPLE: `sched` holds S * rows_per_step rows ([S][rows_per_step][8]),
 * rows_per_step = 1 (identical to pcd_sample) or B.  Needed for noise_schedule='linear': the reference evaluates
 * `torch.cumprod(1 - betas, dim=0)` over the BATCH axis (diffusion.py:202), so with a vector t every sample of the
 * batch gets its own (noise_rate, signal_rate) -- reproduced here row for row instead of being "fixed". */
int pcd_sample_rows(pcd_denoiser* h, const float* sched, int32_t S, int32_t rows_per_step, float* x, const float* noise,
                    uint64_t seed, uint64_t sample_offset, int32_t B, int32_t N, void* stream);

/* Same as pcd_sample with HOST buffers: copies x_T in (H2D), runs the loop, copies the result out
 * (D2H) and synchronises the stream.  This is the end-to-end call bench.py times as `e2e`. */
int pcd_sample_host(pcd_denoiser* h, const float* sched, int32_t S, const float* x_T_host, float* x_out_host,
                    const float* noise_host, uint64_t seed, uint64_t sample_offset, int32_t B, int32_t N,
                    void* stream);

/* pcd_sample_host with one schedule row per sample (`sched` = [S][rows_per_step][8], rows_per_step = 1 or B): the host-buffer
 * entry for noise_schedule='linear' (diffusion.py:189-205, batch-axis cumprod). */
int pcd_sample_host_rows(pcd_denoiser* h, const float* sched, int32_t S, int32_t rows_per_step, const float* x_T_host,
                         float* x_out_host, const float* noise_host, uint64_t seed, uint64_t sample_offset, int32_t B,
                         int32_t N, void* stream);

/* The noise pcd_sample draws at `step` when noise == NULL (so tests can hand the very same
 * tensor to the oracle).  out: device [B][N][3]. */
int pcd_philox_normal(uint64_t seed, uint64_t sample_offset, int32_t step, float* out, int32_t B, int32_t N,
                      void* stream);

/* Debug/parity tap: copy an internal activation of the last forward/step to HOST fp32.
 * names: "temb"[B,256] "x1"[M,128] "x2"[M,256] "x3"[M,512] "x4"[M,1024] "g"[B,4096]
 * "d4"[M,512] "d1"[M,64]  (M = B*Npad padded rows, point-major).  Synchronises. */
int pcd_denoiser_tap(pcd_denoiser* h, const char* name, float* out_host, int64_t count);

/* Measurement hook: run ONE forward eagerly with a CUDA event between consecutive launches and
 * return, per launch, the device time (ms), the algorithmic FLOPs (2*M*K*Cout of the layer; 0 for
 * non-GEMM helpers) and a name ('global_feat.3+maxpool', ...).  Synchronises the stream.
 * ms_out/flops_out: [cap]; names_out: cap * name_stride chars (may be NULL). */
int pcd_denoiser_profile(pcd_denoiser* h, const float* x, const float* t, float* eps, int32_t B, int32_t N,
                         float* ms_out, double* flops_out, char* names_out, int32_t name_stride, int32_t cap,
                         int32_t* n_out, void* stream);

/* One fused per-point layer  out = relu?( [A0|A1] * W^T + bias )  on device bf16 buffers --
 * the PointNetLayer conv->bn->relu unit (networks.py:46) after BN folding; exposed so the
 * tcgen05 kernel can be tested in isolation.  A0 [M,K0], A1 [M,K1] (may be NULL, K1=0),
 * W [Cout, K0+K1] row-major bf16 (uint16 storage); bias fp32 [Cout]; out bf16 [M,Cout].
 * M % 128 == 0, K0 % 64 == 0, K1 % 64 == 0, Cout % 64 == 0. */
int pcd_linear_bf16(const void* A0, int32_t K0, const void* A1, int32_t K1, const void* W, const float* bias,
                    void* out, int32_t M, int32_t Cout, int32_t relu, void* stream);

/* Replaces: metrics.chamfer_distance per pair (metrics.py:23-47) incl. normalize_to_cube
 * (metrics.py:7-21).  x [B,N,3], y [B,M,3] device fp32 -> cd[B] (device) =
 * scaling * (mean_i min_j |x_i-y_j| + mean_j min_i |x_i-y_j|) on cube-normalised clouds.
 * idx_xy [B,N] / idx_yx [B,M] (device int32, may be NULL) receive the nearest-neighbour indices.  Like the reference, a pair
 * with a cloud whose normalisation is not finite (a NaN or +-inf coordinate, a centre that overflows, all points equal or one
 * point) gets NaN; the other pairs are unaffected. */
int pcd_chamfer_pairs(const float* x, const float* y, int32_t B, int32_t N, int32_t M, float scaling, float* cd,
                      int32_t* idx_xy, int32_t* idx_yx, void* stream);

/* All-pairs Chamfer matrix out[i*nR + j] = chamfer_distance(G[i], R[j]) (device fp32) for the
 * set metrics MMD-CD / COV / 1-NNA built on the reference's per-pair semantics.  G == R with nG == nR (a set against itself)
 * evaluates the upper triangle only and mirrors it: the values are those of the full sweep (CD is bit-symmetric here).
 * An entry with a non-finite normalised cloud is NaN, as in pcd_chamfer_pairs. */
int pcd_chamfer_matrix(const float* G, int32_t nG, const float* R, int32_t nR, int32_t N, float scaling,
                       float* out, void* stream);

/* Replaces: metrics.earth_mover_distance_gpu (metrics.py:94-158), the log-domain Sinkhorn approximation that
 * compute_metrics(use_approximate_gpu_emd=True) calls (metrics.py:176).  x [B,N,3], y [B,M,3] device fp32 ->
 * emd[B] (device) = scaling * sum_ij P_ij C_ij per pair, with the reference's exact recipe: cube-normalised
 * clouds, C = cdist / (ONE maximum over the whole batch), duals from 0, alpha then beta per iteration, stop
 * when both max-abs dual changes over the batch are < thresh or after max_iter iterations.  The cost matrix is
 * never materialised.  Like the reference, the convergence test is a host round trip: this entry synchronises
 * `stream` once per Sinkhorn iteration.  iters_out (host, may be NULL) receives the iteration count.  As in the reference, one
 * pair with a non-finite normalised cloud (see pcd_chamfer_pairs) makes the batch maximum and the convergence test NaN: every
 * pair of the call is NaN and max_iter iterations run. */
int pcd_sinkhorn_emd(const float* x, const float* y, int32_t B, int32_t N, int32_t M, float epsilon, float thresh,
                     int32_t max_iter, float scaling, float* emd, int32_t* iters_out, void* stream);

/* Replaces: metrics.earth_mover_distance_cpu (metrics.py:49-92, SciPy linear_sum_assignment) per pair.  x [B,N,3], y [B,M,3]
 * device fp32 -> emd[B] (device) = scaling * (sum of |x_i - y_j| over an optimal matching of the cube-normalised clouds) / 3,
 * the reference's recipe including its divisor of 3 (x_pc.shape[1]).  N != M is allowed: min(N, M) pairs are matched, each
 * point at most once.  The matching is optimal for the distances quantised to 2^-22, so the value is within n / 2^22 (absolute,
 * n = max(N, M)) of the fp64 optimum; it is deterministic and does not depend on the other pairs of the batch.
 * assign_xy [B,N] (device int32, may be NULL) receives the matched y index of every x, or -1 for an unmatched x.  A pair with a
 * non-finite normalised coordinate (see pcd_chamfer_pairs) gets NaN and -1 everywhere; the other pairs are unaffected.
 * N, M <= 4096.
 * The entry synchronises `stream` once, to read back a device flag set when an auction phase exceeds its round cap (then it
 * returns non-zero; such pairs are NaN). */
int pcd_emd_exact(const float* x, const float* y, int32_t B, int32_t N, int32_t M, float scaling, float* emd,
                  int32_t* assign_xy, void* stream);

/* ---- latent-diffusion path (BASELINE config 4) -------------------------------------------------
 * Replaces: LatentDiffusion.__init__/load_state_dict (diffusion.py:361-390) with a
 * SimpleLatentUNetPointNet denoiser (networks.py:962-1106; latent_dim = time_dim = 256, dim = 512)
 * and, when the state_dict holds `vae.decoder.*` / `vae.output_layer.*`, SimplePointNetVAE's decoder
 * (networks.py:1144-1154).  Consumes LatentDiffusion.state_dict() as is (`model.*`, `vae.*`). */
typedef struct pcd_latent pcd_latent;
int pcd_latent_create(const pcd_named_tensor* tensors, int32_t n_tensors, int32_t num_points, int32_t device,
                      pcd_latent** out);
int pcd_latent_destroy(pcd_latent* h);
/* SimpleLatentUNetPointNet.forward(z[B,256], t[B]) -> eps[B,256]  (networks.py:1051-1086) */
int pcd_latent_forward(pcd_latent* h, const float* z, const float* t, float* eps, int32_t B, void* stream);
/* LatentDiffusion.sample / sample2 / sample3 loops on z (diffusion.py:575-707), table driven exactly like
 * pcd_sample; z [B,256] is updated in place and holds z_0 on return; noise: [S-1][B][256] or NULL (Philox). */
int pcd_latent_sample(pcd_latent* h, const float* sched, int32_t S, float* z, const float* noise, uint64_t seed,
                      uint64_t sample_offset, int32_t B, void* stream);
/* Same with rows_per_step schedule rows per step: 1, or B = one row per sample (noise_schedule='linear': the reference's
 * linear_diffusion_schedule cumprods over the BATCH axis, diffusion.py:553-569, so every sample gets its own rates). */
int pcd_latent_sample_rows(pcd_latent* h, const float* sched, int32_t S, int32_t rows_per_step, float* z, const float* noise,
                           uint64_t seed, uint64_t sample_offset, int32_t B, void* stream);
/* SimplePointNetVAE.decode(z[B,256]) -> [B, num_points, 3]  (networks.py:1219-1231) */
int pcd_vae_decode(pcd_latent* h, const float* z, float* out, int32_t B, void* stream);
int pcd_latent_philox_normal(uint64_t seed, uint64_t sample_offset, int32_t step, float* out, int32_t B, int32_t D,
                             void* stream);

/* ---- voxel-VAE decoder (SURVEY 8(f) rank 4; the reference's DEFAULT latent configuration, is_voxel_based=True) -------
 * Replaces: VAE3DLarge.decode (networks.py:2327-2339: decoder_input Linear + the nn.Sequential of 3-D transposed
 * convolutions, ResidualBlock3D blocks (networks.py:471-505) and the final Conv3d + Sigmoid, networks.py:2245-2264).
 * Consumes the decoder half of VAE3DLarge.state_dict() under the `vae.` prefix LatentDiffusion.state_dict() gives it
 * (`vae.decoder_input.*`, `vae.decoder.<i>.*`; BatchNorm3d running statistics are folded, eval mode).
 * precision: PCD_PRECISION_BF16 / _F16 (one tensor-core pass) or _BF16X3 / _F16MIX (hi + lo planes, 3 passes, near fp32). */
typedef struct pcd_vae3d pcd_vae3d;
int pcd_vae3d_create(const pcd_named_tensor* tensors, int32_t n_tensors, int32_t precision, int32_t device, pcd_vae3d** out);
int pcd_vae3d_destroy(pcd_vae3d* h);
/* z [B, latent] device fp32 -> voxel probabilities vox [B, 1, 32, 32, 32] device fp32 */
int pcd_vae3d_decode(pcd_vae3d* h, const float* z, float* vox, int32_t B, void* stream);
/* Debug/parity tap: run the decoder up to and including nn.Sequential index seq_index (0, 2, 3, 5, 6, 8, 9 or 11; -1 =
 * decoder_input) and copy that activation to HOST fp32, channels-last [B][D][H][W][C].  Synchronises. */
int pcd_vae3d_tap(pcd_vae3d* h, const float* z, int32_t B, int32_t seq_index, float* out_host, int64_t count, void* stream);
/* Measurement hook: one eager decode with a CUDA event between launches (same contract as pcd_denoiser_profile). */
int pcd_vae3d_profile(pcd_vae3d* h, const float* z, float* vox, int32_t B, float* ms_out, double* flops_out, char* names_out,
                      int32_t name_stride, int32_t cap, int32_t* n_out, void* stream);
/* ---- voxel-VAE encoder ------------------------------------------------------------------------------------------------
 * Replaces: VAE3DLarge.encode (networks.py, just above decode at :2327): the encoder nn.Sequential of networks.py:2210-2241
 * (Conv3d 1 -> 32 + ReLU, then ResidualBlock3D(c -> 2c) with a 1x1 `downsample` shortcut and Conv3d(k=4, s=2, p=1) + ReLU per
 * stage, 32^3 -> 4^3, then Conv3d(512 -> 512, k=4, p=0) + ReLU + Flatten) and fc_mu / fc_logvar (networks.py:2243-2244).
 * Consumes `vae.encoder.*`, `vae.fc_mu.*` and `vae.fc_logvar.*` (BatchNorm3d folded, eval mode); a missing key is named in
 * the error.  Its own handle, so decoder-only tables keep working with pcd_vae3d_*.  Precisions as for the decoder. */
typedef struct pcd_vae3d_encoder pcd_vae3d_encoder;
int pcd_vae3d_encoder_create(const pcd_named_tensor* tensors, int32_t n_tensors, int32_t precision, int32_t device,
                             pcd_vae3d_encoder** out);
int pcd_vae3d_encoder_destroy(pcd_vae3d_encoder* h);
/* vox [B, 1, 32, 32, 32] device fp32 -> mu, logvar [B, latent] device fp32 */
int pcd_vae3d_encode(pcd_vae3d_encoder* h, const float* vox, float* mu, float* logvar, int32_t B, void* stream);
/* Debug/parity tap: run the encoder up to and including nn.Sequential index seq_index (0, 2, 3, 5, 6, 8, 9, 11 or 12 = after
 * the ReLU, [B][512]) and copy that activation to HOST fp32, channels-last [B][D][H][W][C].  Synchronises. */
int pcd_vae3d_encoder_tap(pcd_vae3d_encoder* h, const float* vox, int32_t B, int32_t seq_index, float* out_host, int64_t count,
                          void* stream);
/* Measurement hook: one eager encode with a CUDA event between launches (same contract as pcd_vae3d_profile). */
int pcd_vae3d_encoder_profile(pcd_vae3d_encoder* h, const float* vox, float* mu, float* logvar, int32_t B, float* ms_out,
                              double* flops_out, char* names_out, int32_t name_stride, int32_t cap, int32_t* n_out, void* stream);
/* ---- point-VAE encoder -------------------------------------------------------------------------------------------------
 * Replaces: SimplePointNetVAE.encode (networks.py:1110-1156; encode between __init__ and decode at :1219): four PointNetLayers
 * (3 -> 64 -> 128 -> 256 -> 512, each three times Conv1d(k=1) + BatchNorm1d + ReLU), AdaptiveMaxPool1d(1) + Flatten,
 * Linear(512, 256) + ReLU, then fc_mu / fc_logvar.  Consumes `vae.encoder.*`, `vae.fc_mu.*` and `vae.fc_logvar.*` (BatchNorm1d
 * folded, eval mode); a missing key is named in the error.  Only hidden_dim = 512 and latent_dim = 256 (the reference defaults)
 * are supported.  Its own handle, so decoder-only tables keep working with pcd_latent_*.  Precisions as for pcd_vae3d. */
typedef struct pcd_point_encoder pcd_point_encoder;
int pcd_point_encoder_create(const pcd_named_tensor* tensors, int32_t n_tensors, int32_t precision, int32_t device,
                             pcd_point_encoder** out);
int pcd_point_encoder_destroy(pcd_point_encoder* h);
/* x [B, N, 3] device fp32 (any N >= 1) -> mu, logvar [B, 256] device fp32.  A cloud with a NaN or +-inf coordinate gets NaN in
 * every mu / logvar entry; the other clouds of the batch do not change. */
int pcd_point_encode(pcd_point_encoder* h, const float* x, float* mu, float* logvar, int32_t B, int32_t N, void* stream);
/* Debug/parity tap: run the encoder up to the tapped tensor and copy it to HOST fp32.  index 0..11 = the activation after
 * encoder.<index / 3>.conv<index % 3 + 1> (+ BatchNorm + ReLU), valid points only, [B][N][C]; 12 = the pooled [B][512];
 * 13 = encoder.7's output [B][256].  Synchronises. */
int pcd_point_encoder_tap(pcd_point_encoder* h, const float* x, int32_t B, int32_t N, int32_t index, float* out_host, int64_t count,
                          void* stream);
/* Measurement hook: one eager encode with a CUDA event between launches (same contract as pcd_vae3d_encoder_profile). */
int pcd_point_encoder_profile(pcd_point_encoder* h, const float* x, float* mu, float* logvar, int32_t B, int32_t N, float* ms_out,
                              double* flops_out, char* names_out, int32_t name_stride, int32_t cap, int32_t* n_out, void* stream);
/* Replaces: utils.voxel_tensor_to_point_clouds (utils.py:511-539), called by LatentDiffusion.sample* on the decoded grid
 * (diffusion.py:611-612, 650-651, 704-705).  Two calls because the output is ragged: pcd_voxel_count gives, per sample, the
 * number of voxels with value > threshold; the caller turns the counts into exclusive offsets (int64) and pcd_voxel_points
 * writes, per sample and in torch.where order (z, y, x ascending), the points (x, y, z) = 2 * index / (dim - 1) - 1 into
 * pts [total, 3] (device fp32).  vox: [B, 1, D, H, W] device fp32. */
int pcd_voxel_count(const float* vox, int32_t B, int32_t D, int32_t H, int32_t W, float threshold, int32_t* counts, void* stream);
int pcd_voxel_points(const float* vox, int32_t B, int32_t D, int32_t H, int32_t W, float threshold, const int64_t* offsets,
                     float* pts, void* stream);

/* number of kernel launches issued by this library since load (bench.py's gpu_launches claim) */
int64_t pcd_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* PCD_B200_H */
