// Implicit-GEMM 3-D convolution for the wide grids of VAE3DLarge.decode (networks.py:2247-2264: the 16^3 -> 32^3 transposed
// conv and every 32^3 layer, all with 64 output channels) on tcgen05, with the activation operand REUSED across the taps of
// one kernel column.
//
// The plain implicit GEMM (gemm_tc.cu, ConvGeom) fetches a fresh 128-voxel A tile from L2 for every tap: 27 x 16 KB per
// 128 x 64 output tile, and at N = 64 the layer is bound by L2 -> SM bandwidth, not by the tensor pipe (measured: 14 % of
// the MMA rate).  Here a 128-row tile is bh whole w-lines of one d-slice (bw = W voxels each), and ONE 5-D TMA load brings
// the box of bh + nt - 1 lines that the nt taps differing only in their h offset need: tap t's A operand is the same shared
// memory shifted by t * bw rows (a multiple of the 1024-byte swizzle atom, so the UMMA descriptor just starts later).  For
// k = 3 that is 24 KB per three taps instead of 48 KB; the weight tile of a CTA pair is fetched once and multicast.
//
//   D[128 x 64] (fp32, TMEM) += A_t[128 x 64] (rows t*bw .. t*bw+127 of the box) * W_t[64 x 64]^T     for every (group, t)
//
// Warp roles, barriers, the split-precision passes (NP = 3: hi/lo planes) and the store epilogue are those of gemm_tc.cu.
#include "pcd_ptx.cuh"
#include "pcd_types.h"

namespace pcd {

constexpr int kCvThreads = 192;
constexpr int kCvBN = 64;
constexpr int kCvMaxTaps = 3;                         // h-taps per stage
constexpr int kCvARows = 192;                         // largest box: (4 + 2) lines of 32 voxels
constexpr int kCvAPlane = kCvARows * 128;             // 24 KB
constexpr int kCvBTap = kCvBN * 128;                  // 8 KB per tap
constexpr int kCvBPlane = kCvMaxTaps * kCvBTap;       // 24 KB

__host__ __device__ constexpr int cv_planes(int np) { return np == 3 ? 2 : 1; }
__host__ __device__ constexpr int cv_stage_bytes(int np) { return cv_planes(np) * (kCvAPlane + kCvBPlane); }
__host__ __device__ constexpr int cv_stages(int np) { return np == 3 ? 2 : 4; }
__host__ __device__ constexpr int cv_smem_bytes(int np) { return cv_stages(np) * cv_stage_bytes(np) + 4 * 4096 + 4096 + 1024; }

template <int NP, int CL, int F16>
__global__ void __launch_bounds__(kCvThreads, 1)
conv3d_tc_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
                 const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmOut, const Conv3dParams p) {
    constexpr int STAGES = cv_stages(NP);
    constexpr int PL = cv_planes(NP);
    constexpr int A_STAGE = PL * kCvAPlane, B_STAGE = PL * kCvBPlane;
    constexpr uint32_t IDESC = make_idesc(128, kCvBN, F16);
    constexpr uint16_t CMASK = static_cast<uint16_t>((1u << CL) - 1);

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sA = smem;
    uint8_t* sB = smem + STAGES * A_STAGE;
    uint8_t* stage_out = sB + STAGES * B_STAGE;                       // 4 epilogue warps x 4 KB
    uint8_t* aux = stage_out + 4 * 4096;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(aux);             // [STAGES]
    uint64_t* empty_bar = full_bar + STAGES;                           // [STAGES]
    uint64_t* tfull_bar = empty_bar + STAGES;                          // [2]
    uint64_t* tempty_bar = tfull_bar + 2;                              // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    float* sbias = reinterpret_cast<float*>(aux + 256);                // [64]

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int crank = CL > 1 ? static_cast<int>(cluster_ctarank()) : 0;
    const int cid = blockIdx.x / CL, num_clusters = gridDim.x / CL;
    const int num_tiles = p.num_m_blocks / CL;
    const int main_stages = p.ngroups * p.cin_kb;
    const int num_stages = main_stages + (p.res ? p.res_kb : 0);

    if (warp == 0 && lane == 0) {
        prefetch_tensormap(&tmA0);
        prefetch_tensormap(&tmA1);
        prefetch_tensormap(&tmB);
        prefetch_tensormap(&tmOut);
        for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], CL); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 128); }
        fence_mbar_init();
    }
    if (warp == 1) { tmem_alloc(tmem_slot, 128); tmem_relinquish(); }
    if (threadIdx.x >= 64 && threadIdx.x < 64 + kCvBN) sbias[threadIdx.x - 64] = p.bias[threadIdx.x - 64];
    tc_fence_before();
    __syncthreads();
    if constexpr (CL > 1) cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int tile = cid; tile < num_tiles; tile += num_clusters) {
                const int m_blk = tile * CL + crank;
                const int line0 = m_blk * p.bh;                       // first w-line of the tile (global line index)
                const int h0 = line0 % p.H, d0 = (line0 / p.H) % p.D, b0 = line0 / (p.H * p.D);
                for (int s = 0; s < num_stages; ++s) {
                    const bool is_res = s >= main_stages;
                    const int g = is_res ? 0 : s / p.cin_kb;
                    const int cb = is_res ? s - main_stages : s - g * p.cin_kb;
                    const int ntap = is_res ? 1 : p.nt;
                    const int kblk0 = is_res ? main_stages * p.nt + cb : s * p.nt;
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    mbar_arrive_expect_tx(&full_bar[stage], PL * (p.a_box_bytes + ntap * kCvBTap));
#pragma unroll
                    for (int pl = 0; pl < PL; ++pl) {
                        uint8_t* da = sA + stage * A_STAGE + pl * kCvAPlane;
                        if (is_res) tma_load_5d(da, &tmA1, &full_bar[stage], cb * 64, 0, h0 - p.res_t, d0, b0 + pl * p.batch_plane);
                        else tma_load_5d(da, &tmA0, &full_bar[stage], cb * 64, p.gdw[g], p.stride * h0 + p.gdh0[g], p.stride * d0 + p.gdd[g],
                                         b0 + pl * p.batch_plane);
                        for (int t = 0; t < ntap; ++t) {
                            uint8_t* db = sB + stage * B_STAGE + pl * kCvBPlane + t * kCvBTap;
                            if constexpr (CL == 1) {
                                tma_load_2d(db, &tmB, &full_bar[stage], (kblk0 + t) * 64, pl * p.b_plane_rows);
                            } else {
                                constexpr int SL = kCvBN / CL;       // my slice of the shared weight tile, delivered to both CTAs
                                tma_load_2d_mcast(db + crank * SL * 128, &tmB, &full_bar[stage], (kblk0 + t) * 64,
                                                  crank * SL + pl * p.b_plane_rows, CMASK);
                            }
                        }
                    }
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int tile = cid; tile < num_tiles; tile += num_clusters) {
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * kCvBN;
                for (int s = 0; s < num_stages; ++s) {
                    const bool is_res = s >= main_stages;
                    const int ntap = is_res ? 1 : p.nt;
                    const int t_first = is_res ? p.res_t : 0;
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    for (int t = 0; t < ntap; ++t) {
                        // tap t reads the box from line t on: (t_first + t) * bw rows = a multiple of 1024 bytes
                        const uint64_t da = make_sw128_kmajor_desc(smem_u32(sA + stage * A_STAGE + (t_first + t) * p.bw * 128));
                        const uint64_t db = make_sw128_kmajor_desc(smem_u32(sB + stage * B_STAGE + t * kCvBTap));
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            constexpr uint64_t A_LO = kCvAPlane >> 4, B_LO = kCvBPlane >> 4;
                            tc_mma_bf16(d_tmem, da + 2 * k, db + 2 * k, IDESC, (s | t | k) != 0 ? 1u : 0u);
                            if constexpr (NP == 3) {
                                tc_mma_bf16(d_tmem, da + 2 * k, db + B_LO + 2 * k, IDESC, 1u);          // hi * lo
                                tc_mma_bf16(d_tmem, da + A_LO + 2 * k, db + 2 * k, IDESC, 1u);          // lo * hi
                            }
                        }
                    }
                    if constexpr (CL == 1) tc_commit(&empty_bar[stage]);
                    else tc_commit_mcast(&empty_bar[stage], CMASK);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                tc_commit(&tfull_bar[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ===================== epilogue (warps 2..5) =====================
        const int q = warp & 3;
        int acc = 0; uint32_t acc_phase = 0;
        uint8_t* stg = stage_out + (warp - 2) * 4096;
        for (int tile = cid; tile < num_tiles; tile += num_clusters) {
            const int m_blk = tile * CL + crank;
            const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * kCvBN;
            mbar_wait(&tfull_bar[acc], acc_phase);
            tc_fence_after();
            uint32_t v0[32], v1[32];
            tmem_ld_32x32(t_addr, v0);
            tmem_ld_32x32(t_addr + 32, v1);
            tc_wait_ld();
            // the accumulator is in registers: hand it back before the store tail
            tc_fence_before();
            mbar_arrive(&tempty_bar[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }

            const float4* sb4 = reinterpret_cast<const float4*>(sbias);
            uint4 pk[8];
            uint4 pk_lo[PL == 2 ? 8 : 1];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const uint32_t* vv = (c < 4) ? &v0[c * 8] : &v1[(c - 4) * 8];
                const float4 b0 = sb4[2 * c], b1 = sb4[2 * c + 1];
                float f[8] = {__uint_as_float(vv[0]) + b0.x, __uint_as_float(vv[1]) + b0.y, __uint_as_float(vv[2]) + b0.z,
                              __uint_as_float(vv[3]) + b0.w, __uint_as_float(vv[4]) + b1.x, __uint_as_float(vv[5]) + b1.y,
                              __uint_as_float(vv[6]) + b1.z, __uint_as_float(vv[7]) + b1.w};
                if (p.relu) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) f[j] = fmaxf(f[j], 0.f);
                }
                const uint32_t h0 = pack16x2(f[0], f[1], F16), h1 = pack16x2(f[2], f[3], F16);
                const uint32_t h2 = pack16x2(f[4], f[5], F16), h3 = pack16x2(f[6], f[7], F16);
                pk[c] = make_uint4(h0, h1, h2, h3);
                if constexpr (PL == 2) {
                    const float2 r0 = unpack16x2(h0, F16), r1 = unpack16x2(h1, F16);
                    const float2 r2 = unpack16x2(h2, F16), r3 = unpack16x2(h3, F16);
                    pk_lo[c] = make_uint4(pack16x2(f[0] - r0.x, f[1] - r0.y, F16), pack16x2(f[2] - r1.x, f[3] - r1.y, F16),
                                          pack16x2(f[4] - r2.x, f[5] - r2.y, F16), pack16x2(f[6] - r3.x, f[7] - r3.y, F16));
                }
            }
            // this warp's 32 rows = voxels [v, v + 32): whole lines or a piece of one line
            const int v = m_blk * 128 + q * 32;
            const int line = v / p.bw, w0 = v - line * p.bw;
            const int hh = line % p.H, dd = (line / p.H) % p.D, bb = line / (p.H * p.D);
#pragma unroll
            for (int pl = 0; pl < PL; ++pl) {
                if (lane == 0) tma_store_wait_read<0>();
                __syncwarp();
#pragma unroll
                for (int c = 0; c < 8; ++c)   // SWIZZLE_128B: 16-byte chunk c of row r lives at chunk c ^ (r & 7)
                    *reinterpret_cast<uint4*>(stg + lane * 128 + ((c ^ (lane & 7)) << 4)) = pl == 0 ? pk[c] : pk_lo[PL == 2 ? c : 0];
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                    if (p.store5d) tma_store_5d(&tmOut, stg, 0, w0, hh, dd, bb + pl * p.batch_plane);
                    else tma_store_2d(&tmOut, stg, 0, v + pl * p.out_plane_rows);
                    tma_store_commit();
                }
            }
        }
        if (lane == 0) tma_store_wait_all();
    }

    tc_fence_before();
    __syncthreads();
    if constexpr (CL > 1) cluster_sync_all();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 128);
    }
}

// ---------------------------------------------------------------------------------------------
// host launcher
// ---------------------------------------------------------------------------------------------
template <int NP, int CL>
static cudaError_t cv_configure_one() {
    cudaError_t e = cudaFuncSetAttribute(conv3d_tc_kernel<NP, CL, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, cv_smem_bytes(NP));
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(conv3d_tc_kernel<NP, CL, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, cv_smem_bytes(NP));
}

cudaError_t configure_conv3d_tc() {
    cudaError_t e;
    if ((e = cv_configure_one<1, 1>()) != cudaSuccess) return e;
    if ((e = cv_configure_one<1, 2>()) != cudaSuccess) return e;
    if ((e = cv_configure_one<3, 1>()) != cudaSuccess) return e;
    return cv_configure_one<3, 2>();
}

template <int NP, int CL>
static cudaError_t cv_launch(const CUtensorMap& a0, const CUtensorMap& a1, const CUtensorMap& b, const CUtensorMap& o,
                             const Conv3dParams& p, int f16, int num_sms, cudaStream_t stream) {
    const int tiles = p.num_m_blocks / CL;
    const int max_clusters = num_sms / CL;
    const int clusters = tiles < max_clusters ? tiles : max_clusters;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(clusters * CL);
    cfg.blockDim = dim3(kCvThreads);
    cfg.dynamicSmemBytes = cv_smem_bytes(NP);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    if (f16) return cudaLaunchKernelEx(&cfg, conv3d_tc_kernel<NP, CL, 1>, a0, a1, b, o, p);
    return cudaLaunchKernelEx(&cfg, conv3d_tc_kernel<NP, CL, 0>, a0, a1, b, o, p);
}

// np: 1 (one pass) or 3 (hi/lo planes); cl: 1 or 2 (CTA pairs, weight tile multicast; needs an even number of tiles)
cudaError_t launch_conv3d_tc(int np, int cl, int f16, const CUtensorMap& a0, const CUtensorMap& a1, const CUtensorMap& b,
                             const CUtensorMap& o, const Conv3dParams& p, int num_sms, cudaStream_t stream) {
    if (p.nt < 1 || p.nt > kCvMaxTaps || p.bw * p.bh != 128 || (p.bh + p.nt - 1) * p.bw > kCvARows || (p.bw * 128) % 1024 != 0)
        return cudaErrorInvalidValue;
    if (cl == 2 && p.num_m_blocks % 2 != 0) cl = 1;
    if (np == 1) return cl == 2 ? cv_launch<1, 2>(a0, a1, b, o, p, f16, num_sms, stream) : cv_launch<1, 1>(a0, a1, b, o, p, f16, num_sms, stream);
    if (np == 3) return cl == 2 ? cv_launch<3, 2>(a0, a1, b, o, p, f16, num_sms, stream) : cv_launch<3, 1>(a0, a1, b, o, p, f16, num_sms, stream);
    return cudaErrorInvalidValue;
}

}  // namespace pcd
