// Per-point shared-MLP layer as a persistent, warp-specialised tcgen05 GEMM (sm_100a).
//
//   D[128 x BN] (fp32, TMEM) = Arole[128 x K] (bf16, smem via TMA) * Brole[BN x K]^T (bf16, smem via TMA)
//
// Replaces the reference's `Conv1d(k=1) -> BatchNorm1d(eval) -> ReLU` triple (networks.py:46-48):
// BN is folded into W/bias on the host, bias(+per-sample time/global bias)+ReLU run in the epilogue.
// Three epilogues:
//   EPI_STORE   lanes = points, columns = channels: bias + ReLU -> bf16 row-major activations
//   EPI_MAXPOOL lanes = channels (weights are the A role), columns = points: running max over the
//               points of a cloud, + bias, ReLU, atomicMax into g[B][4096]  (networks.py:806-807;
//               the 4096-wide activation is never materialised)
//   EPI_FINAL   output.0 (64->64, BN, ReLU) in TMEM, then output.3 (64->3) in registers and the
//               sampler update (diffusion.py:246-257 / 283-287) so x_t never leaves the kernel
//               as an activation (networks.py:816, diffusion.py:167)
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer,
// warps 2..5 = epilogue (TMEM lane quarter = warp % 4).  Pipelines: smem full/empty ring
// (TMA <-> MMA) and a 2-deep TMEM accumulator ring (MMA <-> epilogue).
#include "pcd_launch.h"
#include "pcd_ptx.cuh"
#include "pcd_sampler.cuh"
#include "pcd_types.h"

namespace pcd {

constexpr int kTileM = 128;
constexpr int kTileK = 64;                       // 64 bf16 = one 128-byte swizzle row
constexpr int kABytes = kTileM * kTileK * 2;     // 16 KB
constexpr int kAccStride = 256;                  // TMEM columns per accumulator stage

// NP = number of MMA passes per k-step.  NP == 1: plain bf16.  NP == 3 ("bf16x3"): every operand is the sum of a
// hi and a lo bf16 plane (x = hi + lo to ~16 mantissa bits) and D += Ahi*Bhi + Ahi*Blo + Alo*Bhi with fp32
// accumulation -- near-fp32 products at 1/3 of the tensor throughput (SURVEY H2).  The lo plane of every tensor
// lives `plane_rows` rows below the hi plane in the SAME 2-D tensor, so the TMA maps are shared.
// NP == 4 ("c8", fp16 only): the hi pass runs in fp16 and BOTH correction terms run as ONE fp8 (e5m2) pass at twice the fp16
// rate -- the second plane of every operand is a byte plane that holds, per 64 k-elements, 64 e5m2 residuals and 64 e5m2 copies
// of the hi values (per 32 k-elements [32 x Alo8 | 32 x Ahi8] for the A role, [32 x Bhi8 | 32 x Blo8] for the B role, power-of-two
// scaled into e5m2's range), so a 128-byte swizzle row IS a K = 128 fp8 operand row and  D += Alo8*Bhi8 + Ahi8*Blo8  is four
// kind::f8f6f4 MMAs (K = 32 bytes each: residual x copy, copy x residual, twice) per k-block.
// The residual terms are 2^-11 of the product, so e5m2's 2-bit mantissa leaves ~2^-14 relative error: split-precision
// accuracy at 2 pass-equivalents instead of 3.  Same bytes per stage as NP == 3.
__host__ __device__ constexpr int tc_planes(int np) { return np >= 3 ? 2 : 1; }
// (scales kC8ScaleLo / kC8ScaleHi: pcd_types.h)
// Output staging: NBUF 4 KB tiles per epilogue warp (a ring; one tile is enough -- measured: a ring of 4 bought
// nothing, the cost of the store path is the write traffic itself, see DESIGN.md 5.1 -- and shared memory is better
// spent on pipeline stages).
__host__ __device__ constexpr int tc_store_bufs(int np, int epi) { return epi != EPI_STORE ? 0 : 1; }
// TWO = CTA-pair MMA (cta_group::2): a CTA stages only HALF of the B-role tile, so the same shared memory holds a deeper ring
__host__ __device__ constexpr int tc_stage_bytes(int bn, int np, int two) {
    return tc_planes(np) * (kABytes + (two ? bn / 2 : bn) * kTileK * 2);
}
__host__ __device__ constexpr int tc_stages(int bn, int np, int epi, int two) {
    if (two) {
        const int fit = (200 * 1024) / tc_stage_bytes(bn, np, 1);      // ~200 KB for the ring; the rest is staging + aux
        return fit > 8 ? 8 : fit;
    }
    if (np >= 3) return bn == 128 ? 3 : 4;
    if (epi == EPI_MAXPOOL) return bn == 256 ? 4 : 6;
    return bn == 256 ? 4 : 6;
}
__host__ __device__ constexpr int tc_smem_bytes(int bn, int np, int epi, int two) {
    return tc_stages(bn, np, epi, two) * tc_stage_bytes(bn, np, two) + 4 * tc_store_bufs(np, epi) * 4096 + 4096 /*aux*/ +
           1024 /*alignment slack*/;
}

// Tile order.  Measured with ncu: these GEMMs are bound by L2->SM bandwidth (~13 TB/s), not HBM, and the memory
// system merges concurrent requests for the same lines.  So the CTAs that run at the same time should ask for the
// SAME big operand tile, and each CTA should keep its own small operand between consecutive tiles:
//   MAXPOOL (weights = A role, 128 x K; points = B role, 256 x K): m fastest -- concurrent CTAs share the 32 KB/k-block
//           activation tile and the whole [M, 2048] activation is streamed from HBM exactly once;
//   STORE/FINAL (points = A role, weights = B role, up to 256 x K): waves of gridDim.x row blocks; inside a wave all
//           CTAs work on the same weight tile n_blk (shared 32 KB/k-block) and CTA c keeps row block c across the
//           num_n_blocks tiles it processes, so its activation tile is re-read from L2 and from HBM only once.
// the accumulator-free signal goes to the MMA issuer: this CTA, or the even CTA of the pair
// one arrival per epilogue WARP (after every lane's TMEM reads of the tile have completed): 4 per CTA, 8 for the pair
template <int TWO>
__device__ __forceinline__ void tempty_arrive(uint64_t* bar) {
    __syncwarp();
    if ((threadIdx.x & 31) == 0) {
        if constexpr (TWO) mbar_arrive_cluster(mapa_shared(smem_u32(bar), 0));
        else mbar_arrive(bar);
    }
}

// transposed-conv output (one parity class): 32 consecutive input-grid voxels starting at linear index v go to the strided
// 5-D view of the output grid whose box covers exactly those voxels
__device__ __forceinline__ void conv_store_5d(const CUtensorMap* tm, const void* stg, const ConvGeom& cg, int col, int v, int plane) {
    const int w0 = v % cg.W, h0 = (v / cg.W) % cg.H, d0 = (v / (cg.W * cg.H)) % cg.D;
    const int b0 = v / (cg.W * cg.H * cg.D) + plane * cg.batch_plane;
    tma_store_5d(tm, stg, col, w0, h0, d0, b0);
}

// order 1 (STORE / FINAL): n fastest -- the clusters running at the same time cover num_clusters / num_n row blocks and ALL weight
// tiles, so a row block's activations are fetched from HBM once and shared through L2 by the num_n clusters that need them at
// that moment.  The default order keeps a row block alive in L2 for num_n consecutive tiles of ONE cluster: fine while
// num_clusters x (256 rows x K x planes) fits in L2 next to the output write stream (37 MB in the one-plane modes), but with two
// planes and K = 1024 that is 74 MB and ncu shows the activations being re-read from HBM for every weight tile
// (dec4.conv2, f16mix: 12.7 GB of DRAM reads for 4.3 GB of operand, L2 hit rate 50 %).
template <int EPI>
__device__ __forceinline__ void tile_coords(int tile, int num_m, int num_n, int grid, int order, int& m_blk, int& n_blk) {
    if (EPI == EPI_MAXPOOL) { m_blk = tile % num_m; n_blk = tile / num_m; return; }
    if (order == 1) { m_blk = tile / num_n; n_blk = tile - m_blk * num_n; return; }
    const int per_group = grid * num_n;
    const int group = tile / per_group;
    const int w = tile - group * per_group;
    const int rows_left = num_m - group * grid;
    const int gsz = rows_left < grid ? rows_left : grid;
    n_blk = w / gsz;
    m_blk = group * grid + (w - n_blk * gsz);
}

// CL = cluster size (1 or 2).  With CL = 2 the two CTAs of a cluster work on neighbouring A-role blocks and the SAME
// B-role tile: each CTA fetches half of that tile and TMA-multicasts it into both shared memories, so the L2->SM
// traffic per k-block drops from 16 + 32 KB to 16 + 16 KB per CTA (BN = 256).  A stage may be refilled only when
// BOTH CTAs' MMAs have drained it, so tcgen05.commit arrives on the `empty` barrier of both CTAs (count = CL).
// OP = planes written by the STORE epilogue (2: hi + rounding residual; a single-pass layer feeding a split layer uses NP=1, OP=2)
// TWO = 1 (needs CL = 2): the pair runs ONE tcgen05.mma.cta_group::2 per k-step, issued by the even CTA, on a 256-row tile
// (128 A-role rows from each CTA, B-role tile split in halves between the two shared memories, no multicast).  Per CTA a
// stage shrinks from 48 to 32 KB (BN = 256), so the ring is 6 deep instead of 4 and every SM writes/reads a third less
// shared memory per k-step.  Barriers: `full` and `tempty` live in the even CTA (the odd CTA's TMA and epilogue signal them
// remotely), `empty` and `tfull` exist in both and are signalled by multicast commits.
// F16 = 16-bit operand / activation format (0 bf16, 1 fp16): compile time, because the pack sits in the store epilogue's
// inner loop, which bounds every K <= 512 layer (a runtime flag there cost 5 % of the step)
// EW = epilogue warps: 4 (one per TMEM lane quarter; 64-column groups through 4 KB staging tiles, tmOut box 64 x 32, SWIZZLE_128B)
// or 8 (EPI_STORE, plain 2-D stores only: two warps per lane quarter take alternate 32-column sub-groups through 2 KB staging
// tiles, tmOut box 32 x 32, SWIZZLE_64B).  With ONE warp per scheduler the epilogue issues an instruction every ~2.5 cycles
// (dependent FADD / FMNMX / F2FP chains, nothing to interleave), which makes it longer than the MMAs of a tile for every
// single-pass layer with K <= 512, every split layer with K <= 256 and the single-pass layer that also writes a byte plane
// (ncu, dec4.conv1 in f16mix: tensor pipe 59 % active, 21 % of the samples "selected"); a second warp per scheduler hides that.
template <int BN, int EPI, int NP, int CL, int OP, int TWO, int F16, int EW>
__global__ void __launch_bounds__(64 + 32 * EW, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
               const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmOut,
               const TcGemmParams p) {
    static_assert(TWO == 0 || CL == 2, "the CTA-pair MMA needs a cluster of two");
    static_assert(EW == 4 || (EW == 8 && EPI == EPI_STORE), "eight epilogue warps exist for the store epilogue only");
    constexpr int STAGES = tc_stages(BN, NP, EPI, TWO);
    constexpr int NBUF = tc_store_bufs(NP, EPI);
    constexpr int PL = tc_planes(NP);
    constexpr int B_BYTES = (TWO ? BN / 2 : BN) * kTileK * 2;     // per plane, per CTA
    constexpr int A_STAGE = PL * kABytes, B_STAGE = PL * B_BYTES;
    constexpr uint32_t IDESC = make_idesc(TWO ? 256 : 128, BN, F16);   // fp16 or bf16 operands, fp32 accumulate
    constexpr uint32_t IDESC8 = make_idesc(TWO ? 256 : 128, BN, 0);    // kind::f8f6f4: format code 1 = e5m2 (the bf16 code of kind::f16)
    static_assert(NP != 4 || (F16 == 1 && TWO == 1), "the fp8-corrected form exists for fp16 operands on the pair MMA only");
    static_assert(OP != 3 || F16 == 1, "the c8 output plane goes with fp16 hi planes");
    static_assert(NP == 1 || BN <= 128 || TWO == 1, "split precision uses BN <= 128 unless the CTA pair shares the B tile (shared memory budget)");

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sA = smem;
    uint8_t* sB = smem + STAGES * A_STAGE;
    uint8_t* stage_out = sB + STAGES * B_STAGE;               // 4 epilogue warps x NBUF x 4 KB (1024-aligned)
    uint8_t* aux = stage_out + 4 * NBUF * 4096;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(aux);            // [STAGES]
    uint64_t* empty_bar = full_bar + STAGES;                           // [STAGES]
    uint64_t* tfull_bar = empty_bar + STAGES;                          // [2]
    uint64_t* tempty_bar = tfull_bar + 2;                              // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    float* sbias = reinterpret_cast<float*>(aux + 256);                // [2][BN]  (<= 2 KB)
    float* sw3 = reinterpret_cast<float*>(aux + 256 + 2 * 256 * 4);    // [3*64 + 3]

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    // cluster-level tile schedule: a "cluster tile" = CL neighbouring A-role blocks x one B-role block
    const int crank = CL > 1 ? static_cast<int>(cluster_ctarank()) : 0;
    const int cid = blockIdx.x / CL, num_clusters = gridDim.x / CL;
    const int num_mg = p.num_m_blocks / CL;
    const int num_tiles = num_mg * p.num_n_blocks;
    const int num_kb = p.kb0 + p.kb1;
    constexpr uint16_t CMASK = static_cast<uint16_t>((1u << CL) - 1);

    if (warp == 0 && lane == 0) {
        prefetch_tensormap(&tmA0);
        prefetch_tensormap(&tmA1);
        prefetch_tensormap(&tmB);
        if (EPI == EPI_STORE) prefetch_tensormap(&tmOut);
        for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], TWO ? 1 : CL); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], TWO ? 2 * EW : EW); }
        fence_mbar_init();
    }
    if (warp == 1) {
        if constexpr (TWO) { tmem_alloc_2sm(tmem_slot, 512); tmem_relinquish_2sm(); }
        else { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (CL > 1) cluster_sync_all();   // barrier inits of every CTA are visible before any remote arrive / multicast
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // programmatic dependent launch: everything above ran while the previous kernel of the step was still draining; nothing
    // below touches global memory before that kernel has completed
    pdl_launch();
    pdl_wait();

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int tile = cid; tile < num_tiles; tile += num_clusters) {
                int m_blk, n_blk;
                tile_coords<EPI>(tile, num_mg, p.num_n_blocks, num_clusters, p.tile_order, m_blk, n_blk);
                m_blk = m_blk * CL + crank;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    if constexpr (TWO) {
                        // both CTAs' loads are credited to the EVEN CTA's full barrier, which expects the bytes of the pair
                        if (crank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * (A_STAGE + B_STAGE));
                        const uint32_t fb = mapa_shared(smem_u32(&full_bar[stage]), 0);
#pragma unroll
                        for (int pl = 0; pl < PL; ++pl) {
                            uint8_t* da = sA + stage * A_STAGE + pl * kABytes;
                            const int arow = m_blk * kTileM + pl * p.a_plane_rows;
                            if (kb < p.kb0) tma_load_2d_2sm(da, &tmA0, fb, kb * kTileK, arow);
                            else                 tma_load_2d_2sm(da, &tmA1, fb, (kb - p.kb0) * kTileK, arow);
                            tma_load_2d_2sm(sB + stage * B_STAGE + pl * B_BYTES, &tmB, fb, kb * kTileK,
                                            n_blk * BN + crank * (BN / 2) + pl * p.b_plane_rows);
                        }
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                        continue;
                    }
                    mbar_arrive_expect_tx(&full_bar[stage], A_STAGE + B_STAGE);
#pragma unroll
                    for (int pl = 0; pl < PL; ++pl) {
                        uint8_t* da = sA + stage * A_STAGE + pl * kABytes;
                        const int arow = m_blk * kTileM + pl * p.a_plane_rows;
                        if (p.conv.ntaps > 0) {
                            // implicit-GEMM convolution: the tile's 128 voxels shifted by this k-block's tap
                            const ConvGeom& cg = p.conv;
                            const int v0 = m_blk * kTileM;
                            const int w0 = v0 % cg.W, h0 = (v0 / cg.W) % cg.H, d0 = (v0 / (cg.W * cg.H)) % cg.D;
                            const int b0 = v0 / (cg.W * cg.H * cg.D) + pl * cg.batch_plane;
                            if (kb < p.kb0) {
                                const int tap = kb / cg.cin_kb, cb = kb - tap * cg.cin_kb;
                                tma_load_5d(da, &tmA0, &full_bar[stage], cb * kTileK, cg.stride * w0 + cg.dw[tap], cg.stride * h0 + cg.dh[tap],
                                            cg.stride * d0 + cg.dd[tap], b0);
                            } else {
                                tma_load_5d(da, &tmA1, &full_bar[stage], (kb - p.kb0) * kTileK, w0, h0, d0, b0);
                            }
                        } else if (kb < p.kb0) tma_load_2d(da, &tmA0, &full_bar[stage], kb * kTileK, arow);
                        else                   tma_load_2d(da, &tmA1, &full_bar[stage], (kb - p.kb0) * kTileK, arow);
                        if constexpr (CL == 1) {
                            tma_load_2d(sB + stage * B_STAGE + pl * B_BYTES, &tmB, &full_bar[stage], kb * kTileK,
                                        n_blk * BN + pl * p.b_plane_rows);
                        } else {
                            // my 1/CL slice of the shared B-role tile, delivered to every CTA of the cluster
                            constexpr int SL = BN / CL;
                            tma_load_2d_mcast(sB + stage * B_STAGE + pl * B_BYTES + crank * SL * 128, &tmB, &full_bar[stage],
                                              kb * kTileK, n_blk * BN + crank * SL + pl * p.b_plane_rows, CMASK);
                        }
                    }
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (lane == 0 && (TWO == 0 || crank == 0)) {      // CTA-pair MMA: only the even CTA issues
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int tile = cid; tile < num_tiles; tile += num_clusters) {
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * kAccStride;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint64_t da = make_sw128_kmajor_desc(smem_u32(sA + stage * A_STAGE));
                    const uint64_t db = make_sw128_kmajor_desc(smem_u32(sB + stage * B_STAGE));
#pragma unroll
                    for (int k = 0; k < kTileK / 16; ++k) {
                        // advance 16 bf16 = 32 bytes inside the 128-byte swizzle row: +2 in (addr >> 4) units
                        constexpr uint64_t A_LO = kABytes >> 4, B_LO = B_BYTES >> 4;   // lo planes follow the hi planes
                        if constexpr (TWO) {
                            tc_mma_2sm(d_tmem, da + 2 * k, db + 2 * k, IDESC, (kb | k) != 0 ? 1u : 0u);
                            if constexpr (NP == 3) {
                                tc_mma_2sm(d_tmem, da + 2 * k, db + B_LO + 2 * k, IDESC, 1u);          // hi * lo
                                tc_mma_2sm(d_tmem, da + A_LO + 2 * k, db + 2 * k, IDESC, 1u);          // lo * hi
                            }
                            // c8: 32 e5m2 k-elements (32 bytes) of the byte planes per MMA: [Alo8 | Ahi8] . [Bhi8 | Blo8]
                            if constexpr (NP == 4) tc_mma_2sm_f8(d_tmem, da + A_LO + 2 * k, db + B_LO + 2 * k, IDESC8, 1u);
                        } else {
                            tc_mma_bf16(d_tmem, da + 2 * k, db + 2 * k, IDESC, (kb | k) != 0 ? 1u : 0u);
                            if constexpr (NP == 3) {
                                tc_mma_bf16(d_tmem, da + 2 * k, db + B_LO + 2 * k, IDESC, 1u);          // hi * lo
                                tc_mma_bf16(d_tmem, da + A_LO + 2 * k, db + 2 * k, IDESC, 1u);          // lo * hi
                            }
                        }
                    }
                    // frees the smem slot once these MMAs have read it (in every CTA the slot belongs to)
                    if constexpr (TWO) tc_commit_2sm_mcast(&empty_bar[stage], CMASK);
                    else if constexpr (CL == 1) tc_commit(&empty_bar[stage]);
                    else tc_commit_mcast(&empty_bar[stage], CMASK);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                // accumulator complete -> epilogue (of both CTAs for the pair MMA)
                if constexpr (TWO) tc_commit_2sm_mcast(&tfull_bar[acc], CMASK);
                else tc_commit(&tfull_bar[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ===================== epilogue (warps 2..2+EW) =====================
        const int q = warp & 3;                    // TMEM lanes [32q, 32q+32) are visible to this warp
        const int row_in_tile = q * 32 + lane;
        const int epi_tid = threadIdx.x - 64;      // 0..32*EW-1
        constexpr int ETHREADS = 32 * EW;
        int acc = 0; uint32_t acc_phase = 0;
        int sbuf = 0;                              // staging ring position (EPI_STORE)
        (void)sbuf;

        if constexpr (EPI == EPI_FINAL) {
            for (int i = epi_tid; i < 3 * 64; i += ETHREADS) sw3[i] = p.call->s.w3[i];
            if (epi_tid < 3) sw3[3 * 64 + epi_tid] = p.call->s.b3[epi_tid];
        }

        for (int tile = cid; tile < num_tiles; tile += num_clusters) {
            int m_blk, n_blk;
            tile_coords<EPI>(tile, num_mg, p.num_n_blocks, num_clusters, p.tile_order, m_blk, n_blk);
            m_blk = m_blk * CL + crank;
            const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * kAccStride;

            if constexpr (EPI == EPI_STORE || EPI == EPI_FINAL) {
                // stage this tile's bias row (shared + per-sample part) in smem, double buffered by acc
                float* sb = sbias + acc * BN;
                const int sample = (m_blk * kTileM) / p.rows_per_sample;
                const float* bsrc = p.bias + static_cast<long long>(sample) * p.bias_sample_stride + n_blk * BN;
                for (int i = epi_tid; i < BN; i += ETHREADS) sb[i] = bsrc[i];
                asm volatile("bar.sync 1, %0;" ::"n"(ETHREADS) : "memory");

                mbar_wait(&tfull_bar[acc], acc_phase);
                tc_fence_after();
                const long long row = static_cast<long long>(m_blk) * kTileM + row_in_tile;

                if constexpr (EPI == EPI_STORE && EW == 8) {
                    // two warps per lane quarter: warp `half` takes the 32-column sub-groups half, half + 2, ...
                    const int half = (warp - 2) >> 2;
                    uint8_t* stg = stage_out + (warp - 2) * 2048;          // 32 rows x 64 bytes, SWIZZLE_64B
                    const int swz = (lane >> 1) & 3;                      // 16-byte chunk c of row r lives at chunk c ^ ((r >> 1) & 3)
#pragma unroll 1
                    for (int sg = half; sg < BN / 32; sg += 2) {
                        uint32_t v[32];
                        tmem_ld_32x32(t_addr + sg * 32, v);
                        tc_wait_ld();
                        const float4* sb4 = reinterpret_cast<const float4*>(sb + sg * 32);
                        uint4 pk[4];
                        uint4 pk2[OP >= 2 ? 4 : 1];    // OP == 2: fp16 residuals; OP == 3: [32 x e5m2 residual | 32 x e5m2 copy] (64 bytes)
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const float4 b0 = sb4[2 * c], b1 = sb4[2 * c + 1];
                            float f[8] = {__uint_as_float(v[8 * c]) + b0.x,     __uint_as_float(v[8 * c + 1]) + b0.y,
                                          __uint_as_float(v[8 * c + 2]) + b0.z, __uint_as_float(v[8 * c + 3]) + b0.w,
                                          __uint_as_float(v[8 * c + 4]) + b1.x, __uint_as_float(v[8 * c + 5]) + b1.y,
                                          __uint_as_float(v[8 * c + 6]) + b1.z, __uint_as_float(v[8 * c + 7]) + b1.w};
                            if (p.relu) {
#pragma unroll
                                for (int j = 0; j < 8; ++j) f[j] = fmaxf(f[j], 0.f);
                            }
                            const uint32_t h0 = pack16x2(f[0], f[1], F16), h1 = pack16x2(f[2], f[3], F16);
                            const uint32_t h2 = pack16x2(f[4], f[5], F16), h3 = pack16x2(f[6], f[7], F16);
                            pk[c] = make_uint4(h0, h1, h2, h3);
                            if constexpr (OP >= 2) {
                                const float2 r0 = unpack16x2(h0, F16), r1 = unpack16x2(h1, F16);
                                const float2 r2 = unpack16x2(h2, F16), r3 = unpack16x2(h3, F16);
                                if constexpr (OP == 2) {
                                    pk2[c] = make_uint4(pack16x2(f[0] - r0.x, f[1] - r0.y, F16), pack16x2(f[2] - r1.x, f[3] - r1.y, F16),
                                                        pack16x2(f[4] - r2.x, f[5] - r2.y, F16), pack16x2(f[6] - r3.x, f[7] - r3.y, F16));
                                } else {
                                    const uint32_t l0 = pack_e5m2x4((f[0] - r0.x) * kC8ScaleLo, (f[1] - r0.y) * kC8ScaleLo,
                                                                    (f[2] - r1.x) * kC8ScaleLo, (f[3] - r1.y) * kC8ScaleLo);
                                    const uint32_t l1 = pack_e5m2x4((f[4] - r2.x) * kC8ScaleLo, (f[5] - r2.y) * kC8ScaleLo,
                                                                    (f[6] - r3.x) * kC8ScaleLo, (f[7] - r3.y) * kC8ScaleLo);
                                    const uint32_t g0 = pack_e5m2x4(r0.x * kC8ScaleHi, r0.y * kC8ScaleHi, r1.x * kC8ScaleHi, r1.y * kC8ScaleHi);
                                    const uint32_t g1 = pack_e5m2x4(r2.x * kC8ScaleHi, r2.y * kC8ScaleHi, r3.x * kC8ScaleHi, r3.y * kC8ScaleHi);
                                    // residual bytes [8c, 8c + 8) of the 64-byte row, copy bytes [32 + 8c, ...)
                                    if ((c & 1) == 0) { pk2[c / 2].x = l0; pk2[c / 2].y = l1; pk2[2 + c / 2].x = g0; pk2[2 + c / 2].y = g1; }
                                    else              { pk2[c / 2].z = l0; pk2[c / 2].w = l1; pk2[2 + c / 2].z = g0; pk2[2 + c / 2].w = g1; }
                                }
                            }
                        }
                        if (lane == 0) tma_store_wait_read<0>();      // the previous store of this warp has finished READING the tile
                        __syncwarp();
#pragma unroll
                        for (int c = 0; c < 4; ++c) *reinterpret_cast<uint4*>(stg + lane * 64 + ((c ^ swz) << 4)) = pk[c];
                        fence_proxy_async_smem();
                        __syncwarp();
                        if (lane == 0) {
                            tma_store_2d(&tmOut, stg, n_blk * BN + sg * 32, m_blk * kTileM + q * 32);
                            tma_store_commit();
                        }
                        if constexpr (OP >= 2) {
                            if (lane == 0) tma_store_wait_read<0>();
                            __syncwarp();
#pragma unroll
                            for (int c = 0; c < 4; ++c) *reinterpret_cast<uint4*>(stg + lane * 64 + ((c ^ swz) << 4)) = pk2[c];
                            fence_proxy_async_smem();
                            __syncwarp();
                            if (lane == 0) {
                                tma_store_2d(&tmOut, stg, n_blk * BN + sg * 32, m_blk * kTileM + q * 32 + p.out_plane_rows);
                                tma_store_commit();
                            }
                        }
                    }
                } else if constexpr (EPI == EPI_STORE) {
                    // TMEM -> registers -> (+bias, ReLU, bf16) -> 128B-swizzled smem staging -> TMA store.
                    // Each warp owns a 32-row x 64-column (4 KB) staging tile; a direct st.global from the
                    // TMEM layout (thread = row) would scatter every warp store over 32 cache lines.
                    uint8_t* stg_base = stage_out + (warp - 2) * (NBUF > 0 ? NBUF : 1) * 4096;
#pragma unroll 1
                    for (int g2 = 0; g2 < BN / 64; ++g2) {
                        uint32_t v0[32], v1[32];
                        tmem_ld_32x32(t_addr + g2 * 64, v0);
                        tmem_ld_32x32(t_addr + g2 * 64 + 32, v1);
                        tc_wait_ld();
                        const float4* sb4 = reinterpret_cast<const float4*>(sb + g2 * 64);
                        uint4 pk[8];
                        uint4 pk_lo[OP >= 2 ? 8 : 1];   // OP == 3: per 32 channels [32 e5m2 residuals | 32 e5m2 copies of the values]
#pragma unroll
                        for (int c = 0; c < 8; ++c) {
                            const uint32_t* vv = (c < 4) ? &v0[c * 8] : &v1[(c - 4) * 8];
                            const float4 b0 = sb4[2 * c], b1 = sb4[2 * c + 1];
                            float f[8] = {__uint_as_float(vv[0]) + b0.x, __uint_as_float(vv[1]) + b0.y,
                                          __uint_as_float(vv[2]) + b0.z, __uint_as_float(vv[3]) + b0.w,
                                          __uint_as_float(vv[4]) + b1.x, __uint_as_float(vv[5]) + b1.y,
                                          __uint_as_float(vv[6]) + b1.z, __uint_as_float(vv[7]) + b1.w};
                            if (p.relu) {
#pragma unroll
                                for (int j = 0; j < 8; ++j) f[j] = fmaxf(f[j], 0.f);
                            }
                            const uint32_t h0 = pack16x2(f[0], f[1], F16), h1 = pack16x2(f[2], f[3], F16);
                            const uint32_t h2 = pack16x2(f[4], f[5], F16), h3 = pack16x2(f[6], f[7], F16);
                            pk[c] = make_uint4(h0, h1, h2, h3);
                            if constexpr (OP == 2) {
                                const float2 r0 = unpack16x2(h0, F16), r1 = unpack16x2(h1, F16);
                                const float2 r2 = unpack16x2(h2, F16), r3 = unpack16x2(h3, F16);
                                pk_lo[c] = make_uint4(pack16x2(f[0] - r0.x, f[1] - r0.y, F16), pack16x2(f[2] - r1.x, f[3] - r1.y, F16),
                                                      pack16x2(f[4] - r2.x, f[5] - r2.y, F16), pack16x2(f[6] - r3.x, f[7] - r3.y, F16));
                            }
                            if constexpr (OP == 3) {
                                const float2 r0 = unpack16x2(h0, F16), r1 = unpack16x2(h1, F16);
                                const float2 r2 = unpack16x2(h2, F16), r3 = unpack16x2(h3, F16);
                                const uint32_t l0 = pack_e5m2x4((f[0] - r0.x) * kC8ScaleLo, (f[1] - r0.y) * kC8ScaleLo,
                                                                (f[2] - r1.x) * kC8ScaleLo, (f[3] - r1.y) * kC8ScaleLo);
                                const uint32_t l1 = pack_e5m2x4((f[4] - r2.x) * kC8ScaleLo, (f[5] - r2.y) * kC8ScaleLo,
                                                                (f[6] - r3.x) * kC8ScaleLo, (f[7] - r3.y) * kC8ScaleLo);
                                const uint32_t g0 = pack_e5m2x4(r0.x * kC8ScaleHi, r0.y * kC8ScaleHi, r1.x * kC8ScaleHi, r1.y * kC8ScaleHi);
                                const uint32_t g1 = pack_e5m2x4(r2.x * kC8ScaleHi, r2.y * kC8ScaleHi, r3.x * kC8ScaleHi, r3.y * kC8ScaleHi);
                                // per 32 channels s = c / 4 the 64-byte half row is [32 residual bytes | 32 copy bytes]: values 8c..8c+7 are
                                // residual bytes 64 s + 8 (c % 4) and copy bytes 64 s + 32 + 8 (c % 4); even c fills .xy, odd c .zw
                                const int ch = 4 * (c / 4) + (c % 4) / 2;
                                if ((c & 1) == 0) { pk_lo[ch].x = l0; pk_lo[ch].y = l1; pk_lo[ch + 2].x = g0; pk_lo[ch + 2].y = g1; }
                                else              { pk_lo[ch].z = l0; pk_lo[ch].w = l1; pk_lo[ch + 2].z = g0; pk_lo[ch + 2].w = g1; }
                            }
                        }
                        // the TMA store that used this staging tile NBUF stores ago must have finished READING it
                        uint8_t* stg = stg_base + sbuf * 4096;
                        if constexpr (NBUF > 1) { if (++sbuf == NBUF) sbuf = 0; }
                        if (lane == 0) tma_store_wait_read<(NBUF > 1 ? NBUF - 1 : 0)>();
                        __syncwarp();
#pragma unroll
                        for (int c = 0; c < 8; ++c)   // SWIZZLE_128B: 16-byte chunk c of row r lives at chunk c ^ (r & 7)
                            *reinterpret_cast<uint4*>(stg + lane * 128 + ((c ^ (lane & 7)) << 4)) = pk[c];
                        fence_proxy_async_smem();
                        __syncwarp();
                        if (lane == 0) {
                            if (p.conv.store5d) conv_store_5d(&tmOut, stg, p.conv, n_blk * BN + g2 * 64, m_blk * kTileM + q * 32, 0);
                            else tma_store_2d(&tmOut, stg, n_blk * BN + g2 * 64, m_blk * kTileM + q * 32);
                            tma_store_commit();
                        }
                        if constexpr (OP >= 2) {
                            // lo plane: residual of the 16-bit rounding (OP == 3: the e5m2 byte plane), stored out_plane_rows rows below
                            if (lane == 0) tma_store_wait_read<0>();
                            __syncwarp();
#pragma unroll
                            for (int c = 0; c < 8; ++c)
                                *reinterpret_cast<uint4*>(stg + lane * 128 + ((c ^ (lane & 7)) << 4)) = pk_lo[c];
                            fence_proxy_async_smem();
                            __syncwarp();
                            if (lane == 0) {
                                if (p.conv.store5d) conv_store_5d(&tmOut, stg, p.conv, n_blk * BN + g2 * 64, m_blk * kTileM + q * 32, 1);
                                else tma_store_2d(&tmOut, stg, n_blk * BN + g2 * 64, m_blk * kTileM + q * 32 + p.out_plane_rows);
                                tma_store_commit();
                            }
                        }
                    }
                } else {  // EPI_FINAL, BN == 64
                    float e0 = sw3[192], e1 = sw3[193], e2 = sw3[194];
#pragma unroll 1
                    for (int c = 0; c < 2; ++c) {
                        uint32_t v[32];
                        tmem_ld_32x32(t_addr + c * 32, v);
                        tc_wait_ld();
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float h = fmaxf(__uint_as_float(v[j]) + sb[c * 32 + j], 0.f);
                            e0 = fmaf(sw3[c * 32 + j], h, e0);
                            e1 = fmaf(sw3[64 + c * 32 + j], h, e1);
                            e2 = fmaf(sw3[128 + c * 32 + j], h, e2);
                        }
                    }
                    // all TMEM reads of this tile are done: release the accumulator before the global-memory tail
                    tc_fence_before();
                    tempty_arrive<TWO>(&tempty_bar[acc]);
                    sampler_apply(p.call->s, row, e0, e1, e2);
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                    continue;
                }
            } else {  // EPI_MAXPOOL: lanes = channels, columns = points
                mbar_wait(&tfull_bar[acc], acc_phase);
                tc_fence_after();
                const int ch = m_blk * kTileM + row_in_tile;
                const float bch = p.bias[ch];
#pragma unroll 1
                for (int h = 0; h < BN / 128; ++h) {
                    const long long pt0 = static_cast<long long>(n_blk) * BN + h * 128;
                    const int sample = static_cast<int>(pt0 / p.rows_per_sample);
                    const int n0 = static_cast<int>(pt0 - static_cast<long long>(sample) * p.rows_per_sample);
                    const int nvalid = min(max(p.n_valid - n0, 0), 128);
                    float mx = -3.0e38f;
#pragma unroll 1
                    for (int c = 0; c < 4; ++c) {
                        uint32_t v[32];
                        tmem_ld_32x32(t_addr + h * 128 + c * 32, v);
                        tc_wait_ld();
                        if (c * 32 + 32 <= nvalid) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) mx = fmaxf(mx, __uint_as_float(v[j]));
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (c * 32 + j < nvalid) mx = fmaxf(mx, __uint_as_float(v[j]));
                        }
                    }
                    // max commutes with the monotone (+bias, ReLU): one atomic per channel per 128 points
                    if (nvalid > 0 && sample < p.num_samples)
                        atomic_max_nonneg(&p.gmax[static_cast<long long>(sample) * p.ld_g + ch], fmaxf(mx + bch, 0.f));
                }
            }
            tc_fence_before();
            tempty_arrive<TWO>(&tempty_bar[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if (EPI == EPI_STORE && lane == 0) tma_store_wait_all();
    }

    tc_fence_before();
    __syncthreads();
    if constexpr (CL > 1) cluster_sync_all();   // no CTA may exit while a peer can still multicast into it / arrive on its barriers
    if (warp == 1) {
        tc_fence_after();
        if constexpr (TWO) tmem_dealloc_2sm(tmem_base, 512);
        else tmem_dealloc(tmem_base, 512);
    }
}

// ---------------------------------------------------------------------------------------------
// host launcher
// ---------------------------------------------------------------------------------------------
template <int BN, int EPI, int NP, int CL, int OP, int TWO, int EW>
static cudaError_t configure_ew() {
    if constexpr (NP != 4 && OP != 3) {   // the fp8-corrected forms exist for fp16 hi planes only
        cudaError_t e = cudaFuncSetAttribute(gemm_tc_kernel<BN, EPI, NP, CL, OP, TWO, 0, EW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             tc_smem_bytes(BN, NP, EPI, TWO));
        if (e != cudaSuccess) return e;
    }
    return cudaFuncSetAttribute(gemm_tc_kernel<BN, EPI, NP, CL, OP, TWO, 1, EW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                tc_smem_bytes(BN, NP, EPI, TWO));
}
template <int BN, int EPI, int NP, int CL, int OP, int TWO>
static cudaError_t configure_one() {
    cudaError_t e = configure_ew<BN, EPI, NP, CL, OP, TWO, 4>();
    if (e != cudaSuccess) return e;
    if constexpr (EPI == EPI_STORE) return configure_ew<BN, EPI, NP, CL, OP, TWO, 8>();
    else return cudaSuccess;
}

// opt every instantiation into its dynamic shared memory size (once per device, outside any capture)
cudaError_t configure_gemm_tc() {
    cudaError_t e;
#define CFG(BN, EPI, NP, OP)                                                              \
    if ((e = configure_one<BN, EPI, NP, 1, OP, 0>()) != cudaSuccess) return e;            \
    if ((e = configure_one<BN, EPI, NP, 2, OP, 0>()) != cudaSuccess) return e;            \
    if ((e = configure_one<BN, EPI, NP, 2, OP, 1>()) != cudaSuccess) return e;
    // split precision on 256-column tiles exists only as the pair MMA (each CTA stages half of the B tile: 64 KB per stage)
    if ((e = configure_one<256, EPI_STORE, 3, 2, 2, 1>()) != cudaSuccess) return e;
    if ((e = configure_one<256, EPI_STORE, 3, 2, 1, 1>()) != cudaSuccess) return e;   // ... whose lo output plane nobody reads
    if ((e = configure_one<256, EPI_STORE, 3, 2, 3, 1>()) != cudaSuccess) return e;   // ... or feeds an fp8-corrected layer
    // fp8-corrected split layers (NP = 4): pair MMA on 256-column tiles; output = hi only / hi + lo16 / hi + c8 byte plane
    if ((e = configure_one<256, EPI_STORE, 4, 2, 1, 1>()) != cudaSuccess) return e;
    if ((e = configure_one<256, EPI_STORE, 4, 2, 2, 1>()) != cudaSuccess) return e;
    if ((e = configure_one<256, EPI_STORE, 4, 2, 3, 1>()) != cudaSuccess) return e;
    CFG(64, EPI_STORE, 1, 1) CFG(128, EPI_STORE, 1, 1) CFG(256, EPI_STORE, 1, 1) CFG(128, EPI_MAXPOOL, 1, 1) CFG(256, EPI_MAXPOOL, 1, 1)
    CFG(64, EPI_FINAL, 1, 1) CFG(64, EPI_STORE, 3, 2) CFG(128, EPI_STORE, 3, 2) CFG(128, EPI_MAXPOOL, 3, 2) CFG(64, EPI_FINAL, 3, 2)
    CFG(256, EPI_STORE, 1, 2)
    CFG(256, EPI_STORE, 1, 3) CFG(128, EPI_STORE, 3, 3)     // producers of a c8 byte plane: single-pass / split layers
#undef CFG
    return cudaSuccess;
}

template <int BN, int EPI, int NP, int CL, int OP, int TWO, int EW>
static cudaError_t launch_ew(const CUtensorMap& a0, const CUtensorMap& a1, const CUtensorMap& b, const CUtensorMap& o,
                             const TcGemmParams& p, int num_sms, cudaStream_t stream) {
    constexpr int smem = tc_smem_bytes(BN, NP, EPI, TWO);
    const int tiles = (p.num_m_blocks / CL) * p.num_n_blocks;        // cluster tiles
    const int max_clusters = num_sms / CL;
    const int clusters = tiles < max_clusters ? tiles : max_clusters;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(clusters * CL);
    cfg.blockDim = dim3(64 + 32 * EW);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 2;
    if (p.f16) return cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BN, EPI, NP, CL, OP, TWO, 1, EW>, a0, a1, b, o, p);
    if constexpr (NP == 4 || OP == 3) return cudaErrorInvalidValue;
    else return cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BN, EPI, NP, CL, OP, TWO, 0, EW>, a0, a1, b, o, p);
}
// p.epi_warps == 8 selects the eight-warp store epilogue (the caller's tmOut then has a 32 x 32 box with SWIZZLE_64B)
template <int BN, int EPI, int NP, int CL, int OP, int TWO>
static cudaError_t launch_cl(const CUtensorMap& a0, const CUtensorMap& a1, const CUtensorMap& b, const CUtensorMap& o,
                             const TcGemmParams& p, int num_sms, cudaStream_t stream) {
    if constexpr (EPI == EPI_STORE) {
        if (p.epi_warps == 8) return launch_ew<BN, EPI, NP, CL, OP, TWO, 8>(a0, a1, b, o, p, num_sms, stream);
    }
    return launch_ew<BN, EPI, NP, CL, OP, TWO, 4>(a0, a1, b, o, p, num_sms, stream);
}

// mode: 0 = one CTA per tile, 1 = CTA pair with TMA multicast of the shared tile, 2 = CTA pair with the pair MMA (cta_group::2)
template <int BN, int EPI, int NP, int OP>
static cudaError_t launch_one(int mode, const CUtensorMap& a0, const CUtensorMap& a1, const CUtensorMap& b, const CUtensorMap& o,
                              const TcGemmParams& p, int num_sms, cudaStream_t stream) {
    if (mode == 2) return launch_cl<BN, EPI, NP, 2, OP, 1>(a0, a1, b, o, p, num_sms, stream);
    if (mode == 1) return launch_cl<BN, EPI, NP, 2, OP, 0>(a0, a1, b, o, p, num_sms, stream);
    return launch_cl<BN, EPI, NP, 1, OP, 0>(a0, a1, b, o, p, num_sms, stream);
}

// `cl` = 1: one CTA per tile; 2: CTA pairs (needs num_m_blocks even and a B-role tensor map whose box has BN/2 rows), with
// `two_sm` != 0 selecting the pair MMA (cta_group::2) instead of TMA multicast + per-CTA MMAs;
// `out_planes` = 2 with np == 1: single-pass layer that also writes the lo plane (only BN = 256 STORE is instantiated);
// `out_planes` = 3: the second output plane is the e5m2 byte plane an fp8-corrected consumer (np == 4) reads
cudaError_t launch_gemm_tc(int bn, int epi, int np, int out_planes, int cl, int two_sm, const CUtensorMap& a0, const CUtensorMap& a1,
                           const CUtensorMap& b, const CUtensorMap& o, const TcGemmParams& p, int num_sms, cudaStream_t stream) {
    if (cl != 1 && cl != 2) return cudaErrorInvalidValue;
    const int mode = cl == 1 ? 0 : (two_sm ? 2 : 1);
#define GO(BN, EPI, NP, OP) return launch_one<BN, EPI, NP, OP>(mode, a0, a1, b, o, p, num_sms, stream)
    if (np == 1 && out_planes >= 2) {
        if (epi == EPI_STORE && bn == 256 && out_planes == 2) GO(256, EPI_STORE, 1, 2);
        if (epi == EPI_STORE && bn == 256 && out_planes == 3) GO(256, EPI_STORE, 1, 3);
        return cudaErrorInvalidValue;
    }
    if (np == 4) {
        if (epi != EPI_STORE || bn != 256 || mode != 2) return cudaErrorInvalidValue;
        if (out_planes == 1) return launch_cl<256, EPI_STORE, 4, 2, 1, 1>(a0, a1, b, o, p, num_sms, stream);
        if (out_planes == 2) return launch_cl<256, EPI_STORE, 4, 2, 2, 1>(a0, a1, b, o, p, num_sms, stream);
        return launch_cl<256, EPI_STORE, 4, 2, 3, 1>(a0, a1, b, o, p, num_sms, stream);
    }
    if (np == 1) {
        if (epi == EPI_STORE) {
            if (bn == 64) GO(64, EPI_STORE, 1, 1);
            if (bn == 128) GO(128, EPI_STORE, 1, 1);
            if (bn == 256) GO(256, EPI_STORE, 1, 1);
        } else if (epi == EPI_MAXPOOL) {
            if (bn == 128) GO(128, EPI_MAXPOOL, 1, 1);
            if (bn == 256) GO(256, EPI_MAXPOOL, 1, 1);
        } else if (epi == EPI_FINAL) {
            if (bn == 64) GO(64, EPI_FINAL, 1, 1);
        }
    } else if (np == 3) {
        if (epi == EPI_STORE && bn == 256) {
            if (mode != 2) return cudaErrorInvalidValue;
            if (out_planes == 1) return launch_cl<256, EPI_STORE, 3, 2, 1, 1>(a0, a1, b, o, p, num_sms, stream);
            if (out_planes == 3) return launch_cl<256, EPI_STORE, 3, 2, 3, 1>(a0, a1, b, o, p, num_sms, stream);
            return launch_cl<256, EPI_STORE, 3, 2, 2, 1>(a0, a1, b, o, p, num_sms, stream);
        }
        if (epi == EPI_STORE) {
            if (bn == 128 && out_planes == 3) GO(128, EPI_STORE, 3, 3);
            if (bn == 64) GO(64, EPI_STORE, 3, 2);
            if (bn == 128) GO(128, EPI_STORE, 3, 2);
        } else if (epi == EPI_MAXPOOL) {
            if (bn == 128) GO(128, EPI_MAXPOOL, 3, 2);
        } else if (epi == EPI_FINAL) {
            if (bn == 64) GO(64, EPI_FINAL, 3, 2);
        }
    }
#undef GO
    return cudaErrorInvalidValue;
}

}  // namespace pcd
