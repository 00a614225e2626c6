// Persistent kernel for the latent-diffusion path (BASELINE config 4): the WHOLE reverse loop of
// LatentDiffusion.sample / sample2 / sample3 (reference diffusion.py:575-707) over SimpleLatentUNetPointNet
// (networks.py:962-1106), and SimplePointNetVAE.decode (networks.py:1144-1154, 1219-1231), as one cooperative launch.
//
// Why a persistent kernel: rows are samples (M = B = 128 per GPU at config 4), so a reverse step is 4.9 GFLOP over 76 MB of
// L2-resident fp32 weights -- a few microseconds of math behind ~40 dependent launches.  The CUDA-graph version spent
// 336 us per step almost entirely on launch/drain latency.  Here one CTA per SM walks a small "program" of phases (kept in
// shared memory); phases are separated by a grid barrier (one release-reduction + relaxed polling, 1.5 us), nothing returns
// to the host between the S steps, and the time MLP / t_emb half of enc1 is hoisted out of the loop (one row per step).
//
// Arithmetic: every Linear is a set of 128 x 64 x K tile jobs on tcgen05 (kind::tf32, fp32 accumulators in TMEM) with the
// 3xTF32 split (x = hi + lo; D += lo*hi + hi*lo + hi*hi): < 2^-20 relative per product, i.e. the results sit inside the fp32
// parity bound (2e-5 per forward) that the CUDA-core path was held to.  kind::tf32 ignores the 13 low mantissa bits of its
// fp32 containers (measured, DESIGN.md §5.4), so a value as loaded IS its hi operand and only lo = x - trunc(x) is computed.
// Operands stay fp32 in global memory (weights 76 MB: L2 resident).
//   * Weights are stored tile-major and pre-swizzled, so a 64 x 32 (or 128 x 32) tile is ONE 8 / 16 KB bulk copy (cp.async.bulk, mbarrier
//     complete_tx) that lands in the canonical SWIZZLE_128B K-major layout; warps 4-7 write the lo plane next to it.
//   * Activations (the A operand) are read by the tensor core from TMEM: warps 0-3 stage their rows of the chunk with cp.async,
//     read them back row-per-thread, and tcgen05.st the hi / lo planes into a 4-stage TMEM ring.  In the first version both
//     operands went through shared memory (168 KB of shared-memory traffic per 32-wide chunk: the bound of that version).
//   * One lane of warp 8 issues the twelve MMAs of a chunk and commits them to the barrier that frees both stages.
// History (batch 128, us per reverse step): CUDA graph of ~40 fp32 CUDA-core launches 336; this kernel on warp-level
// mma.sync 296 (30 % of a legacy TF32 rate that is itself 1/8 of tcgen05's); tcgen05, both operands in shared memory 302;
// vectorised epilogues + one-round-trip GroupNorm loads + cheap split 178; program in shared memory + release-red barrier
// 162; no hi write-back 151; activations through TMEM 140; 128-column tiles for the three big layers + ONE call site for the
// phase interpreter (the code is 150 KB, far beyond the instruction cache: halving it sped up every phase) 138; one chunk per split for the small layers 136.  The per-phase
// trace (PCD_LT_TRACE, tools/trace_latent.py) and timing experiments without the split or the MMAs are what found each of these.  Tried and
// rejected: rows straight into registers (32 lines per load instruction: 160), deeper rings (NST 6 / PF 4: 143), A and W work
// shared by all 8 warps (157), two-level grid barrier, more than 168 registers (9 warps: one scheduler holds 3 of them),
// starting the next GEMM phase's first weight tiles before the barrier (145.7 against 139.4 without, same build and box),
// completion counters per (row tile, GroupNorm group) instead of the grid barrier between a GEMM phase and its GroupNorm phase
// (round 2: every worker warp fences + bumps a counter after its partial sums, consumer warps poll: 126.2 against 124.2 us at batch
// 128 and 811 against 533 at batch 1024 -- a device-scope fence per warp and job costs more than one barrier per phase).
//
// Split-K partial sums are written to an fp32 workspace and reduced in a FIXED order by the GroupNorm phase, and the split
// count depends on the layer shape only, so a row's result does not depend on the batch it is in (sharded == unsharded).
#include <cstdio>
#include <cstdlib>
#include <type_traits>
#include <vector>

#include "pcd_ptx.cuh"
#include "pcd_sampler.cuh"
#include "pcd_types.h"

namespace pcd {

namespace {

constexpr int BM = 128, BN = 64, BK = 32, NST = 4, PF = 2;     // rings of NST stages; weight bulk copies run PF chunks ahead
constexpr int BN_MAX = 128;                                     // the big split-K layers run 128-column tiles (op.bn), the rest 64
constexpr int W_TILE = BN * BK;                                 // floats per 64-row weight plane (8 KB); a 128-row tile is two of them
constexpr int W_PLANE = BN_MAX * BK;                            // shared-memory stage: W hi (as landed) | W lo, planes W_PLANE floats apart
constexpr int STAGE = 2 * W_PLANE;
constexpr int NSA = 3, PFA = 2;                                 // activation staging ring (freed as soon as a warp has read its rows)
constexpr int A_PITCH = 36;                                     // floats per staged row: 128 bytes + 16 -> a quarter-warp's 16-byte
constexpr int A_STAGE = BM * A_PITCH;                           // reads of 8 consecutive rows hit 8 distinct bank groups
// TMEM (512 columns): accumulator in [0, 128); activation ring: stage s holds the chunk's hi plane in [128 + 64 s, + 32) and its
// lo plane in the next 32 columns -- lane = tile row, one TF32 element per 32-bit column (the A-operand layout of M = 128 MMAs)
constexpr uint32_t TMEM_COLS = 512, TMEM_A0 = BN_MAX, TMEM_A_STAGE = 64;
constexpr int NWORK = 256;          // warps 0-3: activation rows -> registers -> TMEM; warps 4-7: weight split; all 8: epilogues;
constexpr int NTHREADS = NWORK + 32;   // warp 8: tcgen05.mma issuer
// kind::tf32: D fp32 (bits 4-5 = 1), A/B format 2 = TF32 (bits 7-9, 10-12), K-major, N >> 3 at 17, M >> 4 at 24
__host__ __device__ constexpr uint32_t idesc_tf32(uint32_t bn) { return (1u << 4) | (2u << 7) | (2u << 10) | ((bn >> 3) << 17) | ((BM >> 4) << 24); }

// 16-byte L2-only async copy; src_bytes = 0 zero-fills (rows past the last sample)
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// one 8 KB weight tile, global -> shared, completion counted in bytes on an mbarrier (TMA bulk copy, no tensor map)
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// D[tmem] (+)= A[tmem] * B[smem]^T, tf32 inputs (fp32 containers; the MMA ignores the 13 low mantissa bits), M = 128, N from idesc, K = 8
__device__ __forceinline__ void tc_mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// 32 registers per thread -> 32 lanes x 32 consecutive 32-bit columns (thread = lane = tile row)
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
          "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]),
          "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]),
          "r"(v[30]), "r"(v[31])
        : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// per-CTA state of the tile pipeline (lives for the whole kernel)
struct Pipe {
    float* ring;            // NST weight stages, 1024-byte aligned
    float* aring;           // NSA activation staging stages (behind the weight ring)
    uint64_t* mma_done;     // [NST] one arrival (tcgen05.commit) per use of a stage
    uint64_t* w_full;       // [NST] the weight tile of a stage has landed (bulk copy, complete_tx)
    uint64_t* ready;        // [NST] the stage has been split into hi / lo planes (one arrival per worker warp)
    uint64_t* acc_free;     // the epilogue has read the accumulator out of TMEM (one arrival per worker warp)
    uint32_t tmem;          // accumulator: 128 lanes x 64 fp32 columns
    uint32_t gc;            // chunks issued so far (uniform across the CTA): stage = gc % NST, use = gc / NST
    uint32_t jobs;          // tile jobs done so far by this CTA
};



// Grid barrier: one release-reduction per CTA on a monotonic counter (fire and forget), then relaxed polling -- no L1
// invalidation per poll -- and one acquire fence.  (A two-level version, group counters + top counter + flag, was slower:
// 3.0 us instead of 1.5 us per barrier, every level adds a fence and an L2 round trip.)
__device__ __forceinline__ void grid_sync(unsigned* counter, unsigned& target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        target += gridDim.x;
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;\n" ::"l"(counter) : "memory");
        unsigned v, polls = 0;
        do {
            asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];\n" : "=r"(v) : "l"(counter) : "memory");
            if (++polls > (1u << 26)) __trap();      // ~30 s: a lost CTA must surface as a launch error, never as a hung GPU
        } while (v < target);
        asm volatile("fence.acq_rel.gpu;\n" ::: "memory");
    }
    __syncthreads();
}

struct StepCtx {
    int step;       // reverse-loop step (0 in the prologue and in forward mode)
    int forward;    // 1: per-sample t, eps written to eps_out; 0: sampler
};

__device__ __forceinline__ const float* bias_row(const LtOp& op, int row, const StepCtx& cx) {
    if (op.bias_mode == 0) return op.bias;
    return op.bias + static_cast<long long>(cx.forward ? row : cx.step) * op.bias_ld;
}

// MMA-issuer side of one job (one lane of warp 8): per chunk, wait until the activation warps have put the chunk's hi / lo
// planes into TMEM and the weight warps have written the weight lo plane, issue the twelve MMAs (K = 8 each: lo*hi, hi*lo,
// hi*hi per k-step; A from TMEM, B through a SWIZZLE_128B descriptor) and commit them to the barrier that frees both stages.
template <int BN_>
__device__ void gemm_item_mma(const LtOp& op, Pipe& pp) {
    const int nchunks = op.chunks_per_split;
    const uint32_t gc0 = pp.gc;
    // SWIZZLE_128B K-major descriptor: [0,14) address >> 4, [16,30) LBO (unused) = 1, [32,46) SBO = 1024 >> 4, [46,48) version 1,
    // [61,64) layout 2; everything but the address is constant, and the address advances by whole 16-byte units
    const uint64_t hi_bits = (static_cast<uint64_t>(1024 >> 4) << 32) | (static_cast<uint64_t>(1) << 46) | (static_cast<uint64_t>(2) << 61);
    const uint32_t lo_base = ((smem_u32(pp.ring) & 0x3FFFFu) >> 4) | (1u << 16);
    constexpr uint32_t idesc = idesc_tf32(BN_);
    if (pp.jobs > 0) mbar_wait(pp.acc_free, (pp.jobs - 1) & 1);      // the previous job's epilogue has drained the accumulator
    tc_fence_after();
    for (int ci = 0; ci < nchunks; ++ci) {
        const uint32_t g = gc0 + ci, st = g % NST;
        mbar_wait(&pp.ready[st], (g / NST) & 1);
        tc_fence_after();
        const uint32_t a_hi = pp.tmem + TMEM_A0 + st * TMEM_A_STAGE, a_lo = a_hi + 32;
        const uint32_t w_hi = lo_base + ((st * STAGE * 4) >> 4), w_lo = w_hi + ((W_PLANE * 4) >> 4);
#pragma unroll
        for (int k = 0; k < BK / 8; ++k) {
            tc_mma_tf32_ts(pp.tmem, a_lo + 8 * k, hi_bits | (w_hi + 2 * k), idesc, (ci | k) ? 1u : 0u);     // small terms first
            tc_mma_tf32_ts(pp.tmem, a_hi + 8 * k, hi_bits | (w_lo + 2 * k), idesc, 1u);
            tc_mma_tf32_ts(pp.tmem, a_hi + 8 * k, hi_bits | (w_hi + 2 * k), idesc, 1u);
        }
        tc_commit(&pp.mma_done[st]);
    }
    pp.gc = gc0 + nchunks;
    pp.jobs += 1;
}

// worker side of one (m_tile, n_tile, split) job: acc[128 x 64] (TMEM) = A[m0.., k-range] * W[n0.., k-range]^T
//   warps 0-3: thread = tile row.  A warp stages its own 32 rows of the chunk with cp.async (coalesced: 8 lanes per 128-byte
//              line, two chunks ahead, padded rows so that the row-per-thread reads are conflict free), reads its row back,
//              forms lo = x - trunc(x) in registers and writes hi (as loaded) / lo to the TMEM stage with tcgen05.st: the
//              activation operand is read by the tensor core from TMEM, not from shared memory.  (Loading the row straight into
//              registers, one 128-byte line per lane, was slower: 32 lines per load instruction.)
//   warps 4-7: one thread issues the 8 KB weight-tile bulk copies (PF chunks ahead); all wait for the tile and write its lo plane.
// The 3xTF32 split: tcgen05 kind::tf32 IGNORES the 13 low mantissa bits of its fp32 containers (measured: masking them first
// gives bit-identical results, DESIGN.md §5.4), so the loaded value already is the hi operand (hi = trunc(x)) and only
// lo = x - trunc(x) -- exact in fp32, truncated again by the MMA -- has to be produced.  x - (hi + lo) < 2^-20 |x|.
template <int BN_>
__device__ void gemm_item(const LtOp& op, const LatentCall& c, const StepCtx& cx, int rows, int m_tile, int n_tile, int split,
                          Pipe& pp) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int bn = BN_;                        // 64, or 128 (LT_PARTIAL layers only)
    const int m0 = m_tile * BM, n0 = n_tile * bn;
    const int nchunks = op.chunks_per_split;
    const int kbase = split * nchunks * BK;
    const uint32_t gc0 = pp.gc;

    if (warp < 4) {
        // warp w stages and consumes tile rows 32 w .. 32 w + 31 only (its TMEM lane quarter): no CTA-wide barrier in the loop
        auto issue = [&](int ci) {
            float* sA = pp.aring + ((gc0 + ci) % NSA) * A_STAGE;
            const int kg = kbase + ci * BK;
            const float* src;
            int ld;
            if (kg < op.K0) { src = (op.A0 ? op.A0 : c.z) + kg; ld = op.lda0; }
            else { src = op.A1 + (kg - op.K0); ld = op.lda1; }
#pragma unroll
            for (int i = 0; i < 8; ++i) {                       // 8 lanes cover one row's 128 bytes, 4 rows per instruction
                const int idx = lane + 32 * i, row = warp * 32 + (idx >> 3), cc = idx & 7;
                const int gr = m0 + row;
                const bool ok = gr < rows;
                cp_async16(smem_u32(sA + row * A_PITCH + cc * 4), src + static_cast<long long>(ok ? gr : 0) * ld + cc * 4, ok ? 16 : 0);
            }
        };
#pragma unroll
        for (int s0 = 0; s0 < PFA; ++s0) {
            if (s0 < nchunks) issue(s0);
            cp_async_commit();
        }
        for (int ci = 0; ci < nchunks; ++ci) {
            if (ci + PFA < nchunks) issue(ci + PFA);            // refills the stage this warp read in the previous iteration
            cp_async_commit();
            cp_async_wait<PFA>();
            __syncwarp();
            const uint32_t g = gc0 + ci, st = g % NST;
            const float4* row4 = reinterpret_cast<const float4*>(pp.aring + (g % NSA) * A_STAGE + tid * A_PITCH);
            uint32_t hi[32], lo[32];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 v = row4[j];
                const float x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    hi[4 * j + q] = __float_as_uint(x[q]);
                    lo[4 * j + q] = __float_as_uint(x[q] - __uint_as_float(__float_as_uint(x[q]) & 0xffffe000u));
                }
            }
            if (g >= NST) mbar_wait(&pp.mma_done[st], ((g / NST) - 1) & 1);     // the MMAs that read this TMEM stage have completed
            tc_fence_after();
            const uint32_t ta = pp.tmem + (static_cast<uint32_t>(warp * 32) << 16) + TMEM_A0 + st * TMEM_A_STAGE;
            tmem_st_32x32(ta, hi);
            tmem_st_32x32(ta + 32, lo);
            tc_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&pp.ready[st]);
        }
        cp_async_wait<0>();
    } else {
        const int wt = tid - 128;                     // 0..127
        auto issue = [&](int ci) {                    // weights are stored tile-major and pre-swizzled: one bulk copy per tile
            const uint32_t g = gc0 + ci, st = g % NST;
            if (g >= NST) mbar_wait(&pp.mma_done[st], ((g / NST) - 1) & 1);     // the MMAs that read this stage have completed
            const int kg = kbase + ci * BK;
            const int wt_floats = bn * BK;            // tiles are stored [n_tile][k_chunk][bn x 32], pre-swizzled
            mbar_arrive_expect_tx(&pp.w_full[st], wt_floats * 4);
            bulk_g2s(pp.ring + st * STAGE, op.W + (static_cast<long long>(n_tile) * op.kchunks + (kg >> 5)) * wt_floats, wt_floats * 4,
                     &pp.w_full[st]);
        };
        if (wt == 0)
            for (int s = 0; s < PF; ++s)
                if (s < nchunks) issue(s);
        for (int ci = 0; ci < nchunks; ++ci) {
            if (wt == 0 && ci + PF < nchunks) issue(ci + PF);
            const uint32_t g = gc0 + ci, st = g % NST;
            mbar_wait(&pp.w_full[st], (g / NST) & 1);
#pragma unroll
            for (int half = 0; half < bn / 64; ++half) {         // 512 16-byte pieces per 64 weight rows, 4 per thread
                const uint4* h4 = reinterpret_cast<const uint4*>(pp.ring + st * STAGE + half * W_TILE);
                float4* l4 = reinterpret_cast<float4*>(pp.ring + st * STAGE + W_PLANE + half * W_TILE);
                uint4 x[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) x[i] = h4[wt + i * 128];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    float4 l;
                    l.x = __uint_as_float(x[i].x) - __uint_as_float(x[i].x & 0xffffe000u);
                    l.y = __uint_as_float(x[i].y) - __uint_as_float(x[i].y & 0xffffe000u);
                    l.z = __uint_as_float(x[i].z) - __uint_as_float(x[i].z & 0xffffe000u);
                    l.w = __uint_as_float(x[i].w) - __uint_as_float(x[i].w & 0xffffe000u);
                    l4[wt + i * 128] = l;
                }
            }
            fence_proxy_async_smem();        // generic-proxy writes -> visible to the tensor core's async proxy
            __syncwarp();
            if (lane == 0) mbar_arrive(&pp.ready[st]);
        }
    }
    {
        const uint32_t g = gc0 + nchunks - 1;              // the last commit covers every MMA of the job
        mbar_wait(&pp.mma_done[g % NST], (g / NST) & 1);
        tc_fence_after();
    }
    pp.gc = gc0 + nchunks;
    pp.jobs += 1;

    // epilogue: warp w reads TMEM lanes (w % 4) * 32 .. + 32 (= tile rows), columns (w / 4) * (bn / 2) .. + bn / 2
    const int r = m0 + (warp & 3) * 32 + lane;
    const uint32_t tl = pp.tmem + (static_cast<uint32_t>((warp & 3) * 32) << 16) + static_cast<uint32_t>((warp >> 2) * (bn >> 1));
    uint32_t vraw[32];
    if constexpr (bn == 128) {       // split-K partial sums only: two 32-column reads per warp
        const int nb = n0 + (warp >> 2) * 64;
        uint32_t vraw2[32];
        tmem_ld_32x32(tl, vraw);
        tmem_ld_32x32(tl + 32, vraw2);
        tc_wait_ld();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(pp.acc_free);
        if (r < rows) {
            float4* dst = reinterpret_cast<float4*>(op.out + (static_cast<long long>(split) * rows + r) * op.N + nb);
#pragma unroll
            for (int j = 0; j < 8; ++j)
                __stcg(dst + j, make_float4(__uint_as_float(vraw[4 * j]), __uint_as_float(vraw[4 * j + 1]), __uint_as_float(vraw[4 * j + 2]),
                                            __uint_as_float(vraw[4 * j + 3])));
#pragma unroll
            for (int j = 0; j < 8; ++j)
                __stcg(dst + 8 + j, make_float4(__uint_as_float(vraw2[4 * j]), __uint_as_float(vraw2[4 * j + 1]),
                                                __uint_as_float(vraw2[4 * j + 2]), __uint_as_float(vraw2[4 * j + 3])));
        }
        return;
    } else {
    const int nb = n0 + (warp >> 2) * 32;
    tmem_ld_32x32(tl, vraw);
    tc_wait_ld();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(pp.acc_free);     // TMEM may be overwritten by the next job (the ring is free: its MMAs completed)
    if (op.epi == LT_PARTIAL) {
        if (r < rows) {
            float4* dst = reinterpret_cast<float4*>(op.out + (static_cast<long long>(split) * rows + r) * op.N + nb);
#pragma unroll
            for (int j = 0; j < 8; ++j)
                __stcg(dst + j, make_float4(__uint_as_float(vraw[4 * j]), __uint_as_float(vraw[4 * j + 1]), __uint_as_float(vraw[4 * j + 2]),
                                            __uint_as_float(vraw[4 * j + 3])));
        }
        return;
    }
    if (r >= rows) return;
    // direct epilogues: every bias read here is a constant of the call (read-only path, 16-byte loads)
    const float4* brow = reinterpret_cast<const float4*>(bias_row(op, r, cx) + nb);
    float v[32];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float4 b4 = __ldg(brow + j);
        v[4 * j] = __uint_as_float(vraw[4 * j]) + b4.x; v[4 * j + 1] = __uint_as_float(vraw[4 * j + 1]) + b4.y;
        v[4 * j + 2] = __uint_as_float(vraw[4 * j + 2]) + b4.z; v[4 * j + 3] = __uint_as_float(vraw[4 * j + 3]) + b4.w;
    }
    if (op.epi == LT_BIAS_RELU) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
    } else if (op.epi == LT_BIAS_SILU) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = v[j] / (1.f + expf(-v[j]));
    }
    // No program emits LT_FINAL any more (the tail phase runs the sampler update), but without this epilogue ptxas spills the
    // phase loop's state of latent_mk_kernel (56 bytes at the 168-register cap), so it stays.
    if (op.epi != LT_FINAL) {
        float4* dst = reinterpret_cast<float4*>(op.out + static_cast<long long>(r) * op.ldo + nb);
#pragma unroll
        for (int j = 0; j < 8; ++j) __stcg(dst + j, make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
        return;
    }
    // LT_FINAL: eps = output.2(...) ; z0 = (z - n*eps)/s ; z <- s_next*z0 + n_next*eps + cz*noise
    // (diffusion.py:586-606, 637-645), or eps_out <- eps in forward mode
    const long long i0 = static_cast<long long>(r) * c.D + nb;
    if (cx.forward) {
        float4* dst = reinterpret_cast<float4*>(c.eps_out + i0);
#pragma unroll
        for (int j = 0; j < 8; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        return;
    }
    const int srows = c.sched_rows > 1 ? c.sched_rows : 1;
    const float* sr = c.sched + (static_cast<long long>(cx.step) * srows + (srows > 1 ? r : 0)) * kSchedRow;
    const float nr = sr[0], sg = sr[1], s2 = sr[2], n2 = sr[3], cz = sr[4];
    float zt[32];
    {
        const float4* z4 = reinterpret_cast<const float4*>(c.z + i0);      // all loads first: one L2 round trip, not 32
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float4 t4 = __ldcg(z4 + j);
            zt[4 * j] = t4.x; zt[4 * j + 1] = t4.y; zt[4 * j + 2] = t4.z; zt[4 * j + 3] = t4.w;
        }
    }
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        const float e = v[j];
        const float z0 = __fdiv_rn(__fsub_rn(zt[j], __fmul_rn(nr, e)), sg);
        zt[j] = __fadd_rn(__fmul_rn(s2, z0), __fmul_rn(n2, e));
    }
    if (cz != 0.f) {
        if (c.noise) {
            const float4* n4 = reinterpret_cast<const float4*>(c.noise + static_cast<long long>(cx.step) * c.noise_step_stride + i0);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 w4 = __ldg(n4 + j);
                zt[4 * j] = __fadd_rn(zt[4 * j], __fmul_rn(cz, w4.x)); zt[4 * j + 1] = __fadd_rn(zt[4 * j + 1], __fmul_rn(cz, w4.y));
                zt[4 * j + 2] = __fadd_rn(zt[4 * j + 2], __fmul_rn(cz, w4.z)); zt[4 * j + 3] = __fadd_rn(zt[4 * j + 3], __fmul_rn(cz, w4.w));
            }
        } else {
#pragma unroll 1
            for (int j4 = 0; j4 < 8; ++j4) {
                float w[4], w1, w2;
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    philox_normal3(c.seed, c.sample_offset + r, static_cast<uint32_t>(cx.step), static_cast<uint32_t>(nb + 4 * j4 + q), w[q], w1,
                                   w2);
                // zt[] is indexed statically below (registers): select the quad with a switch-free unrolled compare
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (j == j4) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) zt[4 * j + q] = __fadd_rn(zt[4 * j + q], __fmul_rn(cz, w[q]));
                    }
            }
        }
    }
    {
        float4* z4 = reinterpret_cast<float4*>(c.z + i0);
#pragma unroll
        for (int j = 0; j < 8; ++j) __stcg(z4 + j, make_float4(zt[4 * j], zt[4 * j + 1], zt[4 * j + 2], zt[4 * j + 3]));
    }
    }   // BN_ == 64
}

// y[row, group] <- relu(GroupNorm(bias + sum_s partial[s])) with the statistics of nn.GroupNorm(8, C) on [B, C]
// (biased variance, eps 1e-5).  One warp per (row, group); a lane owns elements lane + 32 j, j < J, and FIRST issues all of its
// J * KS (<= 32) partial-sum loads, so a phase costs one L2 round trip; the sum over splits keeps the fixed order 0..nsplit-1.
template <int KS, int J>
__device__ __forceinline__ void norm_rows(const LtOp& op, const LatentCall& c, const StepCtx& cx, int rows) {
    const int lane = threadIdx.x & 31;
    const int nwarps = gridDim.x * (blockDim.x >> 5);
    const int G = op.C >> 3, nsplit = op.nsplit;
    const long long plane = static_cast<long long>(rows) * op.C;
    for (int wi = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); wi < rows * 8; wi += nwarps) {
        const int b = wi >> 3, grp = wi & 7;
        const float* brow = bias_row(op, b, cx) + grp * G;
        const float* prow = op.partial + static_cast<long long>(b) * op.C + grp * G;
        float* out = (op.out ? op.out : c.eps_out) + static_cast<long long>(b) * op.ldo + grp * G;
        float p[J][KS], v[J], gam[J], bet[J];
#pragma unroll
        for (int j = 0; j < J; ++j) {
            const int i = lane + 32 * j;
#pragma unroll
            for (int sp = 0; sp < KS; ++sp) p[j][sp] = (i < G && sp < nsplit) ? __ldcg(prow + sp * plane + i) : 0.f;
            v[j] = i < G ? __ldcg(brow + i) : 0.f;
            gam[j] = i < G ? __ldg(op.gamma + grp * G + i) : 0.f;
            bet[j] = i < G ? __ldg(op.beta + grp * G + i) : 0.f;
        }
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < J; ++j) {
#pragma unroll
            for (int sp = 0; sp < KS; ++sp)
                if (sp < nsplit) v[j] += p[j][sp];
            if (lane + 32 * j < G) s += v[j];
        }
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        const float mean = s / static_cast<float>(G);
        float q = 0.f;
#pragma unroll
        for (int j = 0; j < J; ++j)
            if (lane + 32 * j < G) { const float d = v[j] - mean; q = fmaf(d, d, q); }
        for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
        const float rstd = rsqrtf(q / static_cast<float>(G) + 1e-5f);
#pragma unroll
        for (int j = 0; j < J; ++j)
            if (lane + 32 * j < G) __stcg(out + lane + 32 * j, fmaxf((v[j] - mean) * rstd * gam[j] + bet[j], 0.f));
    }
}

// no GroupNorm (SimplePointNetVAE.decode layers): out = act(bias + sum_s partial[s]), elementwise, fixed order
__device__ void reduce_phase(const LtOp& op, const LatentCall& c, const StepCtx& cx, int rows) {
    const long long n4 = static_cast<long long>(rows) * op.C / 4, plane4 = n4;
    const float4* part = reinterpret_cast<const float4*>(op.partial);
    float4* out = reinterpret_cast<float4*>(op.out ? op.out : c.eps_out);
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int col = static_cast<int>((i * 4) % op.C);
        float4 a = __ldg(reinterpret_cast<const float4*>(op.bias + col));
        for (int sp = 0; sp < op.nsplit; ++sp) {
            const float4 t = __ldcg(part + sp * plane4 + i);
            a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w;
        }
        if (op.act) { a.x = fmaxf(a.x, 0.f); a.y = fmaxf(a.y, 0.f); a.z = fmaxf(a.z, 0.f); a.w = fmaxf(a.w, 0.f); }
        __stcg(out + i, a);
    }
}

__device__ void norm_phase(const LtOp& op, const LatentCall& c, const StepCtx& cx, int rows) {
    if (op.gamma == nullptr) { reduce_phase(op, c, cx, rows); return; }
    // the workspace rule of pick_ks (ks * N <= 16384) gives ks * (G / 32) <= 64
    const int jn = (op.C >> 3) + 31 >> 5;          // elements per lane; smallest sufficient instantiation (predicated slots cost)
    if (op.nsplit <= 2) norm_rows<2, 16>(op, c, cx, rows);
    else if (op.nsplit <= 4) { if (jn <= 8) norm_rows<4, 8>(op, c, cx, rows); else norm_rows<4, 16>(op, c, cx, rows); }
    else if (op.nsplit <= 8) { if (jn <= 4) norm_rows<8, 4>(op, c, cx, rows); else norm_rows<8, 8>(op, c, cx, rows); }
    else { if (jn <= 2) norm_rows<16, 2>(op, c, cx, rows); else norm_rows<16, 4>(op, c, cx, rows); }
}

// one element of the sampler update (the LT_FINAL epilogue, element-wise): eps -> z_{t-1} in place, or eps_out in forward mode
__device__ __forceinline__ void final_update_one(const LatentCall& c, const StepCtx& cx, int r, int col, float e) {
    const long long i = static_cast<long long>(r) * c.D + col;
    if (cx.forward) { c.eps_out[i] = e; return; }
    const int srows = c.sched_rows > 1 ? c.sched_rows : 1;
    const float* sr = c.sched + (static_cast<long long>(cx.step) * srows + (srows > 1 ? r : 0)) * kSchedRow;
    const float nr = sr[0], sg = sr[1], s2 = sr[2], n2 = sr[3], cz = sr[4];
    float zt = __ldcg(c.z + i);
    const float z0 = __fdiv_rn(__fsub_rn(zt, __fmul_rn(nr, e)), sg);
    zt = __fadd_rn(__fmul_rn(s2, z0), __fmul_rn(n2, e));
    if (cz != 0.f) {
        float w, w1, w2;
        if (c.noise) w = __ldg(c.noise + static_cast<long long>(cx.step) * c.noise_step_stride + i);
        else philox_normal3(c.seed, c.sample_offset + r, static_cast<uint32_t>(cx.step), static_cast<uint32_t>(col), w, w1, w2);
        zt = __fadd_rn(zt, __fmul_rn(cz, w));
    }
    __stcg(c.z + i, zt);
}

// LT_TAIL: for small batches the last three phases (dec1's GroupNorm, output.0, output.2 + sampler update: networks.py:1083-1086,
// diffusion.py:586-606 / 637-645) are 49 k MACs per row behind three grid barriers and two tile-job pipelines that have nothing
// to chew on (2 and 4 busy CTAs, 8 and 10 us at batch 128).  Rows are independent here, so ONE phase does them on CUDA cores, a few rows per CTA:
// dec1 itself (a 384 x 128 matrix-vector product) + GroupNorm(8, 128) + ReLU, a 128 x 128 and a 128 x 256 matrix-vector product against transposed
// weights (coalesced, L2-resident, 192 KB) with 8 independent accumulators per thread, then the update.  fp32 FMAs throughout.
// RT rows per CTA pass share every weight load (RT = ceil(rows / grid) rounded up to 1, 2 or 4); a row's own arithmetic -- order of
// every sum included -- does not depend on RT or on which rows it is grouped with, so results stay batch independent.
// Both matrix-vector products split K over thread groups and read the transposed weights as float4 (a warp reads 512 contiguous
// bytes; a thread has 16 / 32 INDEPENDENT 16-byte loads in flight instead of a chain of 64 / 128 scalar ones -- the phase is a chain
// of L2 latencies, not of FMAs), then reduce the K groups in a fixed order through shared memory.
template <int RT>
__device__ void tail_rows(const LtOp& op, const LatentCall& c, const StepCtx& cx, int rows, float (*sh_h)[128], float (*sh_a)[128],
                          float* sh_p /* [8][RT][128] or [4][RT][256] */, float* sx /* [RT][384], the idle tile-job ring */) {
    const int tid = threadIdx.x;
    for (int r0 = blockIdx.x * RT; r0 < rows; r0 += gridDim.x * RT) {
        // dec1 = Linear(cat([d2, refine1(z1)])) (W = composed weights [384][128]^T)
        for (int i = tid; i < RT * 96; i += NTHREADS) {
            const int rr = i / 96, q = i - rr * 96, r = r0 + rr;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < rows)
                v = q < 64 ? __ldcg(reinterpret_cast<const float4*>(op.A0 + static_cast<long long>(r) * 256) + q)
                           : __ldcg(reinterpret_cast<const float4*>(op.A1 + static_cast<long long>(r) * 128) + (q - 64));
            reinterpret_cast<float4*>(sx)[i] = v;
        }
        __syncthreads();
        if (tid < 256) {                                     // thread = (k group of 48, four outputs)
            const int og = tid & 31, kg = tid >> 5;
            const float4* w = reinterpret_cast<const float4*>(op.W + static_cast<long long>(kg * 48) * 128) + og;
            float4 acc[RT];
#pragma unroll
            for (int i = 0; i < RT; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int kh = 0; kh < 3; ++kh) {
                float4 wv[16];
#pragma unroll
                for (int k = 0; k < 16; ++k) wv[k] = __ldg(w + (kh * 16 + k) * 32);
#pragma unroll
                for (int i = 0; i < RT; ++i)
#pragma unroll
                    for (int k = 0; k < 16; ++k) {
                        const float x = sx[i * 384 + kg * 48 + kh * 16 + k];
                        acc[i].x = fmaf(wv[k].x, x, acc[i].x); acc[i].y = fmaf(wv[k].y, x, acc[i].y);
                        acc[i].z = fmaf(wv[k].z, x, acc[i].z); acc[i].w = fmaf(wv[k].w, x, acc[i].w);
                    }
            }
#pragma unroll
            for (int i = 0; i < RT; ++i) *reinterpret_cast<float4*>(sh_p + (kg * RT + i) * 128 + 4 * og) = acc[i];
        }
        __syncthreads();
        if (tid < 128) {
#pragma unroll
            for (int i = 0; i < RT; ++i) {
                const int r = r0 + i;
                float v = __ldg(bias_row(op, r < rows ? r : 0, cx) + tid);
#pragma unroll
                for (int kg = 0; kg < 8; ++kg) v += sh_p[(kg * RT + i) * 128 + tid];          // fixed order
                float s1 = v;                                    // GroupNorm(8, 128): 16 consecutive channels = half a warp
#pragma unroll
                for (int o = 8; o; o >>= 1) s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                const float mean = s1 * (1.f / 16.f), d = v - mean;
                float q = d * d;
#pragma unroll
                for (int o = 8; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
                const float rstd = rsqrtf(q * (1.f / 16.f) + 1e-5f);
                sh_h[i][tid] = fmaxf(d * rstd * __ldg(op.gamma + tid) + __ldg(op.beta + tid), 0.f);
            }
        }
        __syncthreads();
        if (tid < 256) {                                     // output.0: thread = (k group of 16, four outputs)
            const int og = tid & 31, kg = tid >> 5;
            const float4* w = reinterpret_cast<const float4*>(op.W2 + static_cast<long long>(kg * 16) * 128) + og;
            float4 wv[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) wv[k] = __ldg(w + k * 32);
#pragma unroll
            for (int i = 0; i < RT; ++i) {
                float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const float x = sh_h[i][kg * 16 + k];
                    a.x = fmaf(wv[k].x, x, a.x); a.y = fmaf(wv[k].y, x, a.y); a.z = fmaf(wv[k].z, x, a.z); a.w = fmaf(wv[k].w, x, a.w);
                }
                *reinterpret_cast<float4*>(sh_p + (kg * RT + i) * 128 + 4 * og) = a;
            }
        }
        __syncthreads();
        if (tid < 128) {
#pragma unroll
            for (int i = 0; i < RT; ++i) {
                float v = __ldg(op.b2 + tid);
#pragma unroll
                for (int kg = 0; kg < 8; ++kg) v += sh_p[(kg * RT + i) * 128 + tid];        // fixed order
                sh_a[i][tid] = fmaxf(v, 0.f);
            }
        }
        __syncthreads();
        if (tid < 256) {                                     // output.2: thread = (k group of 32, four outputs)
            const int og = tid & 63, kg = tid >> 6;
            const float4* w = reinterpret_cast<const float4*>(op.W3 + static_cast<long long>(kg * 32) * 256) + og;
            float4 acc[RT];
#pragma unroll
            for (int i = 0; i < RT; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int kh = 0; kh < 2; ++kh) {
                float4 wv[16];
#pragma unroll
                for (int k = 0; k < 16; ++k) wv[k] = __ldg(w + (kh * 16 + k) * 64);
#pragma unroll
                for (int i = 0; i < RT; ++i)
#pragma unroll
                    for (int k = 0; k < 16; ++k) {
                        const float x = sh_a[i][kg * 32 + kh * 16 + k];
                        acc[i].x = fmaf(wv[k].x, x, acc[i].x); acc[i].y = fmaf(wv[k].y, x, acc[i].y);
                        acc[i].z = fmaf(wv[k].z, x, acc[i].z); acc[i].w = fmaf(wv[k].w, x, acc[i].w);
                    }
            }
#pragma unroll
            for (int i = 0; i < RT; ++i) *reinterpret_cast<float4*>(sh_p + (kg * RT + i) * 256 + 4 * og) = acc[i];
        }
        __syncthreads();
        if (tid < 256) {
            const float b3 = __ldg(op.b3 + tid);
#pragma unroll
            for (int i = 0; i < RT; ++i) {
                float e = b3;
#pragma unroll
                for (int kg = 0; kg < 4; ++kg) e += sh_p[(kg * RT + i) * 256 + tid];          // fixed order
                if (r0 + i < rows) final_update_one(c, cx, r0 + i, tid, e);
            }
        }
        __syncthreads();
    }
}

__device__ void tail_phase(const LtOp& op, const LatentCall& c, const StepCtx& cx, int rows, float* scratch) {
    __shared__ float sh_h[4][128], sh_a[4][128];
    __shared__ __align__(16) float sh_p[4 * 4 * 256];
    const int per = (rows + gridDim.x - 1) / gridDim.x;
    if (per <= 1) tail_rows<1>(op, c, cx, rows, sh_h, sh_a, sh_p, scratch);
    else if (per <= 2) tail_rows<2>(op, c, cx, rows, sh_h, sh_a, sh_p, scratch);
    else tail_rows<4>(op, c, cx, rows, sh_h, sh_a, sh_p, scratch);
}

// LT_HEAD: enc1 and enc2 (Linear + GroupNorm(8) + ReLU each, networks.py:984-993, 1068-1070; 64 k MACs per row) were four phases
// behind four grid barriers with 8 busy CTAs in the GEMM ones (6.1 + 3.4 + 6.1 + 3.8 us in the round-1 trace).  Rows are independent
// up to here, so ONE phase does both layers on CUDA cores, a few rows per CTA, exactly like the tail: transposed fp32 weights read as
// float4 with K split over thread groups (16 independent 16-byte loads in flight per thread and batch), fixed-order reductions through
// shared memory (the tile-job rings are idle in this phase and serve as scratch), GroupNorm by warp shuffles.  A row's arithmetic
// does not depend on RT or on the rows it shares a CTA with.
template <int RT>
__device__ void head_rows(const LtOp& op, const LatentCall& c, const StepCtx& cx, int rows, float* scratch) {
    float* sx = scratch;                     // [RT][256] input rows
    float* sh1 = sx + RT * 256;              // [RT][128] enc1 output
    float* sp = sh1 + RT * 128;              // partial sums: [8][RT][128] then [4][RT][256]
    const int tid = threadIdx.x;
    for (int r0 = blockIdx.x * RT; r0 < rows; r0 += gridDim.x * RT) {
        const int og1 = tid & 31, kg1 = tid >> 5;          // enc1: thread = (k group of 32, four outputs), tid < 256
        const float4* w1 = reinterpret_cast<const float4*>(op.W2 + static_cast<long long>(kg1 * 32) * 128) + og1;
        for (int i = tid; i < RT * 64; i += NTHREADS) {
            const int rr = i >> 6, r = r0 + rr;
            reinterpret_cast<float4*>(sx)[i] = r < rows ? __ldcg(reinterpret_cast<const float4*>(c.z + static_cast<long long>(r) * 256) + (i & 63))
                                                        : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        __syncthreads();
        if (tid < 256) {
            float4 acc[RT];
#pragma unroll
            for (int i = 0; i < RT; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int kh = 0; kh < 2; ++kh) {
                float4 wv[16];
#pragma unroll
                for (int k = 0; k < 16; ++k) wv[k] = __ldg(w1 + (kh * 16 + k) * 32);
#pragma unroll
                for (int i = 0; i < RT; ++i)
#pragma unroll
                    for (int k = 0; k < 16; ++k) {
                        const float x = sx[i * 256 + kg1 * 32 + kh * 16 + k];
                        acc[i].x = fmaf(wv[k].x, x, acc[i].x); acc[i].y = fmaf(wv[k].y, x, acc[i].y);
                        acc[i].z = fmaf(wv[k].z, x, acc[i].z); acc[i].w = fmaf(wv[k].w, x, acc[i].w);
                    }
            }
#pragma unroll
            for (int i = 0; i < RT; ++i) *reinterpret_cast<float4*>(sp + (kg1 * RT + i) * 128 + 4 * og1) = acc[i];
        }
        const int og2 = tid & 63, kg2 = tid >> 6;          // enc2: thread = (k group of 32, four outputs), tid < 256
        const float4* w2 = reinterpret_cast<const float4*>(op.W3 + static_cast<long long>(kg2 * 32) * 256) + og2;
        __syncthreads();
        if (tid < 128) {
#pragma unroll
            for (int i = 0; i < RT; ++i) {
                const int r = r0 + i;
                float v = r < rows ? __ldcg(bias_row(op, r, cx) + tid) : 0.f;
#pragma unroll
                for (int kg = 0; kg < 8; ++kg) v += sp[(kg * RT + i) * 128 + tid];          // fixed order
                float s1 = v;                                    // GroupNorm(8, 128): 16 consecutive channels = half a warp
#pragma unroll
                for (int o = 8; o; o >>= 1) s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                const float mean = s1 * (1.f / 16.f), d = v - mean;
                float q = d * d;
#pragma unroll
                for (int o = 8; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
                const float rstd = rsqrtf(q * (1.f / 16.f) + 1e-5f);
                const float hh = fmaxf(d * rstd * __ldg(op.gamma + tid) + __ldg(op.beta + tid), 0.f);
                sh1[i * 128 + tid] = hh;
                if (r < rows) __stcg(op.out + static_cast<long long>(r) * 128 + tid, hh);
            }
        }
        __syncthreads();
        if (tid < 256) {
            float4 acc[RT];
#pragma unroll
            for (int i = 0; i < RT; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int kh = 0; kh < 2; ++kh) {
                float4 wv[16];
#pragma unroll
                for (int k = 0; k < 16; ++k) wv[k] = __ldg(w2 + (kh * 16 + k) * 64);
#pragma unroll
                for (int i = 0; i < RT; ++i)
#pragma unroll
                    for (int k = 0; k < 16; ++k) {
                        const float x = sh1[i * 128 + kg2 * 32 + kh * 16 + k];
                        acc[i].x = fmaf(wv[k].x, x, acc[i].x); acc[i].y = fmaf(wv[k].y, x, acc[i].y);
                        acc[i].z = fmaf(wv[k].z, x, acc[i].z); acc[i].w = fmaf(wv[k].w, x, acc[i].w);
                    }
            }
#pragma unroll
            for (int i = 0; i < RT; ++i) *reinterpret_cast<float4*>(sp + (kg2 * RT + i) * 256 + 4 * og2) = acc[i];
        }
        __syncthreads();
        if (tid < 256) {
            const float b = __ldg(op.b3 + tid), ga = __ldg(op.gamma2 + tid), be = __ldg(op.beta2 + tid);
#pragma unroll
            for (int i = 0; i < RT; ++i) {
                float v = b;
#pragma unroll
                for (int kg = 0; kg < 4; ++kg) v += sp[(kg * RT + i) * 256 + tid];          // fixed order
                float s1 = v;                                    // GroupNorm(8, 256): 32 consecutive channels = one warp
#pragma unroll
                for (int o = 16; o; o >>= 1) s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                const float mean = s1 * (1.f / 32.f), d = v - mean;
                float q = d * d;
#pragma unroll
                for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
                const float rstd = rsqrtf(q * (1.f / 32.f) + 1e-5f);
                if (r0 + i < rows) __stcg(op.out2 + static_cast<long long>(r0 + i) * 256 + tid, fmaxf(d * rstd * ga + be, 0.f));
            }
        }
        __syncthreads();
    }
}

__device__ void head_phase(const LtOp& op, const LatentCall& c, const StepCtx& cx, int rows, float* scratch) {
    const int per = (rows + gridDim.x - 1) / gridDim.x;
    if (per <= 1) head_rows<1>(op, c, cx, rows, scratch);
    else if (per <= 2) head_rows<2>(op, c, cx, rows, scratch);
    else head_rows<4>(op, c, cx, rows, scratch);
}

// sinusoidal timestep embedding (networks.py:1088-1106): emb[r] = [sin(t_r f_j), cos(t_r f_j)], one row per time row
__device__ void emb_phase(const LtOp& op, const LatentCall& c, const StepCtx& cx, int rows) {
    const long long n = static_cast<long long>(rows) * 256;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int r = static_cast<int>(i >> 8), j = static_cast<int>(i & 255);
        // t is the same for every sample of a step (all samplers), also with per-sample schedule rows: row 0 of the step
        const float tt = cx.forward ? c.t_in[r] : c.sched[static_cast<long long>(r) * (c.sched_rows > 1 ? c.sched_rows : 1) * kSchedRow + 5];
        const float a = tt * __ldg(op.bias + (j & 127));     // op.bias = frequency table [128]
        __stcg(op.out + i, j < 128 ? sinf(a) : cosf(a));
    }
}

__device__ void run_op(const LtOp& op, const LatentCall& c, const StepCtx& cx, int R, Pipe& pp) {
    const int rows = op.rows_mode ? R : c.B;
    if (op.kind == LT_GEMM) {
        const int m_tiles = (rows + BM - 1) / BM, n_tiles = op.N / op.bn;
        const int items = m_tiles * n_tiles * op.ks;
        if (threadIdx.x >= NWORK) {
            if (threadIdx.x == NWORK)
                for (int it = blockIdx.x; it < items; it += gridDim.x) {
                    if (op.bn == 128) gemm_item_mma<128>(op, pp);
                    else gemm_item_mma<64>(op, pp);
                }
            __syncwarp();
            return;
        }
        for (int it = blockIdx.x; it < items; it += gridDim.x) {
            const int split = it % op.ks, rest = it / op.ks;
            if (op.bn == 128) gemm_item<128>(op, c, cx, rows, rest / n_tiles, rest % n_tiles, split, pp);
            else gemm_item<64>(op, c, cx, rows, rest / n_tiles, rest % n_tiles, split, pp);
        }
    } else if (op.kind == LT_NORM) {
        norm_phase(op, c, cx, rows);
    } else if (op.kind == LT_TAIL) {
        tail_phase(op, c, cx, rows, pp.ring);
    } else if (op.kind == LT_HEAD) {
        head_phase(op, c, cx, rows, pp.ring);
    } else {
        emb_phase(op, c, cx, rows);
    }
}

}  // namespace

__global__ void __launch_bounds__(NTHREADS, 1) latent_mk_kernel(const LtProgram* __restrict__ prog, const LatentCall* __restrict__ callp,
                                                           int S, int R, int forward, unsigned* bar,
                                                           unsigned long long* trace) {
    extern __shared__ __align__(16) unsigned char lt_smem_raw[];
    __shared__ __align__(8) uint64_t mma_done[NST];
    __shared__ __align__(8) uint64_t w_full[NST];
    __shared__ __align__(8) uint64_t ready[NST];
    __shared__ __align__(8) uint64_t acc_free;
    __shared__ uint32_t tmem_slot;
    Pipe pp;
    pp.ring = reinterpret_cast<float*>(lt_smem_raw + ((1024u - (smem_u32(lt_smem_raw) & 1023u)) & 1023u));
    pp.aring = pp.ring + NST * STAGE;
    pp.mma_done = mma_done;
    pp.w_full = w_full;
    pp.ready = ready;
    pp.acc_free = &acc_free;
    pp.jobs = 0;
    pp.gc = 0;
    if (threadIdx.x == 0) {
        for (int i = 0; i < NST; ++i) { mbar_init(&mma_done[i], 1); mbar_init(&w_full[i], 1); mbar_init(&ready[i], NWORK / 32); }
        mbar_init(&acc_free, NWORK / 32);
        fence_mbar_init();
    }
    if ((threadIdx.x >> 5) == 1) { tmem_alloc(&tmem_slot, TMEM_COLS); tmem_relinquish(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    pp.tmem = tmem_slot;

    const LatentCall c = *callp;
    unsigned target = 0;
    StepCtx cx{0, forward};
    const int n_pre = prog->n_pre, n_loop = prog->n_loop;
    // the program is a constant of the launch: keep it in shared memory, so that no phase starts with (and no chunk loop
    // contains) a dependent global load of its own description
    __shared__ LtOp s_ops[40];
    {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(prog->ops);
        uint32_t* dst = reinterpret_cast<uint32_t*>(s_ops);
        const int nw = (n_pre + n_loop) * static_cast<int>(sizeof(LtOp) / 4);
        for (int i = threadIdx.x; i < nw; i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    // ONE call site for run_op (prologue phases and the S x n_loop loop phases walk the same code): the kernel's code is far
    // larger than the instruction cache, so every duplicated inlining costs instruction-fetch misses in every phase
    const int total = n_pre + S * n_loop;
    int step = 0, li = 0;
    for (int it = 0; it < total; ++it) {
        const bool pre = it < n_pre;
        const int oi = pre ? it : n_pre + li;
        cx.step = step;
        // PCD_LT_TRACE: per CTA and phase of the LAST step, globaltimer at phase start / work done / barrier passed
        unsigned long long* tr = (trace && !pre && step == S - 1 && threadIdx.x == 0)
                                     ? trace + (static_cast<long long>(blockIdx.x) * 40 + li) * 3 : nullptr;
        if (tr) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr[0]));
        run_op(s_ops[oi], c, cx, R, pp);
        if (tr) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr[1]));
        grid_sync(bar, target);
        if (tr) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr[2]));
        if (!pre && ++li == n_loop) { li = 0; ++step; }
    }
    tc_fence_before();
    __syncthreads();
    if ((threadIdx.x >> 5) == 1) { tc_fence_after(); tmem_dealloc(pp.tmem, TMEM_COLS); }
}

// C[i][col0 + j] = sum_m Wd[i][col0 + m] * Wr[m][j]  (double accumulation), cbias[i] = bd[i] + sum_m Wd[i][col0 + m] * br[m]:
// decK(cat([prev, refineK(x_k)])) = Wd[:, :col0] prev + (Wd[:, col0:] Wr) x_k + cbias   (networks.py:1080-1083)
__global__ void compose_refine_kernel(const float* __restrict__ Wd, int ldd, int col0, const float* __restrict__ Wr, int kr,
                                      const float* __restrict__ bd, const float* __restrict__ br, float* __restrict__ C,
                                      float* __restrict__ cbias, int cout) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (i >= cout) return;
    const float* wrow = Wd + static_cast<long long>(i) * ldd + col0;
    if (j < kr) {
        double a = 0.0;
        for (int m = 0; m < kr; ++m) a += static_cast<double>(wrow[m]) * static_cast<double>(Wr[static_cast<long long>(m) * kr + j]);
        C[static_cast<long long>(i) * ldd + col0 + j] = static_cast<float>(a);
    }
    if (j == 0) {
        double a = bd[i];
        for (int m = 0; m < kr; ++m) a += static_cast<double>(wrow[m]) * static_cast<double>(br[m]);
        cbias[i] = static_cast<float>(a);
    }
}

// out[n_tile][k_chunk][row][swizzled 32 floats] <- W[n][col0 + k]: the bn x 32 tiles (bn = 64 or 128) the persistent kernel streams, stored
// contiguously (a job's K range is one sequential read) and already in the SWIZZLE_128B shared-memory layout
__global__ void tile_weights_kernel(const float* __restrict__ W, int ldw, int col0, int N, int K, int bn, float* __restrict__ out) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= static_cast<long long>(N) * K) return;
    const int n = static_cast<int>(i / K), k = static_cast<int>(i - static_cast<long long>(n) * K);
    const int nt = n / bn, row = n % bn, kc = k >> 5, kk = k & 31;
    out[(static_cast<long long>(nt) * (K >> 5) + kc) * (bn * BK) + row * BK + ((((kk >> 2) ^ row) & 7) << 2) + (kk & 3)] =
        W[static_cast<long long>(n) * ldw + col0 + k];
}
cudaError_t launch_tile_weights(const float* W, int ldw, int col0, int N, int K, int bn, float* out, cudaStream_t s) {
    const long long n = static_cast<long long>(N) * K;
    tile_weights_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(W, ldw, col0, N, K, bn, out);
    return cudaGetLastError();
}

cudaError_t launch_compose_refine(const float* Wd, int ldd, int col0, const float* Wr, int kr, const float* bd, const float* br,
                                  float* C, float* cbias, int cout, cudaStream_t s) {
    dim3 grid((kr + 127) / 128, cout);
    compose_refine_kernel<<<grid, 128, 0, s>>>(Wd, ldd, col0, Wr, kr, bd, br, C, cbias, cout);
    return cudaGetLastError();
}

static constexpr int kLtSmemBytes = (NST * STAGE + NSA * A_STAGE) * static_cast<int>(sizeof(float)) + 1024;   // + alignment slack

cudaError_t latent_mk_grid(int num_sms, int* grid_out) {
    cudaError_t e = cudaFuncSetAttribute(latent_mk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLtSmemBytes);
    if (e != cudaSuccess) return e;
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, latent_mk_kernel, NTHREADS, kLtSmemBytes);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorLaunchOutOfResources;
    *grid_out = num_sms;      // one CTA per SM: every phase is sized for it
    return cudaSuccess;
}

cudaError_t launch_latent_mk(const LtProgram* prog, const LatentCall* call, int S, int R, int forward, unsigned* bar, int grid,
                             cudaStream_t stream) {
    cudaError_t e = cudaMemsetAsync(bar, 0, sizeof(unsigned) * kLtBarrierWords, stream);
    if (e != cudaSuccess) return e;
    unsigned long long* trace = nullptr;
    const char* trace_path = std::getenv("PCD_LT_TRACE");     // debugging aid: synchronous, writes one line per CTA and phase
    if (trace_path) {
        e = cudaMalloc(reinterpret_cast<void**>(&trace), sizeof(unsigned long long) * grid * 40 * 3);
        if (e != cudaSuccess) return e;
        cudaMemset(trace, 0, sizeof(unsigned long long) * grid * 40 * 3);
    }
    void* args[] = {&prog, &call, &S, &R, &forward, &bar, &trace};
    e = cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(latent_mk_kernel), dim3(grid), dim3(NTHREADS), args, kLtSmemBytes, stream);
    if (trace) {
        cudaStreamSynchronize(stream);
        std::vector<unsigned long long> hbuf(static_cast<size_t>(grid) * 40 * 3);
        cudaMemcpy(hbuf.data(), trace, hbuf.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
        cudaFree(trace);
        if (FILE* f = std::fopen(trace_path, "w")) {
            for (int b = 0; b < grid; ++b)
                for (int i = 0; i < 40; ++i) {
                    const unsigned long long* t = &hbuf[(static_cast<size_t>(b) * 40 + i) * 3];
                    if (t[0]) std::fprintf(f, "%d %d %llu %llu %llu\n", b, i, t[0], t[1], t[2]);
                }
            std::fclose(f);
        }
    }
    return e;
}

}  // namespace pcd
