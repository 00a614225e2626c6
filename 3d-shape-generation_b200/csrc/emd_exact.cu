// Exact EMD of the reference (metrics.py:49-92, `earth_mover_distance_cpu`: SciPy linear_sum_assignment on the Euclidean
// distance matrix of the two cube-normalised clouds, matched sum / 3) as a batched auction with epsilon scaling (Bertsekas),
// one CTA per cloud pair.
//
//   * Integer costs: c_ij = rint(d_ij * 2^22) with d_ij the fp32 direct-difference distance of the Chamfer kernels.  After cube
//     normalisation d <= 2 sqrt(3), so c < 2^24.  The auction runs on costs scaled by (n + 1) down to eps = 1, which makes the
//     final assignment optimal for the quantised problem (eps < 1/n in unscaled units).  The matched sum differs from the fp64
//     optimum by at most n / 2^22 absolute.
//   * Rectangular pairs are padded to n = max(N, M) with dummy rows / columns of cost 0; they absorb the unmatched points.
//   * Costs are recomputed from the clouds on every scan, never stored.  Shared memory per CTA (n = max(N, M)):
//       y float4 [n] | price int64 [n] | bid key uint64 [n] | owner int32 [n] | assigned object int32 [n] | bidder list int32 [n]
//     = 44 n bytes: 88 KB at n = 2048 (two CTAs per SM), 176 KB at n = 4096 (one CTA per SM).
//   * Jacobi rounds: every unassigned person (one warp each) bids against the same prices; each object takes the highest bid
//     through a shared atomicMax on the packed key (bid << 13 | 8191 - person), so the result does not depend on the order in
//     which warps run: the same input gives the same assignment and the same bits, and no quantity spans the batch.
//   * No hang: a pair with a non-finite normalised coordinate (a cloud of equal points divides by 0) is skipped and gets NaN; every
//     eps phase stops after a round cap derived from the eps schedule and sets *err instead of spinning.
#include <cstdint>
#include <cuda_runtime.h>

namespace pcd {

constexpr int kExactThreads = 512;
constexpr int kExactWarps = kExactThreads / 32;
constexpr int kExactMaxN = 4096;
constexpr int kExactIdxBits = 13;                       // person index field of a bid key (n <= 4096 < 8192)
constexpr long long kExactTheta = 8;                    // eps divisor between phases
constexpr long long kExactCmax = 14529496;              // > 2 sqrt(3) * 2^22: bound of a quantised cost
constexpr long long kNoSecond = 0x3fffffffffffffffLL;   // "no second-best object" (n == 1)

size_t emd_exact_smem(int n) { return static_cast<size_t>(n) * 44; }

__global__ void __launch_bounds__(kExactThreads, 2) emd_exact_kernel(const float4* __restrict__ X, const float4* __restrict__ Y,
                                                                     int N, int M, double scale, float* __restrict__ emd,
                                                                     int* __restrict__ assign_xy, int* __restrict__ err) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    const int n = max(N, M);
    float4* ys = reinterpret_cast<float4*>(sm_raw);
    long long* price = reinterpret_cast<long long*>(ys + n);
    unsigned long long* bidkey = reinterpret_cast<unsigned long long*>(price + n);
    int* owner = reinterpret_cast<int*>(bidkey + n);
    int* assigned = owner + n;
    int* list = assigned + n;
    __shared__ int s_cnt;

    const long long pair = blockIdx.x;
    const float4* x = X + pair * N;
    const float4* y = Y + pair * M;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    int bad = 0;
    for (int j = tid; j < M; j += kExactThreads) {
        const float4 v = y[j];
        bad |= !(isfinite(v.x) && isfinite(v.y) && isfinite(v.z));
        ys[j] = v;
    }
    for (int i = tid; i < N; i += kExactThreads) {
        const float4 v = x[i];
        bad |= !(isfinite(v.x) && isfinite(v.y) && isfinite(v.z));
    }
    for (int j = tid; j < n; j += kExactThreads) { price[j] = 0; bidkey[j] = 0; }
    if (__syncthreads_or(bad)) {
        // normalize_to_cube divided by 0 (all points equal) or the input held NaN / inf: NaN costs would never settle an auction
        if (tid == 0) emd[pair] = __int_as_float(0x7fc00000);
        if (assign_xy)
            for (int i = tid; i < N; i += kExactThreads) assign_xy[pair * N + i] = -1;
        return;
    }

    const long long np1 = n + 1;
    const long long cbound = np1 * kExactCmax;          // every scaled cost lies in [0, cbound)
    long long eps_prev = cbound;                        // zero prices satisfy cbound-complementary slackness with any assignment
    long long eps = cbound / kExactTheta > 1 ? cbound / kExactTheta : 1;
    bool aborted = false;
    for (;;) {
        // Round cap of a phase: a round raises some price by >= eps, and the price rise of a phase is at most
        // n (n - 1) (eps_prev + eps) over all objects (an object's rise is bounded along an alternating path to an object
        // that has not been bid for); 2x margin.
        const long long ratio = (eps_prev + eps - 1) / eps;
        const long long cap = 2LL * n * n * (ratio + 1) + 64;
        for (int j = tid; j < n; j += kExactThreads) { owner[j] = -1; assigned[j] = -1; list[j] = j; }
        __syncthreads();
        int nun = n;
        for (long long round = 0; nun > 0; ++round) {
            if (round >= cap) {                           // uniform: every thread counts the same rounds
                if (tid == 0) atomicExch(err, 1);
                aborted = true;
                break;
            }
            // --- bidding: warp per unassigned person; lanes stride the objects
            for (int k = warp; k < nun; k += kExactWarps) {
                const int i = list[k];
                long long w1 = kNoSecond, w2 = kNoSecond;   // smallest and second smallest scaled cost + price
                int j1 = 0x7fffffff;
                if (i < N) {
                    const float4 xi = x[i];
                    for (int j = lane; j < M; j += 32) {
                        const float4 t = ys[j];
                        const float dx = xi.x - t.x, dy = xi.y - t.y, dz = xi.z - t.z;
                        const float d = sqrtf(fmaf(dz, dz, fmaf(dy, dy, dx * dx)));
                        const long long w = static_cast<long long>(__float2int_rn(d * 4194304.0f)) * np1 + price[j];
                        if (w < w1) { w2 = w1; w1 = w; j1 = j; }
                        else if (w < w2) w2 = w;
                    }
                    for (int j = M + lane; j < n; j += 32) {   // dummy objects: cost 0
                        const long long w = price[j];
                        if (w < w1) { w2 = w1; w1 = w; j1 = j; }
                        else if (w < w2) w2 = w;
                    }
                } else {                                       // dummy person: cost 0 to every object
                    for (int j = lane; j < n; j += 32) {
                        const long long w = price[j];
                        if (w < w1) { w2 = w1; w1 = w; j1 = j; }
                        else if (w < w2) w2 = w;
                    }
                }
                // merge (w1, j1, w2) over the warp; equal values go to the lower object index
#pragma unroll
                for (int o = 16; o; o >>= 1) {
                    const long long b1 = __shfl_xor_sync(0xffffffffu, w1, o);
                    const long long b2 = __shfl_xor_sync(0xffffffffu, w2, o);
                    const int bj = __shfl_xor_sync(0xffffffffu, j1, o);
                    if (b1 < w1 || (b1 == w1 && bj < j1)) { w2 = min(w1, b2); w1 = b1; j1 = bj; }
                    else w2 = min(w2, b1);
                }
                if (lane == 0) {
                    const long long bid = price[j1] + (w2 == kNoSecond ? 0 : w2 - w1) + eps;
                    atomicMax(&bidkey[j1], (static_cast<unsigned long long>(bid) << kExactIdxBits) |
                                               static_cast<unsigned long long>(8191 - i));
                }
            }
            __syncthreads();
            // --- every object with bids goes to its highest bidder; its previous owner becomes unassigned
            if (tid == 0) s_cnt = 0;
            for (int j = tid; j < n; j += kExactThreads) {
                const unsigned long long key = bidkey[j];
                if (key) {
                    bidkey[j] = 0;
                    const int winner = 8191 - static_cast<int>(key & 8191u);
                    const int prev = owner[j];
                    if (prev >= 0) assigned[prev] = -1;      // prev did not bid this round: it owned j
                    owner[j] = winner;
                    assigned[winner] = j;
                    price[j] = static_cast<long long>(key >> kExactIdxBits);
                }
            }
            __syncthreads();
            for (int i = tid; i < n; i += kExactThreads)
                if (assigned[i] < 0) list[atomicAdd(&s_cnt, 1)] = i;
            __syncthreads();
            nun = s_cnt;
        }
        if (aborted || eps == 1) break;
        eps_prev = eps;
        eps = eps / kExactTheta > 1 ? eps / kExactTheta : 1;
    }
    if (aborted) {
        if (tid == 0) emd[pair] = __int_as_float(0x7fc00000);
        if (assign_xy)
            for (int i = tid; i < N; i += kExactThreads) assign_xy[pair * N + i] = -1;
        return;
    }
    // value: fp32 distances of the matched real pairs, summed in fp64 in x-index order
    double* dist = reinterpret_cast<double*>(bidkey);
    for (int i = tid; i < N; i += kExactThreads) {
        const int j = assigned[i];
        double v = 0.0;
        if (j < M) {
            const float4 xi = x[i], t = ys[j];
            const float dx = xi.x - t.x, dy = xi.y - t.y, dz = xi.z - t.z;
            v = static_cast<double>(sqrtf(fmaf(dz, dz, fmaf(dy, dy, dx * dx))));
        }
        dist[i] = v;
        if (assign_xy) assign_xy[pair * N + i] = j < M ? j : -1;
    }
    __syncthreads();
    if (tid == 0) {
        double s = 0.0;
        for (int i = 0; i < N; ++i) s += dist[i];
        emd[pair] = static_cast<float>(s / 3.0 * scale);   // the reference divides by x_pc.shape[1] == 3 (SURVEY C8)
    }
}

bool emd_exact_fits(int N, int M) { return N <= kExactMaxN && M <= kExactMaxN; }

cudaError_t launch_emd_exact(const float4* X, const float4* Y, int pairs, int N, int M, float scaling, float* emd, int* assign_xy,
                             int* err, cudaStream_t s) {
    const size_t smem = emd_exact_smem(N > M ? N : M);
    cudaError_t e = cudaFuncSetAttribute(emd_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(emd_exact_smem(kExactMaxN)));
    if (e != cudaSuccess) return e;
    emd_exact_kernel<<<pairs, kExactThreads, smem, s>>>(X, Y, N, M, static_cast<double>(scaling), emd, assign_xy, err);
    return cudaGetLastError();
}

}  // namespace pcd
