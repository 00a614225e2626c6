// C ABI of the point-VAE encoder: pcd_point_encoder_* (include/pcd_b200.h).
//
// SimplePointNetVAE.encode (networks.py:1110-1156; encode / reparameterize / forward between __init__ and decode at :1219):
//   x [B, N, 3] -> channels-first -> encoder.0..3 = PointNetLayer(3 -> 64 -> 128 -> 256 -> 512), each three times
//   Conv1d(k=1) -> BatchNorm1d (eval) -> ReLU -> encoder.4/5 AdaptiveMaxPool1d(1) + Flatten [B, 512]
//   -> encoder.6/7 Linear(512, 256) + ReLU -> fc_mu, fc_logvar (Linear(256, 256) each)
// * Rows are points, padded per cloud to Npad = ceil(N / 128) * 128 as in the denoiser (api.cu); the two plane layout is the
//   denoiser's too (lo plane M rows below the hi plane of the same 2-D tensor).
// * encoder.0.conv1 (K = 3) is the denoiser's CUDA-core first layer (launch_enc1_first) with one shared folded bias.
// * The other 11 convs run on the tcgen05 GEMM of gemm_tc.cu with BatchNorm folded on the host (fold_conv_bn) and the tile
//   shapes of tc_shape.  There are no skip connections, so two ping-pong buffers [planes * M, 512] hold every activation.
// * encoder.3.conv3 runs the EPI_MAXPOOL epilogue: max over the valid points of a cloud (padded rows masked by n_valid), + bias,
//   ReLU into the zeroed [B, 512] pool, since max_n relu(a_n + b) = relu(max_n a_n + b).  Its [M, 512] output is never written.
// * encoder.6 + ReLU and the two heads (one [512, 256] weight: fc_mu rows, then fc_logvar rows) run on the fp32 CUDA-core GEMM
//   with K splits that do not depend on the batch, so a cloud's latent does not depend on its neighbours.
// * Non-finite clouds: in the reference a NaN (or +-inf) coordinate makes every mu / logvar entry of its cloud NaN (ReLU, max
//   and Linear propagate it), while the shared epilogues' fmaxf drops NaN and would return finite values.  A per-cloud flag
//   computed from x makes the head reduction write NaN for that cloud; rows are independent, so its neighbours do not change.
#include <cmath>
#include <cstring>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include "api_common.h"
#include "pcd_launch.h"
#include "pcd_types.h"

using namespace pcd;

namespace pcd {
cudaError_t launch_rows16_to_f32(const void* hi, const void* lo, int ld, float* out, int c_keep, long long rows, int f16, cudaStream_t s);

// flag[b] = 1 when a coordinate of cloud b is NaN or +-inf (one CTA per cloud)
__global__ void __launch_bounds__(256) point_nonfinite_kernel(const float* __restrict__ x, long long n3, int* __restrict__ flag) {
    const float* xb = x + static_cast<long long>(blockIdx.x) * n3;
    int bad = 0;
    for (long long i = threadIdx.x; i < n3; i += 256) bad |= !isfinite(xb[i]);
    bad = __syncthreads_or(bad);
    if (threadIdx.x == 0) flag[blockIdx.x] = bad;
}

// [mu | logvar][b][c] = bias[c] + sum_s partial[s][b][c] in a fixed order (as splitk_reduce_kernel); NaN for a flagged cloud
__global__ void __launch_bounds__(256) point_heads_reduce_kernel(const float* __restrict__ partial, int nsplit, const float* __restrict__ bias,
                                                                 const int* __restrict__ flag, float* __restrict__ mu,
                                                                 float* __restrict__ logvar, int B, int latent) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long n = static_cast<long long>(B) * 2 * latent;
    if (i >= n) return;
    const int r = static_cast<int>(i / (2 * latent)), c = static_cast<int>(i - static_cast<long long>(r) * 2 * latent);
    float v = bias[c];
    for (int s = 0; s < nsplit; ++s) v += partial[s * n + i];
    if (flag[r]) v = __int_as_float(0x7fc00000);
    if (c < latent) mu[static_cast<long long>(r) * latent + c] = v;
    else logvar[static_cast<long long>(r) * latent + c - latent] = v;
}
}  // namespace pcd

namespace {

constexpr int kHidden = 512;       // hidden_dim: encoder.3's width and the pooled feature
constexpr int kMid = 256;          // encoder.6 output (hidden_dim / 2)
constexpr int kLatent = 256;
constexpr int kConvs = 12;         // encoder.<blk>.conv<j>: index 3 * blk + j - 1
constexpr int kSplits6 = 4;        // encoder.6: K = 512 -> 128 per split, fixed
constexpr int kSplitsHead = 2;     // heads: K = 256 -> 128 per split, fixed
constexpr int kStages = 15;        // flag, 12 convs, encoder.6, heads

struct PLayer {
    int cin = 0, cout = 0;
    void* w16 = nullptr;           // [planes * cout][cin] 16-bit (hi plane, then the residual plane in the split modes)
    float* b = nullptr;            // [cout] folded
};

struct PTcOp {
    int layer = 0, epi = EPI_STORE, np = 1, out_planes = 1;
    TcShape sh;
    CUtensorMap a0, b, o;
    TcGemmParams p{};
};

struct PPlan {
    int B = 0, N = 0, Npad = 0;
    long long M = 0;
    void* T[2] = {nullptr, nullptr};   // ping-pong activations [planes * M][512] 16-bit
    float* pool = nullptr;             // [B][512] encoder.5
    float* hid = nullptr;              // [B][256] encoder.7
    float* part = nullptr;             // split-K partial sums, [kSplits6][B][256] or [kSplitsHead][B][512]
    int* flag = nullptr;               // [B] non-finite cloud
    CallArgs* call = nullptr;          // x for launch_enc1_first
    PTcOp ops[kConvs];                 // ops[1..11]: encoder.0.conv2 .. encoder.3.conv3 + max-pool
    PTcOp tap_last;                    // encoder.3.conv3 as a STORE layer (tap hook only)
    int out_buf[kConvs] = {};          // buffer written by conv l (encoder.3.conv3: by tap_last)
    std::vector<void*> owned;
    ~PPlan() { for (void* p : owned) cudaFree(p); }
};

}  // namespace

struct pcd_point_encoder {
    int precision = 0, device = 0, num_sms = 148, f16 = 0, planes = 1;
    float *Wx = nullptr, *b0 = nullptr;       // encoder.0.conv1 folded: [64][3], [64]
    PLayer L[kConvs];                         // L[0] unused (encoder.0.conv1 runs on CUDA cores)
    float *w6 = nullptr, *b6 = nullptr;       // encoder.6: [256][512], [256]
    float *wh = nullptr, *bh = nullptr;       // fc_mu | fc_logvar: [512][256], [512]
    PlanCache<std::pair<int, int>, PPlan> plans;
    std::vector<void*> owned;
};

template <typename T>
static int pup(pcd_point_encoder* h, const std::vector<T>& v, T** out) {
    void* p = nullptr;
    CU(cudaMalloc(&p, v.size() * sizeof(T)));
    h->owned.push_back(p);
    CU(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    *out = static_cast<T*>(p);
    return 0;
}

static int upload_conv(pcd_point_encoder* h, const HostMat& m, PLayer* L) {
    L->cin = m.k; L->cout = m.cout;
    float* w32 = nullptr;
    if (pup(h, m.w, &w32) || pup(h, m.b, &L->b)) return 1;
    const long long n = static_cast<long long>(m.w.size());
    CU(cudaMalloc(&L->w16, n * 2 * h->planes));
    h->owned.push_back(L->w16);
    if (h->planes == 2) LAUNCH(launch_f32_split_16(w32, L->w16, static_cast<char*>(L->w16) + n * 2, n, h->f16, 0));
    else LAUNCH(launch_f32_to_16(w32, L->w16, n, h->f16, 0));
    return 0;
}

extern "C" int pcd_point_encoder_destroy(pcd_point_encoder* h);

extern "C" int pcd_point_encoder_create(const pcd_named_tensor* tensors, int32_t n_tensors, int32_t precision, int32_t device,
                                        pcd_point_encoder** out) {
    REQ(tensors && out, "null argument");
    REQ(precision == PCD_PRECISION_BF16 || precision == PCD_PRECISION_BF16X3 || precision == PCD_PRECISION_F16 ||
            precision == PCD_PRECISION_F16MIX,
        "pcd_point_encoder: precision must be bf16, bf16x3, f16 or f16mix (= fp16 hi+lo planes on every layer)");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
        return fail("pcd: no CUDA device available -- this library has no CPU fallback");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    REQ(prop.major == 10, "the tcgen05 path requires an sm_100-class GPU (B200)");
    CU(configure_gemm_tc());

    TensorTable tt;
    for (int i = 0; i < n_tensors; ++i) tt.m[tensors[i].name] = &tensors[i];
    std::string err;
    auto h = std::unique_ptr<pcd_point_encoder>(new pcd_point_encoder());
    h->precision = precision; h->device = device; h->num_sms = prop.multiProcessorCount;
    h->f16 = (precision == PCD_PRECISION_F16 || precision == PCD_PRECISION_F16MIX) ? 1 : 0;
    h->planes = (precision == PCD_PRECISION_BF16X3 || precision == PCD_PRECISION_F16MIX) ? 2 : 1;

    // the widths are fixed to the reference defaults; a table with another hidden_dim / latent_dim is named as such
    {
        auto it = tt.m.find("vae.encoder.3.conv3.weight");
        const long long hidden = it == tt.m.end() ? kHidden : it->second->shape[0];
        it = tt.m.find("vae.fc_mu.weight");
        const long long latent = it == tt.m.end() ? kLatent : it->second->shape[0];
        REQ(hidden == kHidden && latent == kLatent,
            "pcd_point_encoder: only hidden_dim = 512 and latent_dim = 256 (the reference defaults) are supported, got hidden_dim = " +
                std::to_string(hidden) + ", latent_dim = " + std::to_string(latent));
    }
    static const int kIn[4] = {3, 64, 128, 256}, kOut[4] = {64, 128, 256, 512};
    for (int blk = 0; blk < 4; ++blk) {
        const std::string n = "vae.encoder." + std::to_string(blk);
        for (int j = 1; j <= 3; ++j) {
            HostMat m;
            if (!fold_conv_bn(tt, n + ".conv" + std::to_string(j), n + ".bn" + std::to_string(j), kOut[blk], j == 1 ? kIn[blk] : kOut[blk],
                              &m, &err))
                return fail(err);
            if (blk == 0 && j == 1) {
                if (pup(h.get(), m.w, &h->Wx) || pup(h.get(), m.b, &h->b0)) return 1;
            } else if (upload_conv(h.get(), m, &h->L[3 * blk + j - 1])) {
                return 1;
            }
        }
    }
    {
        const float *w6, *b6, *wm, *bm, *wl, *bl;
        const long long nh = 1LL * kLatent * kMid;
        if (!fetch(tt, "vae.encoder.6.weight", 1LL * kMid * kHidden, &w6, &err) || !fetch(tt, "vae.encoder.6.bias", kMid, &b6, &err) ||
            !fetch(tt, "vae.fc_mu.weight", nh, &wm, &err) || !fetch(tt, "vae.fc_mu.bias", kLatent, &bm, &err) ||
            !fetch(tt, "vae.fc_logvar.weight", nh, &wl, &err) || !fetch(tt, "vae.fc_logvar.bias", kLatent, &bl, &err))
            return fail(err);
        std::vector<float> wh(wm, wm + nh), bh(bm, bm + kLatent);
        wh.insert(wh.end(), wl, wl + nh);
        bh.insert(bh.end(), bl, bl + kLatent);
        if (pup(h.get(), std::vector<float>(w6, w6 + 1LL * kMid * kHidden), &h->w6) || pup(h.get(), std::vector<float>(b6, b6 + kMid), &h->b6) ||
            pup(h.get(), wh, &h->wh) || pup(h.get(), bh, &h->bh))
            return 1;
    }
    CU(cudaDeviceSynchronize());
    *out = h.release();
    return 0;
}

extern "C" int pcd_point_encoder_destroy(pcd_point_encoder* h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    h->plans.clear();
    for (void* p : h->owned) cudaFree(p);
    delete h;
    return 0;
}

// conv l (1..11) reading `src`; STORE into `dst`, or the max-pool epilogue into pl->pool
static int make_op(const pcd_point_encoder* h, const PPlan* pl, int l, const void* src, void* dst, int epi, PTcOp* out) {
    const PLayer& L = h->L[l];
    PTcOp op;
    op.layer = l; op.epi = epi;
    const int PL = h->planes;
    const long long M = pl->M, Mrows = M * PL;
    op.np = PL == 2 ? 3 : 1;
    op.out_planes = epi == EPI_STORE ? PL : 1;
    op.sh = tc_shape(epi, op.np, M, L.cout, L.cin, h->num_sms);
    TcGemmParams& p = op.p;
    p.kb0 = L.cin / 64; p.kb1 = 0; p.f16 = h->f16; p.tile_order = op.sh.tile_order;
    p.bias = L.b; p.bias_sample_stride = 0; p.rows_per_sample = pl->Npad; p.relu = 1;
    if (epi == EPI_MAXPOOL) {        // weights take the A role (128 channels per tile), points the B role
        p.num_m_blocks = L.cout / 128; p.num_n_blocks = static_cast<int>(M / op.sh.bn);
        p.a_plane_rows = PL == 2 ? L.cout : 0; p.b_plane_rows = PL == 2 ? static_cast<int>(M) : 0; p.out_plane_rows = 0;
        p.gmax = pl->pool; p.ld_g = kHidden; p.n_valid = pl->N; p.num_samples = pl->B;
        if (make_tmap(&op.a0, L.w16, static_cast<long long>(L.cout) * PL, L.cin, L.cin, 128)) return 1;
        if (make_tmap(&op.b, src, Mrows, L.cin, L.cin, op.sh.bn / op.sh.cl)) return 1;
        op.o = op.a0;
    } else {
        p.num_m_blocks = static_cast<int>(M / 128); p.num_n_blocks = L.cout / op.sh.bn;
        p.out = static_cast<__nv_bfloat16*>(dst); p.ldo = L.cout;
        p.a_plane_rows = PL == 2 ? static_cast<int>(M) : 0; p.b_plane_rows = PL == 2 ? L.cout : 0;
        p.out_plane_rows = PL == 2 ? static_cast<int>(M) : 0;
        p.epi_warps = 8;
        if (make_tmap(&op.a0, src, Mrows, L.cin, L.cin, 128)) return 1;
        if (make_tmap(&op.b, L.w16, static_cast<long long>(L.cout) * PL, L.cin, L.cin, op.sh.bn / op.sh.cl)) return 1;
        if (make_tmap_out32(&op.o, dst, Mrows, L.cout, L.cout)) return 1;
    }
    *out = op;
    return 0;
}

static int build_plan(pcd_point_encoder* h, int B, int N, PPlan** out) {
    const auto key = std::make_pair(B, N);
    if (PPlan* hit = h->plans.find(key)) { *out = hit; return 0; }
    h->plans.make_room();
    auto pl = std::unique_ptr<PPlan>(new PPlan());
    pl->B = B; pl->N = N; pl->Npad = (N + 127) / 128 * 128;
    pl->M = static_cast<long long>(B) * pl->Npad;
    REQ(pl->M < (1LL << 31), "pcd_point_encoder: B * Npad must be below 2^31 (shard the batch)");
    auto alloc = [&](void** p, size_t bytes) -> int {
        CU(cudaMalloc(p, bytes));
        pl->owned.push_back(*p);
        return 0;
    };
    const size_t act = static_cast<size_t>(h->planes) * pl->M * kHidden * 2;
    void *pool, *hid, *part, *flag, *call;
    if (alloc(&pl->T[0], act) || alloc(&pl->T[1], act) || alloc(&pool, sizeof(float) * B * kHidden) ||
        alloc(&hid, sizeof(float) * B * kMid) || alloc(&part, sizeof(float) * B * 2 * kHidden) || alloc(&flag, sizeof(int) * B) ||
        alloc(&call, sizeof(CallArgs)))
        return 1;
    pl->pool = static_cast<float*>(pool); pl->hid = static_cast<float*>(hid); pl->part = static_cast<float*>(part);
    pl->flag = static_cast<int*>(flag); pl->call = static_cast<CallArgs*>(call);
    // encoder.0.conv1 writes T[0]; conv l reads the buffer conv l - 1 wrote and writes the other one
    int src = 0;
    pl->out_buf[0] = 0;
    for (int l = 1; l < kConvs; ++l) {
        const int dst = 1 - src;
        const int epi = l == kConvs - 1 ? EPI_MAXPOOL : EPI_STORE;
        if (make_op(h, pl.get(), l, pl->T[src], epi == EPI_STORE ? pl->T[dst] : nullptr, epi, &pl->ops[l])) return 1;
        pl->out_buf[l] = dst;               // the max-pool layer: where tap_last writes
        if (epi == EPI_STORE) src = dst;
    }
    if (make_op(h, pl.get(), kConvs - 1, pl->T[src], pl->T[1 - src], EPI_STORE, &pl->tap_last)) return 1;
    *out = h->plans.insert(key, std::move(pl));
    return 0;
}

static int launch_tc(const pcd_point_encoder* h, const PTcOp& op, cudaStream_t s) {
    LAUNCH(launch_gemm_tc(op.sh.bn, op.epi, op.np, op.out_planes, op.sh.cl, op.sh.two_sm, op.a0, op.a0, op.b, op.o, op.p, h->num_sms, s));
    return 0;
}

// Stage i of one encode: 0 = non-finite flag, 1..12 = conv i - 1 (1 = encoder.0.conv1 on CUDA cores, 12 = encoder.3.conv3 +
// max-pool), 13 = encoder.6 + ReLU, 14 = fc_mu + fc_logvar (+ the NaN rule).  `last_store` runs stage 12 as a STORE layer.
static int run_stage(pcd_point_encoder* h, PPlan* pl, int i, const float* x, float* mu, float* logvar, bool last_store, cudaStream_t s) {
    const int B = pl->B;
    if (i == 0) {
        // pageable -> device copy of the per-call block: the runtime stages the source before returning
        CallArgs ca{};
        ca.s.x = const_cast<float*>(x); ca.s.N = pl->N; ca.s.Npad = pl->Npad;
        CU(cudaMemcpyAsync(pl->call, &ca, sizeof(CallArgs), cudaMemcpyHostToDevice, s));
        point_nonfinite_kernel<<<B, 256, 0, s>>>(x, 3LL * pl->N, pl->flag);
        LAUNCH(cudaGetLastError());
    } else if (i == 1) {
        char* T0 = static_cast<char*>(pl->T[0]);
        LAUNCH(launch_enc1_first(2, h->f16, pl->call, h->Wx, h->b0, 0, T0, h->planes == 2 ? T0 + pl->M * 64 * 2 : nullptr, B, pl->N,
                                 pl->Npad, s));
    } else if (i < kConvs) {
        if (launch_tc(h, pl->ops[i - 1], s)) return 1;
    } else if (i == kConvs) {
        if (last_store) return launch_tc(h, pl->tap_last, s);
        LAUNCH(launch_zero_f32(pl->pool, static_cast<long long>(B) * kHidden, s));
        if (launch_tc(h, pl->ops[kConvs - 1], s)) return 1;
    } else if (i == kConvs + 1) {
        SimtGemmParams p{};
        p.A0 = pl->pool; p.lda0 = kHidden; p.K0 = kHidden; p.A1 = nullptr; p.lda1 = 0; p.K1 = 0;
        p.W = h->w6; p.ldw = kHidden; p.M = B; p.Nout = kMid; p.out = pl->hid; p.ldo = kMid;
        p.bias = nullptr; p.bias_sample_stride = 0; p.rows_per_sample = 1 << 30; p.relu = 0;
        p.partial = pl->part; p.splits = kSplits6;
        LAUNCH(launch_gemm_simt(EPI_STORE, p, s));
        LAUNCH(launch_splitk_reduce(pl->part, kSplits6, h->b6, pl->hid, B, kMid, 1, s));
    } else {
        SimtGemmParams p{};
        p.A0 = pl->hid; p.lda0 = kMid; p.K0 = kMid; p.A1 = nullptr; p.lda1 = 0; p.K1 = 0;
        p.W = h->wh; p.ldw = kMid; p.M = B; p.Nout = 2 * kLatent; p.out = nullptr; p.ldo = 2 * kLatent;
        p.bias = nullptr; p.bias_sample_stride = 0; p.rows_per_sample = 1 << 30; p.relu = 0;
        p.partial = pl->part; p.splits = kSplitsHead;
        LAUNCH(launch_gemm_simt(EPI_STORE, p, s));
        const long long n = static_cast<long long>(B) * 2 * kLatent;
        point_heads_reduce_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(pl->part, kSplitsHead, h->bh, pl->flag, mu, logvar,
                                                                                           B, kLatent);
        LAUNCH(cudaGetLastError());
    }
    return 0;
}

static int prepare(pcd_point_encoder* h, int B, int N, PPlan** pl) {
    REQ(B > 0 && N > 0, "pcd_point_encoder: B and N must be positive (got B = " + std::to_string(B) + ", N = " + std::to_string(N) + ")");
    REQ(h != nullptr, "null argument");
    CU(cudaSetDevice(h->device));
    return build_plan(h, B, N, pl);
}

extern "C" int pcd_point_encode(pcd_point_encoder* h, const float* x, float* mu, float* logvar, int32_t B, int32_t N, void* stream) {
    PPlan* pl = nullptr;
    if (prepare(h, B, N, &pl)) return 1;
    REQ(x && mu && logvar, "null argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    for (int i = 0; i < kStages; ++i)
        if (run_stage(h, pl, i, x, mu, logvar, false, s)) return 1;
    return 0;
}

extern "C" int pcd_point_encoder_tap(pcd_point_encoder* h, const float* x, int32_t B, int32_t N, int32_t index, float* out_host,
                                     int64_t count, void* stream) {
    PPlan* pl = nullptr;
    if (prepare(h, B, N, &pl)) return 1;
    REQ(x && out_host, "null argument");
    REQ(index >= 0 && index <= kConvs + 1,
        "pcd_point_encoder_tap: index must be 0..11 (encoder.<i / 3>.conv<i % 3 + 1>), 12 (pooled) or 13 (encoder.7)");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int last = index < kConvs ? index + 1 : index;     // stage that produces the tapped tensor
    for (int i = 0; i <= last; ++i)
        if (run_stage(h, pl, i, x, nullptr, nullptr, index == kConvs - 1, s)) return 1;
    if (index >= kConvs) {
        const long long n = static_cast<long long>(B) * (index == kConvs ? kHidden : kMid);
        REQ(count == n, "pcd_point_encoder_tap: count must be B * " + std::to_string(index == kConvs ? kHidden : kMid));
        CU(cudaMemcpyAsync(out_host, index == kConvs ? pl->pool : pl->hid, sizeof(float) * n, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        return 0;
    }
    // activation after conv `index` (BN + ReLU), valid points only: [B][N][C]
    const int C = index == 0 ? 64 : h->L[index].cout;
    REQ(count == static_cast<long long>(B) * N * C, "pcd_point_encoder_tap: count must be B * N * " + std::to_string(C));
    const char* src = static_cast<const char*>(pl->T[pl->out_buf[index]]);
    float* tmp = nullptr;
    CU(cudaMalloc(reinterpret_cast<void**>(&tmp), sizeof(float) * pl->M * C));
    int rc = 0;
    cudaError_t e = launch_rows16_to_f32(src, h->planes == 2 ? src + pl->M * C * 2 : nullptr, C, tmp, C, pl->M, h->f16, s);
    for (int b = 0; b < B && e == cudaSuccess; ++b)
        e = cudaMemcpyAsync(out_host + static_cast<long long>(b) * N * C, tmp + static_cast<long long>(b) * pl->Npad * C,
                            sizeof(float) * N * C, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) rc = fail(std::string("pcd_point_encoder_tap: ") + cudaGetErrorString(e));
    cudaFree(tmp);
    return rc;
}

extern "C" int pcd_point_encoder_profile(pcd_point_encoder* h, const float* x, float* mu, float* logvar, int32_t B, int32_t N,
                                         float* ms_out, double* flops_out, char* names_out, int32_t name_stride, int32_t cap,
                                         int32_t* n_out, void* stream) {
    PPlan* pl = nullptr;
    if (prepare(h, B, N, &pl)) return 1;
    REQ(x && mu && logvar && ms_out && flops_out && n_out, "null argument");
    REQ(cap >= kStages, "pcd_point_encoder_profile: cap too small");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    std::vector<cudaEvent_t> ev(kStages + 1);
    for (auto& e : ev) CU(cudaEventCreate(&e));
    int rc = 0;
    if (cudaEventRecord(ev[0], s) != cudaSuccess) rc = fail("pcd_point_encoder_profile: event record failed");
    for (int i = 0; i < kStages && !rc; ++i) {
        rc = run_stage(h, pl, i, x, mu, logvar, false, s);
        if (!rc && cudaEventRecord(ev[i + 1], s) != cudaSuccess) rc = fail("pcd_point_encoder_profile: event record failed");
    }
    if (!rc && cudaStreamSynchronize(s) != cudaSuccess) rc = fail("pcd_point_encoder_profile: stream synchronisation failed");
    const double pts = static_cast<double>(B) * N;     // useful FLOPs: valid points only
    for (int i = 0; i < kStages && !rc; ++i) {
        cudaEventElapsedTime(&ms_out[i], ev[i], ev[i + 1]);
        std::string name;
        double fl = 0;
        if (i == 0) name = "nonfinite_flag";
        else if (i <= kConvs) {
            const int l = i - 1;
            const int cin = l == 0 ? 3 : h->L[l].cin, cout = l == 0 ? 64 : h->L[l].cout;
            name = "encoder." + std::to_string(l / 3) + ".conv" + std::to_string(l % 3 + 1) + (l == kConvs - 1 ? "+maxpool" : "");
            fl = 2.0 * pts * cin * cout;
        } else if (i == kConvs + 1) { name = "encoder.6+relu"; fl = 2.0 * B * kHidden * kMid; }
        else { name = "fc_mu+fc_logvar"; fl = 2.0 * B * kMid * 2 * kLatent; }
        flops_out[i] = fl;
        if (names_out && name_stride > 0) {
            std::strncpy(names_out + static_cast<size_t>(i) * name_stride, name.c_str(), name_stride - 1);
            names_out[static_cast<size_t>(i) * name_stride + name_stride - 1] = 0;
        }
    }
    for (auto& e : ev) cudaEventDestroy(e);
    *n_out = rc ? 0 : kStages;
    return rc;
}
