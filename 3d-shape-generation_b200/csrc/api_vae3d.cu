// C ABI of the voxel-VAE decoder: pcd_vae3d_* and pcd_voxel_* (include/pcd_b200.h).
//
// VAE3DLarge.decode (networks.py:2247-2264, 2327-2339):
//   decoder_input Linear(latent -> 512*4^3) -> view [B,512,4,4,4]
//   -> 3 x ( ConvTranspose3d(k=4, s=2, p=1) + ReLU -> ResidualBlock3D )      4^3 -> 8^3 -> 16^3 -> 32^3, 512 -> 256 -> 128 -> 64 ch
//   -> Conv3d(64 -> 32, k=3) + ReLU -> ResidualBlock3D(32) -> Conv3d(32 -> 1, k=3) -> Sigmoid
//
// Every convolution with >= 32 output channels is an IMPLICIT GEMM on the tcgen05 kernel of gemm_tc.cu: activations live
// channels-last ([plane][sample][d][h][w][C], 16-bit, the same row-major [voxel][C] matrix the per-point layers use), a 128-row
// A tile is a box of 128 consecutive voxels fetched by ONE 5-D TMA load per (tap, 64-channel block) with the box shifted by the
// tap offset -- TMA's out-of-bounds zero fill is the convolution's zero padding, so no im2col buffer and no halo logic exist.
//   * Conv3d k=3 p=1: 27 taps, K = 27 * Cin.
//   * ConvTranspose3d k=4 s=2 p=1: out[o] gathers in[i] * w[k] with o = 2i - 1 + k, so outputs of one parity class
//     (o mod 2 per axis) see exactly 2 taps per axis: 8 classes x (8 taps, K = 8 * Cin).  A class is one GEMM over the INPUT grid
//     whose output tile is scattered through a 5-D TMA store on a stride-2 view of the output grid.
//   * ResidualBlock3D (networks.py:471-505): BatchNorm3d (eval) folded into both convs; the identity shortcut rides along as Cin
//     extra K columns against an identity weight block (exact in split precision: hi + lo planes both pass through).
// decoder.12 (32 -> 1) + Sigmoid is a CUDA-core kernel (vae3d.cu); decoder_input is the fp32 CUDA-core GEMM.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <map>
#include <memory>
#include <tuple>

#include "api_common.h"
#include "pcd_launch.h"
#include "pcd_types.h"

using namespace pcd;

namespace pcd {
cudaError_t launch_vae3d_final_conv(const void* x, long long plane_elems, int planes, int f16, int ldc, int cin, int D, int H, int W,
                                    long long nvox_total, const float* w, const float* bias, float* out, cudaStream_t s);
cudaError_t launch_voxel_count(const float* vox, int B, int nvox, float threshold, int* counts, cudaStream_t s);
cudaError_t launch_voxel_points(const float* vox, int B, int D, int H, int W, float threshold, const long long* offsets, float* pts,
                                cudaStream_t s);
cudaError_t launch_f32_rows_to_16(const float* in, int c_src, void* hi, void* lo, int c_dst, long long rows, int f16, cudaStream_t s);
cudaError_t launch_rows16_to_f32(const void* hi, const void* lo, int ld, float* out, int c_keep, long long rows, int f16, cudaStream_t s);
}  // namespace pcd

namespace {

constexpr int kG0 = 4;             // decoder_input grid edge
constexpr int kC0 = 512;           // decoder_input channels
constexpr int kVox = 32 * 32 * 32;
constexpr int kTailLd = 32;        // channels per voxel row of decoder.12's input (dense 32-channel voxels)

inline int pad64(int c) { return (c + 63) / 64 * 64; }

struct Tap { int dd = 0, dh = 0, dw = 0; std::vector<float> w; };   // w: [cout_pad][cin_pad] fp32

struct ConvW {                     // one implicit GEMM: B-role weights [planes * cout_pad][K] 16-bit + folded fp32 bias
    int seq = 0;                   // index in the reference's nn.Sequential (decoder.<seq> / encoder.<seq>)
    std::string name;
    int cin_pad = 0, cout_pad = 0, K = 0;
    int W = 0, H = 0, D = 0;       // INPUT grid as the GEMM sees it (W halves for the voxel-pair layers); OUTPUT grid if stride 2
    int stride = 1;                // 2: Conv3d k=4 s=2 p=1, the GEMM rows are output voxels (input grid = 2W x 2H x 2D)
    int in_ld = 0;                 // channels per input voxel in memory (default cin_pad; 32 = dense 32-channel rows, the TMA box
                                   // of 64 channels zero-fills the rest)
    int res_pad = 0, res_ld = 0;   // residual: shortcut K columns (64-multiple) and channels per shortcut-source voxel in memory
                                   // (default cin_pad: the identity shortcut of a cin == cout block)
    int out_ld = 0;                // channels per output row in memory (64-multiple, or 32 = dense 32-channel voxels)
    int out_c = 0, out_rows = 0;   // debug tap: real channels per voxel and voxels per sample of the output
    bool residual = false, transposed = false, grouped = false;
    int par[3] = {0, 0, 0};        // transposed: output parity (d, h, w)
    // plain form (gemm_tc.cu, one A load per tap): offsets per tap
    int ntaps = 0;
    signed char dw[64] = {}, dh[64] = {}, dd[64] = {};
    // grouped form (conv3d_tc.cu): taps that differ only in dh share one A load
    int ngroups = 0, nt = 0;
    signed char gdw[32] = {}, gdh0[32] = {}, gdd[32] = {};
    void* w16 = nullptr;
    float* bias = nullptr;
    double flops = 0;              // algorithmic (unpadded, without identity shortcut columns), per sample
};

struct GemmOp {
    const ConvW* L = nullptr;
    CUtensorMap a0, a1, b, o;
    TcGemmParams p{};
    Conv3dParams cp{};
    int bn = 0, np = 1, out_planes = 1, cl = 1;
};

struct VPlan {
    int B = 0, Bpad = 0;
    void* buf[3] = {nullptr, nullptr, nullptr};
    float* lin = nullptr;          // decoder_input output [B][64 voxels][512] fp32
    std::vector<GemmOp> ops;
    std::vector<int> out_buf;      // per op: index of the buffer it writes
    int final_in = 0;              // buffer read by decoder.12
    std::vector<void*> owned;
    ~VPlan() { for (void* p : owned) cudaFree(p); }
};

}  // namespace

// What the implicit-GEMM layers of one half of the VAE share: precision, the packed layers, the device allocations
struct ConvNet {
    int precision = 0, device = 0, num_sms = 148, f16 = 0, planes = 1;
    std::vector<ConvW> convs;
    std::vector<void*> owned;
};

struct pcd_vae3d : ConvNet {
    int latent = 256;
    float *Win = nullptr, *bin = nullptr;     // decoder_input, rows permuted to channels-last: [(voxel * 512 + c)][latent]
    float *wf = nullptr, *bf = nullptr;       // decoder.12: [27][32] tap-major, [1]
    PlanCache<int, VPlan> plans;
};

template <typename T>
static int vup(ConvNet* h, const std::vector<T>& v, T** out) {
    void* p = nullptr;
    CU(cudaMalloc(&p, v.size() * sizeof(T)));
    h->owned.push_back(p);
    CU(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    *out = static_cast<T*>(p);
    return 0;
}

// fp32 [cout_pad][K] -> 16-bit planes on the device
static int upload_conv(ConvNet* h, const std::vector<float>& w, const std::vector<float>& b, ConvW* L) {
    float* w32 = nullptr;
    CU(cudaMalloc(reinterpret_cast<void**>(&w32), w.size() * sizeof(float)));
    CU(cudaMemcpy(w32, w.data(), w.size() * sizeof(float), cudaMemcpyHostToDevice));
    void* p = nullptr;
    CU(cudaMalloc(&p, w.size() * 2 * h->planes));
    h->owned.push_back(p);
    L->w16 = p;
    const long long n = static_cast<long long>(w.size());
    if (h->planes == 2) LAUNCH(launch_f32_split_16(w32, p, static_cast<char*>(p) + n * 2, n, h->f16, 0));
    else LAUNCH(launch_f32_to_16(w32, p, n, h->f16, 0));
    CU(cudaDeviceSynchronize());
    cudaFree(w32);
    return vup(h, b, &L->bias);
}

// Lay the per-tap matrices out along K and upload.  Plain: K = [tap][cin_pad] (+ [res_pad] shortcut columns for a residual
// block: identity, or the 1x1 `res_w` [cout_pad][res_pad]).  Grouped (64 output channels, whole w-lines per tile): taps that
// differ only in dh form a group that shares one A load; K = [group][64-channel block][h-tap][64] so that the group's weight
// tiles are consecutive k-blocks.  With stride 2 a group is the taps of one dh parity (box line t = input row 2 h + dh0 + 2 t).
static int pack_conv(ConvNet* h, ConvW L, std::vector<Tap>& taps, const std::vector<float>& bias,
                     const std::vector<float>* res_w = nullptr) {
    if (L.in_ld == 0) L.in_ld = L.cin_pad;
    if (L.residual && L.res_pad == 0) L.res_pad = L.cin_pad;
    if (L.residual && L.res_ld == 0) L.res_ld = L.res_pad;
    const int cin_kb = L.cin_pad / 64;
    const int bw = L.W, bh = bw > 0 && 128 % bw == 0 ? 128 / bw : 0;
    bool can_group = L.cout_pad == 64 && bh >= 1 && bw % 8 == 0 && L.H % bh == 0;
    std::map<std::tuple<int, int, int>, std::vector<int>> groups;    // (dd, dw, dh parity if stride 2) -> tap indices sorted by dh
    if (can_group) {
        for (size_t i = 0; i < taps.size(); ++i)
            groups[std::make_tuple(taps[i].dd, taps[i].dw, L.stride == 2 ? (taps[i].dh & 1) : 0)].push_back(static_cast<int>(i));
        int nt = -1;
        for (auto& g : groups) {
            std::sort(g.second.begin(), g.second.end(), [&](int a, int b) { return taps[a].dh < taps[b].dh; });
            for (size_t j = 1; j < g.second.size(); ++j)
                if (taps[g.second[j]].dh != taps[g.second[j - 1]].dh + L.stride) can_group = false;
            if (nt < 0) nt = static_cast<int>(g.second.size());
            if (nt != static_cast<int>(g.second.size())) can_group = false;
        }
        if (nt < 1 || nt > 3 || (bh + nt - 1) * bw > 192 || groups.size() > 32) can_group = false;
        if (L.residual && nt != 1 && nt != 3) can_group = false;
        if (can_group) L.nt = nt;
    }
    L.grouped = can_group;
    const int res_cols = L.residual ? L.res_pad : 0;
    L.K = static_cast<int>(taps.size()) * L.cin_pad + res_cols;
    std::vector<float> wm(static_cast<size_t>(L.cout_pad) * L.K, 0.f);
    auto put = [&](int kblk, const Tap& t, int cb) {
        for (int co = 0; co < L.cout_pad; ++co)
            std::memcpy(&wm[static_cast<size_t>(co) * L.K + static_cast<size_t>(kblk) * 64],
                        &t.w[static_cast<size_t>(co) * L.cin_pad + cb * 64], sizeof(float) * 64);
    };
    if (can_group) {
        int g = 0;
        for (auto& kv : groups) {
            L.gdd[g] = static_cast<signed char>(std::get<0>(kv.first)); L.gdw[g] = static_cast<signed char>(std::get<1>(kv.first));
            L.gdh0[g] = static_cast<signed char>(taps[kv.second[0]].dh);
            for (int cb = 0; cb < cin_kb; ++cb)
                for (int t = 0; t < L.nt; ++t) put((g * cin_kb + cb) * L.nt + t, taps[kv.second[t]], cb);
            ++g;
        }
        L.ngroups = g;
    } else {
        REQ(taps.size() <= 64, "internal: too many taps");
        L.ntaps = static_cast<int>(taps.size());
        for (int i = 0; i < L.ntaps; ++i) {
            L.dd[i] = static_cast<signed char>(taps[i].dd); L.dh[i] = static_cast<signed char>(taps[i].dh);
            L.dw[i] = static_cast<signed char>(taps[i].dw);
            for (int cb = 0; cb < cin_kb; ++cb) put(i * cin_kb + cb, taps[i], cb);
        }
    }
    if (L.residual && res_w) {
        for (int co = 0; co < L.cout_pad; ++co)
            std::memcpy(&wm[static_cast<size_t>(co) * L.K + taps.size() * L.cin_pad], &(*res_w)[static_cast<size_t>(co) * L.res_pad],
                        sizeof(float) * L.res_pad);
    } else if (L.residual) {
        for (int c = 0; c < L.cin_pad && c < L.cout_pad; ++c)
            wm[static_cast<size_t>(c) * L.K + static_cast<size_t>(taps.size()) * L.cin_pad + c] = 1.f;
    }
    if (upload_conv(h, wm, bias, &L)) return 1;
    h->convs.push_back(L);
    return 0;
}

// eval-mode BatchNorm3d scale/shift (networks.py:484-487): y = s * (x - mu) + beta, s = gamma / sqrt(var + 1e-5)
static bool bn_fold(const TensorTable& tt, const std::string& bn, int c, std::vector<double>* s, std::vector<double>* t, std::string* err) {
    const float *g, *beta, *mu, *var;
    if (!fetch(tt, bn + ".weight", c, &g, err) || !fetch(tt, bn + ".bias", c, &beta, err) ||
        !fetch(tt, bn + ".running_mean", c, &mu, err) || !fetch(tt, bn + ".running_var", c, &var, err))
        return false;
    s->resize(c); t->resize(c);
    for (int i = 0; i < c; ++i) {
        (*s)[i] = static_cast<double>(g[i]) / std::sqrt(static_cast<double>(var[i]) + 1e-5);
        (*t)[i] = static_cast<double>(beta[i]) - (*s)[i] * mu[i];
    }
    return true;
}

// Conv3d(cin -> cout, k=3, p=1) [+ BatchNorm3d] [+ identity shortcut] at grid edge G.
// `pairs`: 32-channel layers (cin == cout == 32) run on the grid of VOXEL PAIRS along w: the dense [voxel][32] activation IS a
// [pair][64] matrix, so K and N are not padded.  Output voxel 2j + ho takes input voxel 2(j + s) + hi through kernel column
// kw = 2s + hi - ho + 1 (when that is 0..2): three pair-taps s = -1, 0, +1 with 64 x 64 blocks (half of the entries zero).
// `dense_out`: cout == 32 written as dense 32-channel rows (the TMA store clips the padded columns).
static int add_conv3(ConvNet* h, const TensorTable& tt, const std::string& conv, const std::string& bn, int seq, int cin, int cout,
                     int G, bool residual, bool pairs, bool dense_out) {
    std::string err;
    const float *w, *b;
    if (!fetch(tt, conv + ".weight", 27LL * cin * cout, &w, &err) || !fetch(tt, conv + ".bias", cout, &b, &err)) return fail(err);
    std::vector<double> s(cout, 1.0), t(cout, 0.0);
    if (!bn.empty() && !bn_fold(tt, bn, cout, &s, &t, &err)) return fail(err);
    ConvW L;
    L.seq = seq; L.name = conv; L.residual = residual;
    L.W = pairs ? G / 2 : G; L.H = G; L.D = G;
    L.cin_pad = pairs ? 64 : pad64(cin); L.cout_pad = pairs ? 64 : pad64(cout);
    L.out_ld = (pairs || !dense_out) ? L.cout_pad : cout;
    L.out_c = cout; L.out_rows = G * G * G;
    L.flops = 2.0 * 27 * cin * cout * G * G * G;
    std::vector<Tap> taps;
    std::vector<float> bm(L.cout_pad, 0.f);
    auto wref = [&](int co, int ci, int kd, int kh, int kw) {      // nn.Conv3d weight [cout][cin][kd][kh][kw], BN scale folded
        return static_cast<float>(s[co] * w[(static_cast<size_t>(co) * cin + ci) * 27 + (kd * 3 + kh) * 3 + kw]);
    };
    for (int kd = 0; kd < 3; ++kd)
        for (int kh = 0; kh < 3; ++kh)
            for (int ks = 0; ks < 3; ++ks) {           // cross-correlation: out[o] += w[k] * in[o + k - 1]
                Tap tp; tp.dd = kd - 1; tp.dh = kh - 1; tp.dw = ks - 1;
                tp.w.assign(static_cast<size_t>(L.cout_pad) * L.cin_pad, 0.f);
                if (!pairs) {
                    for (int co = 0; co < cout; ++co)
                        for (int ci = 0; ci < cin; ++ci) tp.w[static_cast<size_t>(co) * L.cin_pad + ci] = wref(co, ci, kd, kh, ks);
                } else {
                    for (int ho = 0; ho < 2; ++ho)
                        for (int hi = 0; hi < 2; ++hi) {
                            const int kw = 2 * (ks - 1) + hi - ho + 1;
                            if (kw < 0 || kw > 2) continue;
                            for (int co = 0; co < cout; ++co)
                                for (int ci = 0; ci < cin; ++ci)
                                    tp.w[static_cast<size_t>(ho * 32 + co) * 64 + hi * 32 + ci] = wref(co, ci, kd, kh, kw);
                        }
                }
                taps.push_back(std::move(tp));
            }
    for (int co = 0; co < cout; ++co) {
        bm[co] = static_cast<float>(s[co] * b[co] + t[co]);
        if (pairs) bm[32 + co] = bm[co];
    }
    return pack_conv(h, L, taps, bm);
}

// ConvTranspose3d(cin -> cout, k=4, s=2, p=1): 8 output-parity classes at INPUT grid edge G
static int add_convT(ConvNet* h, const TensorTable& tt, const std::string& conv, int seq, int cin, int cout, int G) {
    std::string err;
    const float *w, *b;
    if (!fetch(tt, conv + ".weight", 64LL * cin * cout, &w, &err) || !fetch(tt, conv + ".bias", cout, &b, &err)) return fail(err);
    // per axis: parity 0 (o = 2j): (di, k) = (0, 1), (-1, 3);  parity 1 (o = 2j + 1): (0, 2), (+1, 0)
    static const int DI[2][2] = {{0, -1}, {0, 1}}, KI[2][2] = {{1, 3}, {2, 0}};
    for (int cls = 0; cls < 8; ++cls) {
        ConvW L;
        L.seq = seq; L.name = conv + "[" + std::to_string(cls) + "]";
        L.cin_pad = pad64(cin); L.cout_pad = pad64(cout); L.W = L.H = L.D = G; L.transposed = true;
        L.out_ld = L.cout_pad; L.out_c = cout; L.out_rows = 8 * G * G * G;
        L.par[0] = (cls >> 2) & 1; L.par[1] = (cls >> 1) & 1; L.par[2] = cls & 1;
        L.flops = 2.0 * 8 * cin * cout * G * G * G;
        std::vector<Tap> taps;
        std::vector<float> bm(L.cout_pad, 0.f);
        for (int tap = 0; tap < 8; ++tap) {
            const int td = (tap >> 2) & 1, th = (tap >> 1) & 1, tw = tap & 1;
            Tap tp; tp.dd = DI[L.par[0]][td]; tp.dh = DI[L.par[1]][th]; tp.dw = DI[L.par[2]][tw];
            const int kd = KI[L.par[0]][td], kh = KI[L.par[1]][th], kw = KI[L.par[2]][tw];
            tp.w.assign(static_cast<size_t>(L.cout_pad) * L.cin_pad, 0.f);
            for (int co = 0; co < cout; ++co)
                for (int ci = 0; ci < cin; ++ci)     // nn.ConvTranspose3d weight [cin][cout][kd][kh][kw]
                    tp.w[static_cast<size_t>(co) * L.cin_pad + ci] = w[((static_cast<size_t>(ci) * cout + co) * 4 + kd) * 16 + kh * 4 + kw];
            taps.push_back(std::move(tp));
        }
        for (int co = 0; co < cout; ++co) bm[co] = b[co];
        if (pack_conv(h, L, taps, bm)) return 1;
    }
    return 0;
}

extern "C" int pcd_vae3d_destroy(pcd_vae3d* h);

extern "C" int pcd_vae3d_create(const pcd_named_tensor* tensors, int32_t n_tensors, int32_t precision, int32_t device,
                                pcd_vae3d** out) {
    REQ(tensors && out, "null argument");
    REQ(precision == PCD_PRECISION_BF16 || precision == PCD_PRECISION_BF16X3 || precision == PCD_PRECISION_F16 ||
            precision == PCD_PRECISION_F16MIX,
        "pcd_vae3d: precision must be bf16, bf16x3, f16 or f16mix (= fp16 hi+lo planes on every layer)");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
        return fail("pcd: no CUDA device available -- this library has no CPU fallback");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    REQ(prop.major == 10, "the tcgen05 path requires an sm_100-class GPU (B200)");
    CU(configure_gemm_tc());
    CU(configure_conv3d_tc());

    TensorTable tt;
    for (int i = 0; i < n_tensors; ++i) tt.m[tensors[i].name] = &tensors[i];
    std::string err;
    auto h = std::unique_ptr<pcd_vae3d>(new pcd_vae3d());
    h->precision = precision; h->device = device; h->num_sms = prop.multiProcessorCount;
    h->f16 = (precision == PCD_PRECISION_F16 || precision == PCD_PRECISION_F16MIX) ? 1 : 0;
    h->planes = (precision == PCD_PRECISION_BF16X3 || precision == PCD_PRECISION_F16MIX) ? 2 : 1;

    // ---- decoder_input (networks.py:2245, 2337-2338): row c * 64 + v of the reference -> row v * 512 + c (channels-last)
    {
        const pcd_named_tensor* t = tt.get("vae.decoder_input.weight", &err);
        if (!t) return fail(err);
        REQ(t->ndim == 2 && t->shape[0] == kC0 * kG0 * kG0 * kG0 && t->shape[1] % 4 == 0, "vae.decoder_input.weight must be [32768, latent]");
        h->latent = static_cast<int>(t->shape[1]);
        const float *w, *b;
        const int rows = kC0 * 64;
        if (!fetch(tt, "vae.decoder_input.weight", 1LL * rows * h->latent, &w, &err) || !fetch(tt, "vae.decoder_input.bias", rows, &b, &err))
            return fail(err);
        std::vector<float> wp(static_cast<size_t>(rows) * h->latent), bp(rows);
        for (int c = 0; c < kC0; ++c)
            for (int v = 0; v < 64; ++v) {
                std::memcpy(&wp[(static_cast<size_t>(v) * kC0 + c) * h->latent], &w[(static_cast<size_t>(c) * 64 + v) * h->latent],
                            sizeof(float) * h->latent);
                bp[v * kC0 + c] = b[c * 64 + v];
            }
        if (vup(h.get(), wp, &h->Win) || vup(h.get(), bp, &h->bin)) return 1;
    }
    // ---- the nn.Sequential decoder (networks.py:2247-2264)
    struct Stage { int seqT, seqR, cin, cout, G; };
    const Stage stages[3] = {{0, 2, 512, 256, 4}, {3, 5, 256, 128, 8}, {6, 8, 128, 64, 16}};
    auto res = [&](int seq, int c, int G, bool pairs) -> int {
        const std::string n = "vae.decoder." + std::to_string(seq);
        if (add_conv3(h.get(), tt, n + ".conv1", n + ".bn1", seq, c, c, G, false, pairs, false)) return 1;
        return add_conv3(h.get(), tt, n + ".conv2", n + ".bn2", seq, c, c, G, true, pairs, false);
    };
    for (const Stage& s : stages) {
        if (add_convT(h.get(), tt, "vae.decoder." + std::to_string(s.seqT), s.seqT, s.cin, s.cout, s.G)) return 1;
        if (res(s.seqR, s.cout, 2 * s.G, false)) return 1;
    }
    // the 32-channel tail: dense 32-channel rows, decoder.11 on voxel pairs
    if (add_conv3(h.get(), tt, "vae.decoder.9", "", 9, 64, 32, 32, false, false, true)) return 1;
    if (res(11, 32, 32, true)) return 1;
    {
        const float *w, *b;
        if (!fetch(tt, "vae.decoder.12.weight", 27 * 32, &w, &err) || !fetch(tt, "vae.decoder.12.bias", 1, &b, &err)) return fail(err);
        std::vector<float> wf(27 * 32), bf(1, b[0]);
        for (int ci = 0; ci < 32; ++ci)
            for (int tap = 0; tap < 27; ++tap) wf[tap * 32 + ci] = w[ci * 27 + tap];
        if (vup(h.get(), wf, &h->wf) || vup(h.get(), bf, &h->bf)) return 1;
    }
    CU(cudaDeviceSynchronize());
    *out = h.release();
    return 0;
}

extern "C" int pcd_vae3d_destroy(pcd_vae3d* h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    h->plans.clear();
    for (void* p : h->owned) cudaFree(p);
    delete h;
    return 0;
}

// box of `rows` consecutive voxels of a W x H x D grid (w fastest), as (bw, bh, bd, bb)
static void voxel_box(int W, int H, int D, int rows, int box[4]) {
    const int dims[3] = {W, H, D};
    int rem = rows;
    for (int i = 0; i < 3; ++i) { box[i] = rem < dims[i] ? rem : dims[i]; rem /= box[i]; }
    box[3] = rem;
}

// One implicit-GEMM launch of layer L over Bp samples per plane: A source 0 = the grid at `src`, A source 1 = the shortcut
// source grid at `res` (residual layers), output grid at `dst`.
static int make_conv_op(const ConvNet* h, const ConvW& L, void* src, void* res, void* dst, int Bp, GemmOp* out) {
    GemmOp op;
    op.L = &L;
    const int PL = h->planes;
    const long long nb = static_cast<long long>(PL) * Bp;             // samples incl. the lo plane (plane p at batch index p * Bpad)
    const long long vox_in = static_cast<long long>(L.W) * L.H * L.D;
    const long long M = static_cast<long long>(Bp) * vox_in;              // rows of one plane
    REQ(M % 128 == 0 && M * PL < (1LL << 31), "pcd_vae3d: batch too large for one call (shard the batch)");
    op.np = PL == 2 ? 3 : 1; op.out_planes = PL;
    const int cin_kb = L.cin_pad / 64;
    const long long Co = L.cout_pad;
    const int Wo = 2 * L.W, Ho = 2 * L.H, Do = 2 * L.D;                    // transposed: output grid
    // A source 0: the input grid (stride 2: twice the GEMM grid, stepped 2 voxels per box element); source 1: the shortcut source
    const int S = L.stride;
    const long long Ci = L.in_ld, Wi = S * L.W, Hi = S * L.H, Di = S * L.D, Cr = L.residual ? L.res_ld : 0;
    int box[4];
    if (L.grouped) {
        Conv3dParams& q = op.cp;
        q.num_m_blocks = static_cast<int>(M / 128);
        q.W = L.W; q.H = L.H; q.D = L.D; q.bw = L.W; q.bh = 128 / L.W;
        q.ngroups = L.ngroups; q.nt = L.nt; q.cin_kb = cin_kb;
        q.res = L.residual ? 1 : 0; q.res_t = L.nt == 3 ? 1 : 0; q.res_kb = L.residual ? L.res_pad / 64 : 0; q.stride = S;
        q.a_box_bytes = (q.bh + q.nt - 1) * q.bw * 128;
        q.batch_plane = Bp; q.b_plane_rows = PL == 2 ? L.cout_pad : 0; q.out_plane_rows = PL == 2 ? static_cast<int>(M) : 0;
        q.store5d = L.transposed ? 1 : 0; q.relu = 1; q.bias = L.bias;
        std::memcpy(q.gdw, L.gdw, 32); std::memcpy(q.gdh0, L.gdh0, 32); std::memcpy(q.gdd, L.gdd, 32);
        op.bn = 64;
        op.cl = q.num_m_blocks % 2 == 0 ? 2 : 1;
        const int bhh = q.bh + q.nt - 1;
        if (make_tmap5(&op.a0, src, static_cast<int>(Ci), static_cast<int>(Wi), static_cast<int>(Hi), static_cast<int>(Di), nb, Ci, Ci * Wi,
                       Ci * Wi * Hi, Ci * Wi * Hi * Di, q.bw, bhh, 1, 1, S))
            return 1;
        if (L.residual) {
            if (make_tmap5(&op.a1, res, static_cast<int>(Cr), L.W, L.H, L.D, nb, Cr, Cr * L.W, Cr * L.W * L.H, Cr * vox_in, q.bw, bhh, 1, 1))
                return 1;
        } else op.a1 = op.a0;
        if (make_tmap(&op.b, L.w16, static_cast<long long>(L.cout_pad) * PL, L.K, L.K, 64 / op.cl)) return 1;
    } else {
        TcGemmParams& q = op.p;
        op.bn = PL == 2 ? (L.cout_pad >= 128 ? 128 : L.cout_pad) : (L.cout_pad >= 256 ? 256 : L.cout_pad);
        q.conv.ntaps = L.ntaps; q.conv.cin_kb = cin_kb; q.conv.W = L.W; q.conv.H = L.H; q.conv.D = L.D; q.conv.batch_plane = Bp;
        q.conv.store5d = L.transposed ? 1 : 0; q.conv.stride = S;
        std::memcpy(q.conv.dw, L.dw, 64); std::memcpy(q.conv.dh, L.dh, 64); std::memcpy(q.conv.dd, L.dd, 64);
        q.num_m_blocks = static_cast<int>(M / 128); q.num_n_blocks = L.cout_pad / op.bn;
        q.kb0 = L.ntaps * cin_kb; q.kb1 = L.residual ? L.res_pad / 64 : 0;
        q.a_plane_rows = 0; q.b_plane_rows = PL == 2 ? L.cout_pad : 0; q.out_plane_rows = PL == 2 ? static_cast<int>(M) : 0;
        q.bias = L.bias; q.bias_sample_stride = 0; q.rows_per_sample = 1 << 30; q.relu = 1; q.f16 = h->f16;
        q.num_samples = Bp;
        voxel_box(L.W, L.H, L.D, 128, box);
        if (make_tmap5(&op.a0, src, static_cast<int>(Ci), static_cast<int>(Wi), static_cast<int>(Hi), static_cast<int>(Di), nb, Ci, Ci * Wi,
                       Ci * Wi * Hi, Ci * Wi * Hi * Di, box[0], box[1], box[2], box[3], S))
            return 1;
        if (L.residual) {
            if (make_tmap5(&op.a1, res, static_cast<int>(Cr), L.W, L.H, L.D, nb, Cr, Cr * L.W, Cr * L.W * L.H, Cr * vox_in, box[0], box[1],
                           box[2], box[3]))
                return 1;
        } else op.a1 = op.a0;
        if (make_tmap(&op.b, L.w16, static_cast<long long>(L.cout_pad) * PL, L.K, L.K, op.bn)) return 1;
    }
    if (L.transposed) {
        // stride-2 view of the output grid that holds this parity class: voxel (d, h, w) of the view = output voxel
        // (2d + pd, 2h + ph, 2w + pw)
        voxel_box(L.W, L.H, L.D, 32, box);
        char* base = static_cast<char*>(dst) + ((static_cast<long long>(L.par[0]) * Ho + L.par[1]) * Wo + L.par[2]) * Co * 2;
        if (make_tmap5(&op.o, base, L.cout_pad, L.W, L.H, L.D, nb, 2 * Co, 2 * Co * Wo, 2 * Co * Wo * Ho, Co * Wo * Ho * Do, box[0], box[1],
                       box[2], box[3]))
            return 1;
    } else {
        // out_ld < cout_pad (dense 32-channel rows): the store box is still 64 columns wide, TMA clips columns >= out_ld
        if (make_tmap(&op.o, dst, M * PL, L.out_ld, L.out_ld, 32)) return 1;
    }
    *out = op;
    return 0;
}

static int build_vplan(pcd_vae3d* h, int B, VPlan** out) {
    if (VPlan* hit = h->plans.find(B)) { *out = hit; return 0; }
    h->plans.make_room();
    auto pl = std::unique_ptr<VPlan>(new VPlan());
    pl->B = B; pl->Bpad = (B + 1) / 2 * 2;          // a 128-row tile of the 4^3 grid spans two samples
    const int PL = h->planes, Bp = pl->Bpad;
    const long long nb = static_cast<long long>(PL) * Bp;          // samples incl. the lo plane (plane p at batch index p * Bpad)
    const size_t buf_bytes = static_cast<size_t>(nb) * kVox * 64 * 2;   // largest grid: 32^3 x 64 channels
    for (int i = 0; i < 3; ++i) {
        CU(cudaMalloc(&pl->buf[i], buf_bytes));
        pl->owned.push_back(pl->buf[i]);
        CU(cudaMemset(pl->buf[i], 0, buf_bytes));
    }
    void* p = nullptr;
    CU(cudaMalloc(&p, sizeof(float) * B * 64 * kC0));
    pl->owned.push_back(p); pl->lin = static_cast<float*>(p);

    // buffer rotation: `cur` holds the current activation, `res_in` the input of the residual block being built, `t_dst` the
    // output grid the 8 parity classes of a transposed conv scatter into
    int cur = 0, res_in = 0, t_dst = 0;
    auto free_buf = [&](int x, int y) { for (int i = 0; i < 3; ++i) if (i != x && i != y) return i; return -1; };
    for (size_t li = 0; li < h->convs.size(); ++li) {
        const ConvW& L = h->convs[li];
        const int src = cur;
        int dst;
        if (L.transposed) {
            if (L.par[0] + L.par[1] + L.par[2] == 0) t_dst = free_buf(cur, cur);
            dst = t_dst;
        } else if (L.residual) {
            dst = free_buf(cur, res_in);        // conv2: reads conv1's output (cur) and the block input (res_in)
        } else {
            dst = free_buf(cur, cur);
        }
        GemmOp op;
        if (make_conv_op(h, L, pl->buf[src], pl->buf[res_in], pl->buf[dst], Bp, &op)) return 1;
        pl->ops.push_back(op);
        pl->out_buf.push_back(dst);
        if (L.transposed) {
            if (L.par[0] + L.par[1] + L.par[2] == 3) cur = dst;
        } else {
            if (!L.residual) res_in = src;      // a following conv2 takes this op's input as its shortcut
            cur = dst;
        }
    }
    pl->final_in = cur;
    *out = h->plans.insert(B, std::move(pl));
    return 0;
}

static int launch_op(const ConvNet* h, const GemmOp& op, cudaStream_t s) {
    if (op.L->grouped) LAUNCH(launch_conv3d_tc(op.np, op.cl, h->f16, op.a0, op.a1, op.b, op.o, op.cp, h->num_sms, s));
    else LAUNCH(launch_gemm_tc(op.bn, EPI_STORE, op.np, op.out_planes, 1, 0, op.a0, op.a1, op.b, op.o, op.p, h->num_sms, s));
    return 0;
}

// decoder_input + conversion into the first activation grid
static int launch_head(pcd_vae3d* h, VPlan* pl, const float* z, cudaStream_t s) {
    SimtGemmParams p{};
    p.A0 = z; p.lda0 = h->latent; p.K0 = h->latent; p.A1 = nullptr; p.lda1 = 0; p.K1 = 0;
    p.W = h->Win; p.ldw = h->latent; p.M = pl->B; p.Nout = kC0 * 64; p.out = pl->lin; p.ldo = kC0 * 64;
    p.bias = h->bin; p.bias_sample_stride = 0; p.rows_per_sample = 1 << 30; p.relu = 0;
    p.partial = nullptr; p.splits = 1;
    LAUNCH(launch_gemm_simt(EPI_STORE, p, s));
    const long long rows = static_cast<long long>(pl->B) * 64;
    char* hi = static_cast<char*>(pl->buf[0]);
    char* lo = h->planes == 2 ? hi + static_cast<long long>(pl->Bpad) * 64 * kC0 * 2 : nullptr;
    LAUNCH(launch_f32_rows_to_16(pl->lin, kC0, hi, lo, kC0, rows, h->f16, s));
    return 0;
}

static int launch_tail(pcd_vae3d* h, VPlan* pl, float* vox, cudaStream_t s) {
    const long long plane_elems = static_cast<long long>(pl->Bpad) * kVox * kTailLd;
    LAUNCH(launch_vae3d_final_conv(pl->buf[pl->final_in], plane_elems, h->planes, h->f16, kTailLd, 32, 32, 32, 32,
                                   static_cast<long long>(pl->B) * kVox, h->wf, h->bf, vox, s));
    return 0;
}

extern "C" int pcd_vae3d_decode(pcd_vae3d* h, const float* z, float* vox, int32_t B, void* stream) {
    REQ(h && z && vox, "null argument");
    REQ(B > 0, "B must be positive");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    VPlan* pl = nullptr;
    if (build_vplan(h, B, &pl)) return 1;
    if (launch_head(h, pl, z, s)) return 1;
    for (const GemmOp& op : pl->ops)
        if (launch_op(h, op, s)) return 1;
    return launch_tail(h, pl, vox, s);
}

extern "C" int pcd_vae3d_tap(pcd_vae3d* h, const float* z, int32_t B, int32_t seq_index, float* out_host, int64_t count, void* stream) {
    REQ(h && z && out_host, "null argument");
    REQ(B > 0, "B must be positive");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    VPlan* pl = nullptr;
    if (build_vplan(h, B, &pl)) return 1;
    if (launch_head(h, pl, z, s)) return 1;
    int last = -1;
    if (seq_index >= 0) {
        for (size_t i = 0; i < pl->ops.size(); ++i) {
            if (pl->ops[i].L->seq > seq_index) break;
            if (launch_op(h, pl->ops[i], s)) return 1;
            last = static_cast<int>(i);
        }
        REQ(last >= 0 && pl->ops[last].L->seq == seq_index, "pcd_vae3d_tap: seq_index must be -1 (decoder_input) or one of 0,2,3,5,6,8,9,11");
    }
    const long long vps = last < 0 ? 64 : pl->ops[last].L->out_rows;      // voxels per sample of the tapped activation
    const int creal = last < 0 ? kC0 : pl->ops[last].L->out_c;
    // channels per voxel row in memory (a voxel-pair layer stores [pair][64] = dense [voxel][32])
    const int ld = last < 0 ? kC0 : (pl->ops[last].L->out_ld == 64 && creal == 32 ? 32 : pl->ops[last].L->out_ld);
    const void* src = last < 0 ? pl->buf[0] : pl->buf[pl->out_buf[last]];
    const long long rows = static_cast<long long>(B) * vps;
    REQ(count == rows * creal, "pcd_vae3d_tap: count must be B * G^3 * C of the tapped layer (channels-last)");
    const char* lo = h->planes == 2 ? static_cast<const char*>(src) + static_cast<long long>(pl->Bpad) * vps * ld * 2 : nullptr;
    float* tmp = nullptr;
    CU(cudaMalloc(reinterpret_cast<void**>(&tmp), sizeof(float) * count));
    LAUNCH(launch_rows16_to_f32(src, lo, ld, tmp, creal, rows, h->f16, s));
    CU(cudaMemcpyAsync(out_host, tmp, sizeof(float) * count, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    cudaFree(tmp);
    return 0;
}

extern "C" int pcd_vae3d_profile(pcd_vae3d* h, const float* z, float* vox, int32_t B, float* ms_out, double* flops_out, char* names_out,
                                 int32_t name_stride, int32_t cap, int32_t* n_out, void* stream) {
    REQ(h && z && vox && ms_out && flops_out && n_out, "null argument");
    REQ(B > 0, "B must be positive");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    VPlan* pl = nullptr;
    if (build_vplan(h, B, &pl)) return 1;
    const int n = static_cast<int>(pl->ops.size()) + 2;
    REQ(cap >= n, "pcd_vae3d_profile: cap too small");
    std::vector<cudaEvent_t> ev(n + 1);
    for (auto& e : ev) CU(cudaEventCreate(&e));
    CU(cudaEventRecord(ev[0], s));
    if (launch_head(h, pl, z, s)) return 1;
    CU(cudaEventRecord(ev[1], s));
    for (size_t i = 0; i < pl->ops.size(); ++i) {
        if (launch_op(h, pl->ops[i], s)) return 1;
        CU(cudaEventRecord(ev[i + 2], s));
    }
    if (launch_tail(h, pl, vox, s)) return 1;
    CU(cudaEventRecord(ev[n], s));
    CU(cudaStreamSynchronize(s));
    for (int i = 0; i < n; ++i) {
        CU(cudaEventElapsedTime(&ms_out[i], ev[i], ev[i + 1]));
        std::string name; double fl = 0;
        if (i == 0) { name = "decoder_input"; fl = 2.0 * h->latent * kC0 * 64 * B; }
        else if (i == n - 1) { name = "decoder.12+sigmoid"; fl = 2.0 * 27 * 32 * kVox * B; }
        else { name = pl->ops[i - 1].L->name.substr(4); fl = pl->ops[i - 1].L->flops * B; }
        flops_out[i] = fl;
        if (names_out && name_stride > 0) {
            std::strncpy(names_out + static_cast<size_t>(i) * name_stride, name.c_str(), name_stride - 1);
            names_out[static_cast<size_t>(i) * name_stride + name_stride - 1] = 0;
        }
    }
    for (auto& e : ev) cudaEventDestroy(e);
    *n_out = n;
    return 0;
}

extern "C" int pcd_voxel_count(const float* vox, int32_t B, int32_t D, int32_t H, int32_t W, float threshold, int32_t* counts,
                               void* stream) {
    REQ(vox && counts, "null argument");
    REQ(B > 0 && D > 0 && H > 0 && W > 0 && 1LL * D * H * W < (1LL << 30), "bad voxel grid shape");
    LAUNCH(launch_voxel_count(vox, B, D * H * W, threshold, counts, static_cast<cudaStream_t>(stream)));
    return 0;
}

extern "C" int pcd_voxel_points(const float* vox, int32_t B, int32_t D, int32_t H, int32_t W, float threshold, const int64_t* offsets,
                                float* pts, void* stream) {
    REQ(vox && offsets && pts, "null argument");
    REQ(B > 0 && D > 0 && H > 0 && W > 0 && 1LL * D * H * W < (1LL << 30), "bad voxel grid shape");
    LAUNCH(launch_voxel_points(vox, B, D, H, W, threshold, reinterpret_cast<const long long*>(offsets), pts,
                               static_cast<cudaStream_t>(stream)));
    return 0;
}

// =====================================================================================================================
// VAE3DLarge.encode (networks.py:2208-2243 encoder / fc_mu / fc_logvar; encode just above decode at :2327):
//   encoder.0  Conv3d(1 -> 32, k=3, p=1) + ReLU                        CUDA cores (vae3d.cu), dense 32-channel rows
//   3 x ( ResidualBlock3D(c -> 2c) -> Conv3d(2c -> 2c, k=4, s=2, p=1) + ReLU )    32^3 -> 16^3 -> 8^3 -> 4^3
//   ResidualBlock3D(256 -> 512) at 4^3 -> Conv3d(512 -> 512, k=4, p=0) + ReLU -> Flatten -> fc_mu, fc_logvar
// * ResidualBlock3D with cin != cout: relu(bn2(conv2(relu(bn1(conv1 x)))) + downsample(x)), downsample a biased 1x1 Conv3d.
//   The 1x1 weights sit in conv2's shortcut K columns (read from the block input at offset 0), their bias joins conv2's folded bias.
// * Conv3d(k=4, s=2, p=1): output o reads input 2o - 1 + k.  The GEMM runs over the OUTPUT grid with 64 taps (K = 64 * Cin, no
//   zero MACs); tap k's A tile is ONE 5-D TMA load through a map whose box steps 2 input voxels per element (elementStrides 2 on
//   w, h, d), started at input voxel 2o - 1 + k; the borders fall into TMA's zero fill.  The 64-channel layer (encoder.3) runs
//   on the tap-grouped kernel: taps kh and kh + 2 read the same box one line apart.
// * The 32-channel input of encoder.2 is stored dense ([voxel][32]); its maps have 32 channels and the 64-channel box zero-fills
//   channels 32..63, so conv1 and the shortcut see cin_pad = 64 with half of their weight columns zero.
// * encoder.12 sees the 4^3 x 512 activation as one [B, 32768] row per sample (channels-last columns, host-permuted weight):
//   an fp32 CUDA-core GEMM with a fixed 16-way K split (batch-independent summation order), then fc_mu / fc_logvar.
// =====================================================================================================================
namespace {
constexpr int kEncSplits = 16;     // K splits of encoder.12 (32768 / 16 = 2048 per split): fixed, so a sample's result is batch-independent
constexpr int kEncFlat = 64 * 512;
}  // namespace

namespace pcd {
cudaError_t launch_vae3d_first_conv(const float* vox, long long nvox_total, const float* w, const float* bias, void* hi, void* lo,
                                    int f16, cudaStream_t s);
}

struct pcd_vae3d_encoder : ConvNet {
    int latent = 256;
    float *w0 = nullptr, *b0 = nullptr;       // encoder.0: [27][32] tap-major, [32]
    float *w12 = nullptr, *b12 = nullptr;     // encoder.12: [512][64 voxels x 512 channels], [512]
    float *wmu = nullptr, *bmu = nullptr, *wlv = nullptr, *blv = nullptr;   // fc_mu / fc_logvar: [latent][512], [latent]
    PlanCache<int, VPlan> plans;              // VPlan::lin = [B][32768] flattened 4^3 input of encoder.12, then the split-K partial
                                              // sums [16][B][512] and encoder.12's output [B][512]
};

// Conv3d(cin -> cout, k=3 p=1 or k=4 s=2 p=1) + BatchNorm3d (bn non-empty) + 1x1 `downsample` shortcut of a res_cin-channel block
// input (ds non-empty).  G = output grid edge; in_ld / res_ld: channels per voxel of the input / shortcut source in memory.
static int add_enc_conv(ConvNet* h, const TensorTable& tt, const std::string& conv, const std::string& bn, const std::string& ds, int seq,
                        int cin, int cout, int k, int G, int in_ld, int res_cin, int res_ld) {
    std::string err;
    const int kk = k * k * k;
    const float *w, *b, *wd = nullptr, *bd = nullptr;
    if (!fetch(tt, conv + ".weight", 1LL * kk * cin * cout, &w, &err) || !fetch(tt, conv + ".bias", cout, &b, &err)) return fail(err);
    if (!ds.empty() && (!fetch(tt, ds + ".weight", 1LL * res_cin * cout, &wd, &err) || !fetch(tt, ds + ".bias", cout, &bd, &err)))
        return fail(err);
    std::vector<double> s(cout, 1.0), t(cout, 0.0);
    if (!bn.empty() && !bn_fold(tt, bn, cout, &s, &t, &err)) return fail(err);
    ConvW L;
    L.seq = seq; L.name = conv; L.residual = !ds.empty(); L.stride = k == 4 ? 2 : 1;
    L.W = L.H = L.D = G;
    L.cin_pad = pad64(cin); L.cout_pad = pad64(cout); L.in_ld = in_ld;
    L.out_ld = L.cout_pad; L.out_c = cout; L.out_rows = G * G * G;
    L.flops = 2.0 * kk * cin * cout * G * G * G + (L.residual ? 2.0 * res_cin * cout * G * G * G : 0.0);
    std::vector<Tap> taps;
    for (int kd = 0; kd < k; ++kd)
        for (int kh = 0; kh < k; ++kh)
            for (int kw = 0; kw < k; ++kw) {           // both forms: out[o] += w[k] * in[stride * o + k - 1]
                Tap tp; tp.dd = kd - 1; tp.dh = kh - 1; tp.dw = kw - 1;
                tp.w.assign(static_cast<size_t>(L.cout_pad) * L.cin_pad, 0.f);
                for (int co = 0; co < cout; ++co)
                    for (int ci = 0; ci < cin; ++ci)   // nn.Conv3d weight [cout][cin][kd][kh][kw], BN scale folded
                        tp.w[static_cast<size_t>(co) * L.cin_pad + ci] =
                            static_cast<float>(s[co] * w[(static_cast<size_t>(co) * cin + ci) * kk + (kd * k + kh) * k + kw]);
                taps.push_back(std::move(tp));
            }
    std::vector<float> bm(L.cout_pad, 0.f), rw;
    for (int co = 0; co < cout; ++co) bm[co] = static_cast<float>(s[co] * b[co] + t[co] + (bd ? bd[co] : 0.0));
    if (L.residual) {
        L.res_pad = pad64(res_cin); L.res_ld = res_ld;
        rw.assign(static_cast<size_t>(L.cout_pad) * L.res_pad, 0.f);
        for (int co = 0; co < cout; ++co)
            for (int ci = 0; ci < res_cin; ++ci) rw[static_cast<size_t>(co) * L.res_pad + ci] = wd[static_cast<size_t>(co) * res_cin + ci];
    }
    return pack_conv(h, L, taps, bm, L.residual ? &rw : nullptr);
}

extern "C" int pcd_vae3d_encoder_destroy(pcd_vae3d_encoder* h);

extern "C" int pcd_vae3d_encoder_create(const pcd_named_tensor* tensors, int32_t n_tensors, int32_t precision, int32_t device,
                                        pcd_vae3d_encoder** out) {
    REQ(tensors && out, "null argument");
    REQ(precision == PCD_PRECISION_BF16 || precision == PCD_PRECISION_BF16X3 || precision == PCD_PRECISION_F16 ||
            precision == PCD_PRECISION_F16MIX,
        "pcd_vae3d_encoder: precision must be bf16, bf16x3, f16 or f16mix (= fp16 hi+lo planes on every layer)");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
        return fail("pcd: no CUDA device available -- this library has no CPU fallback");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    REQ(prop.major == 10, "the tcgen05 path requires an sm_100-class GPU (B200)");
    CU(configure_gemm_tc());
    CU(configure_conv3d_tc());

    TensorTable tt;
    for (int i = 0; i < n_tensors; ++i) tt.m[tensors[i].name] = &tensors[i];
    std::string err;
    auto h = std::unique_ptr<pcd_vae3d_encoder>(new pcd_vae3d_encoder());
    h->precision = precision; h->device = device; h->num_sms = prop.multiProcessorCount;
    h->f16 = (precision == PCD_PRECISION_F16 || precision == PCD_PRECISION_F16MIX) ? 1 : 0;
    h->planes = (precision == PCD_PRECISION_BF16X3 || precision == PCD_PRECISION_F16MIX) ? 2 : 1;

    {   // encoder.0: [32][1][27] -> tap-major [27][32]
        const float *w, *b;
        if (!fetch(tt, "vae.encoder.0.weight", 27 * 32, &w, &err) || !fetch(tt, "vae.encoder.0.bias", 32, &b, &err)) return fail(err);
        std::vector<float> wf(27 * 32);
        for (int co = 0; co < 32; ++co)
            for (int tap = 0; tap < 27; ++tap) wf[tap * 32 + co] = w[co * 27 + tap];
        if (vup(h.get(), wf, &h->w0) || vup(h.get(), std::vector<float>(b, b + 32), &h->b0)) return 1;
    }
    {   // fc_mu / fc_logvar (networks.py:2243-2244) fix the latent width
        const pcd_named_tensor* t = tt.get("vae.fc_mu.weight", &err);
        if (!t) return fail(err);
        REQ(t->ndim == 2 && t->shape[1] == 512 && t->shape[0] > 0, "vae.fc_mu.weight must be [latent, 512]");
        h->latent = static_cast<int>(t->shape[0]);
        const float *wm, *bm, *wl, *bl;
        const long long n = 512LL * h->latent;
        if (!fetch(tt, "vae.fc_mu.weight", n, &wm, &err) || !fetch(tt, "vae.fc_mu.bias", h->latent, &bm, &err) ||
            !fetch(tt, "vae.fc_logvar.weight", n, &wl, &err) || !fetch(tt, "vae.fc_logvar.bias", h->latent, &bl, &err))
            return fail(err);
        if (vup(h.get(), std::vector<float>(wm, wm + n), &h->wmu) || vup(h.get(), std::vector<float>(bm, bm + h->latent), &h->bmu) ||
            vup(h.get(), std::vector<float>(wl, wl + n), &h->wlv) || vup(h.get(), std::vector<float>(bl, bl + h->latent), &h->blv))
            return 1;
    }
    // residual blocks and strided convs (networks.py:2210-2241): block (seqR, c -> 2c) at grid G, then seqS (2c -> 2c) to G / 2
    struct Stage { int seqR, cin, G, seqS; };
    const Stage stages[4] = {{2, 32, 32, 3}, {5, 64, 16, 6}, {8, 128, 8, 9}, {11, 256, 4, 12}};
    for (const Stage& st : stages) {
        const std::string n = "vae.encoder." + std::to_string(st.seqR);
        const int c = 2 * st.cin;               // the block input is stored with st.cin channels per voxel (encoder.0: dense 32)
        if (add_enc_conv(h.get(), tt, n + ".conv1", n + ".bn1", "", st.seqR, st.cin, c, 3, st.G, st.cin, 0, 0)) return 1;
        if (add_enc_conv(h.get(), tt, n + ".conv2", n + ".bn2", n + ".downsample", st.seqR, c, c, 3, st.G, c, st.cin, st.cin)) return 1;
        if (st.seqS == 12) break;
        const std::string m = "vae.encoder." + std::to_string(st.seqS);
        if (add_enc_conv(h.get(), tt, m, "", "", st.seqS, c, c, 4, st.G / 2, c, 0, 0)) return 1;
    }
    {   // encoder.12: [512][512][4][4][4] -> [co][(voxel, ci)], the channels-last order of the flattened 4^3 grid
        const float *w, *b;
        if (!fetch(tt, "vae.encoder.12.weight", 512LL * kEncFlat, &w, &err) || !fetch(tt, "vae.encoder.12.bias", 512, &b, &err))
            return fail(err);
        std::vector<float> wp(static_cast<size_t>(512) * kEncFlat);
        for (int co = 0; co < 512; ++co)
            for (int ci = 0; ci < 512; ++ci)
                for (int v = 0; v < 64; ++v)
                    wp[static_cast<size_t>(co) * kEncFlat + v * 512 + ci] = w[(static_cast<size_t>(co) * 512 + ci) * 64 + v];
        if (vup(h.get(), wp, &h->w12) || vup(h.get(), std::vector<float>(b, b + 512), &h->b12)) return 1;
    }
    CU(cudaDeviceSynchronize());
    *out = h.release();
    return 0;
}

extern "C" int pcd_vae3d_encoder_destroy(pcd_vae3d_encoder* h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    h->plans.clear();
    for (void* p : h->owned) cudaFree(p);
    delete h;
    return 0;
}

static int build_eplan(pcd_vae3d_encoder* h, int B, VPlan** out) {
    if (VPlan* hit = h->plans.find(B)) { *out = hit; return 0; }
    h->plans.make_room();
    auto pl = std::unique_ptr<VPlan>(new VPlan());
    pl->B = B; pl->Bpad = (B + 1) / 2 * 2;          // a 128-row tile of the 4^3 grid spans two samples
    const int Bp = pl->Bpad;
    const size_t buf_bytes = static_cast<size_t>(h->planes) * Bp * kVox * 64 * 2;   // largest grid: 32^3 x 64 channels
    for (int i = 0; i < 3; ++i) {
        CU(cudaMalloc(&pl->buf[i], buf_bytes));
        pl->owned.push_back(pl->buf[i]);
        CU(cudaMemset(pl->buf[i], 0, buf_bytes));
    }
    void* p = nullptr;
    CU(cudaMalloc(&p, sizeof(float) * B * (kEncFlat + (kEncSplits + 1) * 512)));
    pl->owned.push_back(p); pl->lin = static_cast<float*>(p);
    // buffer rotation as in the decoder: encoder.0 writes buffer 0
    int cur = 0, res_in = 0;
    auto free_buf = [&](int x, int y) { for (int i = 0; i < 3; ++i) if (i != x && i != y) return i; return -1; };
    for (const ConvW& L : h->convs) {
        const int src = cur, dst = L.residual ? free_buf(cur, res_in) : free_buf(cur, cur);
        GemmOp op;
        if (make_conv_op(h, L, pl->buf[src], pl->buf[res_in], pl->buf[dst], Bp, &op)) return 1;
        pl->ops.push_back(op);
        pl->out_buf.push_back(dst);
        if (!L.residual) res_in = src;
        cur = dst;
    }
    pl->final_in = cur;
    *out = h->plans.insert(B, std::move(pl));
    return 0;
}

static int launch_enc_first(pcd_vae3d_encoder* h, VPlan* pl, const float* vox, cudaStream_t s) {
    char* hi = static_cast<char*>(pl->buf[0]);
    char* lo = h->planes == 2 ? hi + static_cast<long long>(pl->Bpad) * kVox * 32 * 2 : nullptr;
    LAUNCH(launch_vae3d_first_conv(vox, static_cast<long long>(pl->B) * kVox, h->w0, h->b0, hi, lo, h->f16, s));
    return 0;
}

// encoder.12 + ReLU -> pl->lin + B * (kEncFlat + kEncSplits * 512), [B][512]
static int launch_enc_flat(pcd_vae3d_encoder* h, VPlan* pl, cudaStream_t s) {
    const long long rows = static_cast<long long>(pl->B) * 64;
    const char* src = static_cast<const char*>(pl->buf[pl->final_in]);
    const char* lo = h->planes == 2 ? src + static_cast<long long>(pl->Bpad) * 64 * 512 * 2 : nullptr;
    float* flat = pl->lin;
    float* part = flat + static_cast<long long>(pl->B) * kEncFlat;
    float* hid = part + static_cast<long long>(kEncSplits) * pl->B * 512;
    LAUNCH(launch_rows16_to_f32(src, lo, 512, flat, 512, rows, h->f16, s));
    SimtGemmParams p{};
    p.A0 = flat; p.lda0 = kEncFlat; p.K0 = kEncFlat; p.A1 = nullptr; p.lda1 = 0; p.K1 = 0;
    p.W = h->w12; p.ldw = kEncFlat; p.M = pl->B; p.Nout = 512; p.out = hid; p.ldo = 512;
    p.bias = nullptr; p.bias_sample_stride = 0; p.rows_per_sample = 1 << 30; p.relu = 0;
    p.partial = part; p.splits = kEncSplits;
    LAUNCH(launch_gemm_simt(EPI_STORE, p, s));
    LAUNCH(launch_splitk_reduce(part, kEncSplits, h->b12, hid, pl->B, 512, 1, s));
    return 0;
}

static const float* enc_hidden(const VPlan* pl) { return pl->lin + static_cast<long long>(pl->B) * (kEncFlat + kEncSplits * 512); }

// fc_mu, fc_logvar (fp32 CUDA-core GEMMs on encoder.12's output)
static int launch_enc_heads(pcd_vae3d_encoder* h, VPlan* pl, float* mu, float* logvar, cudaStream_t s) {
    for (int i = 0; i < 2; ++i) {
        SimtGemmParams p{};
        p.A0 = enc_hidden(pl); p.lda0 = 512; p.K0 = 512; p.A1 = nullptr; p.lda1 = 0; p.K1 = 0;
        p.W = i == 0 ? h->wmu : h->wlv; p.ldw = 512; p.M = pl->B; p.Nout = h->latent; p.out = i == 0 ? mu : logvar; p.ldo = h->latent;
        p.bias = i == 0 ? h->bmu : h->blv; p.bias_sample_stride = 0; p.rows_per_sample = 1 << 30; p.relu = 0;
        p.partial = nullptr; p.splits = 1;
        LAUNCH(launch_gemm_simt(EPI_STORE, p, s));
    }
    return 0;
}

extern "C" int pcd_vae3d_encode(pcd_vae3d_encoder* h, const float* vox, float* mu, float* logvar, int32_t B, void* stream) {
    REQ(B > 0, "B must be positive");
    REQ(h && vox && mu && logvar, "null argument");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    VPlan* pl = nullptr;
    if (build_eplan(h, B, &pl)) return 1;
    if (launch_enc_first(h, pl, vox, s)) return 1;
    for (const GemmOp& op : pl->ops)
        if (launch_op(h, op, s)) return 1;
    if (launch_enc_flat(h, pl, s)) return 1;
    return launch_enc_heads(h, pl, mu, logvar, s);
}

extern "C" int pcd_vae3d_encoder_tap(pcd_vae3d_encoder* h, const float* vox, int32_t B, int32_t seq_index, float* out_host, int64_t count,
                                     void* stream) {
    REQ(B > 0, "B must be positive");
    REQ(h && vox && out_host, "null argument");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    VPlan* pl = nullptr;
    if (build_eplan(h, B, &pl)) return 1;
    if (launch_enc_first(h, pl, vox, s)) return 1;
    if (seq_index == 12) {
        for (const GemmOp& op : pl->ops)
            if (launch_op(h, op, s)) return 1;
        if (launch_enc_flat(h, pl, s)) return 1;
        REQ(count == 512LL * B, "pcd_vae3d_encoder_tap: count must be B * 512 for encoder.12");
        CU(cudaMemcpyAsync(out_host, enc_hidden(pl), sizeof(float) * count, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        return 0;
    }
    int last = -1;
    if (seq_index != 0) {
        for (size_t i = 0; i < pl->ops.size(); ++i) {
            if (pl->ops[i].L->seq > seq_index) break;
            if (launch_op(h, pl->ops[i], s)) return 1;
            last = static_cast<int>(i);
        }
        REQ(last >= 0 && pl->ops[last].L->seq == seq_index, "pcd_vae3d_encoder_tap: seq_index must be one of 0,2,3,5,6,8,9,11,12");
    }
    const long long vps = last < 0 ? kVox : pl->ops[last].L->out_rows;      // voxels per sample of the tapped activation
    const int creal = last < 0 ? 32 : pl->ops[last].L->out_c;
    const int ld = last < 0 ? 32 : pl->ops[last].L->out_ld;
    const void* src = last < 0 ? pl->buf[0] : pl->buf[pl->out_buf[last]];
    const long long rows = static_cast<long long>(B) * vps;
    REQ(count == rows * creal, "pcd_vae3d_encoder_tap: count must be B * G^3 * C of the tapped layer (channels-last)");
    const char* lo = h->planes == 2 ? static_cast<const char*>(src) + static_cast<long long>(pl->Bpad) * vps * ld * 2 : nullptr;
    float* tmp = nullptr;
    CU(cudaMalloc(reinterpret_cast<void**>(&tmp), sizeof(float) * count));
    LAUNCH(launch_rows16_to_f32(src, lo, ld, tmp, creal, rows, h->f16, s));
    CU(cudaMemcpyAsync(out_host, tmp, sizeof(float) * count, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    cudaFree(tmp);
    return 0;
}

extern "C" int pcd_vae3d_encoder_profile(pcd_vae3d_encoder* h, const float* vox, float* mu, float* logvar, int32_t B, float* ms_out,
                                         double* flops_out, char* names_out, int32_t name_stride, int32_t cap, int32_t* n_out,
                                         void* stream) {
    REQ(B > 0, "B must be positive");
    REQ(h && vox && mu && logvar && ms_out && flops_out && n_out, "null argument");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    VPlan* pl = nullptr;
    if (build_eplan(h, B, &pl)) return 1;
    const int n = static_cast<int>(pl->ops.size()) + 3;
    REQ(cap >= n, "pcd_vae3d_encoder_profile: cap too small");
    std::vector<cudaEvent_t> ev(n + 1);
    for (auto& e : ev) CU(cudaEventCreate(&e));
    CU(cudaEventRecord(ev[0], s));
    if (launch_enc_first(h, pl, vox, s)) return 1;
    CU(cudaEventRecord(ev[1], s));
    for (size_t i = 0; i < pl->ops.size(); ++i) {
        if (launch_op(h, pl->ops[i], s)) return 1;
        CU(cudaEventRecord(ev[i + 2], s));
    }
    if (launch_enc_flat(h, pl, s)) return 1;
    CU(cudaEventRecord(ev[n - 1], s));
    if (launch_enc_heads(h, pl, mu, logvar, s)) return 1;
    CU(cudaEventRecord(ev[n], s));
    CU(cudaStreamSynchronize(s));
    for (int i = 0; i < n; ++i) {
        CU(cudaEventElapsedTime(&ms_out[i], ev[i], ev[i + 1]));
        std::string name; double fl = 0;
        if (i == 0) { name = "encoder.0"; fl = 2.0 * 27 * 32 * kVox * B; }
        else if (i == n - 2) { name = "encoder.12"; fl = 2.0 * kEncFlat * 512 * B; }
        else if (i == n - 1) { name = "fc_mu+fc_logvar"; fl = 2.0 * 2 * 512 * h->latent * B; }
        else { name = pl->ops[i - 1].L->name.substr(4); fl = pl->ops[i - 1].L->flops * B; }
        flops_out[i] = fl;
        if (names_out && name_stride > 0) {
            std::strncpy(names_out + static_cast<size_t>(i) * name_stride, name.c_str(), name_stride - 1);
            names_out[static_cast<size_t>(i) * name_stride + name_stride - 1] = 0;
        }
    }
    for (auto& e : ev) cudaEventDestroy(e);
    *n_out = n;
    return 0;
}
