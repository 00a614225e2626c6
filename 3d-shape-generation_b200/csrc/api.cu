// C ABI (include/pcd_b200.h): weight preparation, per-(B,N) execution plan, CUDA-graph step loop.
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include <cuda.h>
#include <cuda_runtime.h>

#include "../../include/pcd_b200.h"
#include "api_common.h"
#include "pcd_launch.h"
#include "pcd_types.h"

using namespace pcd;

// ------------------------------------------------------------------------------------------
// error plumbing (macros and helpers in api_common.h)
// ------------------------------------------------------------------------------------------
thread_local std::string g_pcd_err;
std::atomic<long long> g_pcd_launches{0};

extern "C" int pcd_abi_version(void) { return PCD_ABI_VERSION; }
extern "C" const char* pcd_last_error(void) { return g_pcd_err.c_str(); }
extern "C" int64_t pcd_launch_count(void) { return g_pcd_launches.load(); }

// ------------------------------------------------------------------------------------------
// TMA descriptor creation through the driver entry point (no link-time libcuda dependency, so
// the library also loads on a CPU-only box)
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;

static int get_encode() {
    if (g_encode) return 0;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    CU(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    REQ(fn != nullptr && q == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available");
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
    return 0;
}

// 16-bit channels-last grid [nb][D][H][W][C] seen through arbitrary element strides (sw, sh, sd, sb; channel stride 1):
// box = 64 channels x (bw, bh, bd, bb) voxels, 128B swizzle, zero fill outside the extents (= convolution padding)
int make_tmap5(CUtensorMap* tm, const void* base, int C, int W, int H, int D, long long nb, long long sw, long long sh,
               long long sd, long long sb, int bw, int bh, int bd, int bb, int es) {
    if (get_encode()) return 1;
    cuuint64_t gdim[5] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H),
                          static_cast<cuuint64_t>(D), static_cast<cuuint64_t>(nb)};
    cuuint64_t gstr[4] = {static_cast<cuuint64_t>(sw * 2), static_cast<cuuint64_t>(sh * 2), static_cast<cuuint64_t>(sd * 2),
                          static_cast<cuuint64_t>(sb * 2)};
    // es > 1: the box steps es voxels per element along w, h and d (TMA loads boxDim / es elements, so boxDim = count * es)
    cuuint32_t box[5] = {64u, static_cast<cuuint32_t>(bw * es), static_cast<cuuint32_t>(bh * es), static_cast<cuuint32_t>(bd * es),
                         static_cast<cuuint32_t>(bb)};
    cuuint32_t estr[5] = {1u, static_cast<cuuint32_t>(es), static_cast<cuuint32_t>(es), static_cast<cuuint32_t>(es), 1u};
    CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(base), gdim, gstr, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled (5-D) failed, CUresult=" + std::to_string(static_cast<int>(r)));
    return 0;
}

// 16-bit row-major [rows, cols] (row stride ld elements), box = 32 columns x 32 rows, 64B swizzle: the store map of the eight-warp epilogue
int make_tmap_out32(CUtensorMap* tm, const void* base, long long rows, long long cols, long long ld) {
    if (get_encode()) return 1;
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    cuuint64_t gstr[1] = {static_cast<cuuint64_t>(ld * 2)};
    cuuint32_t box[2] = {32u, 32u};
    cuuint32_t estr[2] = {1u, 1u};
    CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled (store, 32 x 32) failed, CUresult=" + std::to_string(static_cast<int>(r)));
    return 0;
}

// bf16 row-major [rows, cols] (row stride ld elements), box = 64 columns x box_rows rows, 128B swizzle
int make_tmap(CUtensorMap* tm, const void* base, long long rows, long long cols, long long ld, int box_rows) {
    if (get_encode()) return 1;
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    cuuint64_t gstr[1] = {static_cast<cuuint64_t>(ld * 2)};
    cuuint32_t box[2] = {64u, static_cast<cuuint32_t>(box_rows)};
    cuuint32_t estr[2] = {1u, 1u};
    CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed, CUresult=" + std::to_string(static_cast<int>(r)));
    return 0;
}

// ------------------------------------------------------------------------------------------
// weights
// ------------------------------------------------------------------------------------------
struct DevLayer {
    int cout = 0, k = 0;
    float* w32 = nullptr;   // [cout][k] fp32
    void* w16 = nullptr;    // [planes * cout][k] 16-bit: hi plane, lo plane (split modes), e5m2 byte plane (fp8-corrected layers)
    int wplanes = 1;
    float* b = nullptr;     // [cout]
};

// conv (k=1) followed by eval-mode BatchNorm1d folded into one affine map (networks.py:46-48):
//   y = (W x + b - mu) * gamma / sqrt(var + eps) + beta  =  (s*W) x + (s*(b - mu) + beta)
bool fold_conv_bn(const TensorTable& tt, const std::string& conv, const std::string& bn, int cout, int cin,
                  HostMat* out, std::string* err) {
    const float *w, *b;
    if (!fetch(tt, conv + ".weight", 1LL * cout * cin, &w, err)) return false;
    if (!fetch(tt, conv + ".bias", cout, &b, err)) return false;
    out->cout = cout; out->k = cin;
    out->w.resize(1LL * cout * cin); out->b.resize(cout);
    if (bn.empty()) {
        std::memcpy(out->w.data(), w, sizeof(float) * cout * cin);
        std::memcpy(out->b.data(), b, sizeof(float) * cout);
        return true;
    }
    const float *g, *beta, *mu, *var;
    if (!fetch(tt, bn + ".weight", cout, &g, err) || !fetch(tt, bn + ".bias", cout, &beta, err) ||
        !fetch(tt, bn + ".running_mean", cout, &mu, err) || !fetch(tt, bn + ".running_var", cout, &var, err))
        return false;
    for (int c = 0; c < cout; ++c) {
        const double s = static_cast<double>(g[c]) / std::sqrt(static_cast<double>(var[c]) + 1e-5);
        for (int k = 0; k < cin; ++k) out->w[1LL * c * cin + k] = static_cast<float>(s * w[1LL * c * cin + k]);
        out->b[c] = static_cast<float>(s * (static_cast<double>(b[c]) - mu[c]) + beta[c]);
    }
    return true;
}

enum LayerId {
    L_E1C2, L_E1C3, L_E2C1, L_E2C2, L_E2C3, L_E3C1, L_E3C2, L_E3C3, L_E4C1, L_E4C2, L_E4C3, L_G0, L_G3,
    L_D4C1, L_D4C2, L_D4C3, L_D3C1, L_D3C2, L_D3C3, L_D2C1, L_D2C2, L_D2C3, L_D1C1, L_D1C2, L_D1C3, L_O0, L_COUNT
};

struct Plan;

struct pcd_denoiser {
    int precision = 0, device = 0, num_sms = 148;
    int T = 256;       // dim == time_dim of the checkpoint (networks.py:737-744): width of the time MLP and of enc1.conv1's temb columns
    int f16 = 0;       // 16-bit format of weights/activations: 0 = bf16, 1 = fp16
    int planes = 1;    // 2 = every 16-bit tensor carries a hi and a lo plane (split operands, 3 MMAs per k-step)
    bool single_pass[L_COUNT] = {};   // f16mix only: layers that still run ONE pass on the hi planes (kMixSinglePass)
    bool c8[L_COUNT] = {};            // f16mix only: split layers whose two correction terms run as ONE fp8 (e5m2) pass (gemm_tc.cu NP == 4);
                                      // their weights carry a third plane (the e5m2 byte plane) and their inputs' second plane is a byte plane
    bool taps = false;
    // GEMM layers in execution order (index constants below)
    std::vector<DevLayer> L;
    // small fp32 pieces
    float *freqs = nullptr, *W1T = nullptr, *b1 = nullptr, *W2T = nullptr, *b2 = nullptr;
    float *WtT = nullptr, *bt = nullptr;     // hoisted time columns of enc1.conv1, transposed [256][64]
    float* Wx = nullptr;                     // xyz columns of enc1.conv1 [64][3]
    float *Wg = nullptr, *bg = nullptr;      // hoisted global-feature columns of dec4.conv1 [1024][4096] + folded bias
    float *w3 = nullptr, *b3 = nullptr;      // output.3
    PlanCache<std::pair<int, int>, Plan> plans;
    std::vector<void*> owned;
};


template <typename T>
static int dev_upload(pcd_denoiser* h, const std::vector<T>& v, T** out) {
    void* p = nullptr;
    CU(cudaMalloc(&p, v.size() * sizeof(T)));
    h->owned.push_back(p);
    CU(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    *out = static_cast<T*>(p);
    return 0;
}

static int upload_layer(pcd_denoiser* h, const HostMat& m, DevLayer* d, bool c8 = false) {
    d->cout = m.cout; d->k = m.k;
    if (dev_upload(h, m.w, &d->w32)) return 1;
    if (dev_upload(h, m.b, &d->b)) return 1;
    void* p = nullptr;
    const int planes = h->planes + (c8 ? 1 : 0);
    d->wplanes = planes;
    CU(cudaMalloc(&p, m.w.size() * 2 * planes));
    h->owned.push_back(p);
    d->w16 = p;
    if (h->planes == 2)   // [2*cout][k]: hi plane, then the 16-bit residual plane
        LAUNCH(launch_f32_split_16(d->w32, d->w16, static_cast<char*>(d->w16) + m.w.size() * 2, static_cast<long long>(m.w.size()), h->f16, 0));
    else
        LAUNCH(launch_f32_to_16(d->w32, d->w16, static_cast<long long>(m.w.size()), h->f16, 0));
    if (c8)               // third plane: e5m2 copies of hi and lo, laid out as the K = 128 rows of the fp8 correction pass
        LAUNCH(launch_f32_split_c8(d->w32, d->w16, static_cast<char*>(d->w16) + m.w.size() * 4, m.cout, m.k, 0));
    return 0;
}

// ---- which second plane does a layer's output need?  (1 = none, 2 = 16-bit residual, 3 = e5m2 byte plane)
// consumers of every GEMM layer's output in the U-Net (networks.py:799-816)
static const int kConsumers[L_COUNT][2] = {
    /*E1C2*/ {L_E1C3, -1}, /*E1C3*/ {L_E2C1, L_D1C1}, /*E2C1*/ {L_E2C2, -1}, /*E2C2*/ {L_E2C3, -1}, /*E2C3*/ {L_E3C1, L_D2C1},
    /*E3C1*/ {L_E3C2, -1}, /*E3C2*/ {L_E3C3, -1}, /*E3C3*/ {L_E4C1, L_D3C1}, /*E4C1*/ {L_E4C2, -1}, /*E4C2*/ {L_E4C3, -1},
    /*E4C3*/ {L_G0, L_D4C1}, /*G0*/ {L_G3, -1}, /*G3*/ {-1, -1}, /*D4C1*/ {L_D4C2, -1}, /*D4C2*/ {L_D4C3, -1}, /*D4C3*/ {L_D3C1, -1},
    /*D3C1*/ {L_D3C2, -1}, /*D3C2*/ {L_D3C3, -1}, /*D3C3*/ {L_D2C1, -1}, /*D2C1*/ {L_D2C2, -1}, /*D2C2*/ {L_D2C3, -1},
    /*D2C3*/ {L_D1C1, -1}, /*D1C1*/ {L_D1C2, -1}, /*D1C2*/ {L_D1C3, -1}, /*D1C3*/ {L_O0, -1}, /*O0*/ {-1, -1}};

// f16mix: global_feat.0 / global_feat.3 hold 67 % of the FLOPs and each contributes only ~3-4.5e-4 relative error when run as ONE
// fp16 pass (measured per layer against the fp32 oracle); dec4.conv1 (6.7 % of the FLOPs, ~3.6e-4) as well: eps error 4.7e-4 ->
// ~6e-4, step time -8 %.  Everything else stays split (3 passes).
static const int kMixSinglePass[] = {L_G0, L_G3, L_D4C1};
// f16mix: the tensor-bound split layers (K >= 512: enc4.*, dec4.conv2/3, dec3.*; 46 % of the split-mode step) run their two correction
// terms as one fp8 pass: 2 pass-equivalents instead of 3.  Every one has cout >= 256: the fp8 form needs 256-column pair-MMA tiles.
static const int kMixC8[] = {L_E4C1, L_E4C2, L_E4C3, L_D4C2, L_D4C3, L_D3C1, L_D3C2, L_D3C3};

// pass structure of a layer in a plan: 1 = one pass on the hi planes, 3 = split (hi*hi + hi*lo + lo*hi), 4 = hi*hi + one fp8 pass
static int layer_np(const pcd_denoiser* h, int layer, bool plan_c8) {
    if (h->planes != 2 || h->single_pass[layer]) return 1;
    return (plan_c8 && h->c8[layer]) ? 4 : 3;
}
// -1 = the consumers disagree (a tensor has ONE second plane)
static int out_format(const pcd_denoiser* h, int layer, bool plan_c8) {
    int fmt = 1;
    for (int c : kConsumers[layer]) {
        if (c < 0) continue;
        const int np = layer_np(h, c, plan_c8);
        const int want = np == 1 ? 1 : (np == 4 ? 3 : 2);
        if (want == 1) continue;
        if (fmt != 1 && fmt != want) return -1;
        fmt = want;
    }
    return fmt;
}

// P[cout][cs] = Wskip[cout][cs] * Wr[cs][cs]  computed on the GPU in fp32 (networks.py:811-814:
// decK.conv1 applied to refineK(x_k) == (WdecK[:, skip] * WrK) x_k + WdecK[:, skip] * brK)
static int compose_on_gpu(const std::vector<float>& wskip, int cout, int cs, const std::vector<float>& wr,
                          std::vector<float>* out) {
    std::vector<float> wrT(1LL * cs * cs);
    for (int i = 0; i < cs; ++i)
        for (int j = 0; j < cs; ++j) wrT[1LL * j * cs + i] = wr[1LL * i * cs + j];
    float *dA = nullptr, *dW = nullptr, *dO = nullptr;
    CU(cudaMalloc(&dA, sizeof(float) * cout * cs));
    CU(cudaMalloc(&dW, sizeof(float) * cs * cs));
    CU(cudaMalloc(&dO, sizeof(float) * cout * cs));
    CU(cudaMemcpy(dA, wskip.data(), sizeof(float) * cout * cs, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dW, wrT.data(), sizeof(float) * cs * cs, cudaMemcpyHostToDevice));
    SimtGemmParams p{};
    p.A0 = dA; p.lda0 = cs; p.K0 = cs; p.A1 = nullptr; p.lda1 = 0; p.K1 = 0;
    p.W = dW; p.ldw = cs; p.M = cout; p.Nout = cs; p.out = dO; p.ldo = cs;
    p.bias = nullptr; p.bias_sample_stride = 0; p.rows_per_sample = 1 << 30; p.relu = 0;
    LAUNCH(launch_gemm_simt(EPI_STORE, p, 0));
    out->resize(1LL * cout * cs);
    CU(cudaMemcpy(out->data(), dO, sizeof(float) * cout * cs, cudaMemcpyDeviceToHost));
    cudaFree(dA); cudaFree(dW); cudaFree(dO);
    return 0;
}

extern "C" int pcd_denoiser_destroy(pcd_denoiser* h);

extern "C" int pcd_denoiser_create(const pcd_named_tensor* tensors, int32_t n_tensors, int32_t precision,
                                   int32_t device, pcd_denoiser** out) {
    REQ(tensors && out, "null argument");
    REQ(precision >= PCD_PRECISION_BF16 && precision <= PCD_PRECISION_F16MIX, "unknown precision");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
        return fail("pcd: no CUDA device available -- this library has no CPU fallback");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (precision != PCD_PRECISION_FP32) {
        REQ(prop.major == 10, "bf16 (tcgen05) path requires an sm_100-class GPU (B200)");
        CU(configure_gemm_tc());
        CU(configure_chain_tc());
    }

    TensorTable tt;
    for (int i = 0; i < n_tensors; ++i) tt.m[tensors[i].name] = &tensors[i];
    std::string err;
    auto h = std::unique_ptr<pcd_denoiser>(new pcd_denoiser());
    h->precision = precision; h->device = device; h->num_sms = prop.multiProcessorCount;
    h->f16 = (precision == PCD_PRECISION_F16 || precision == PCD_PRECISION_F16MIX) ? 1 : 0;
    h->planes = (precision == PCD_PRECISION_BF16X3 || precision == PCD_PRECISION_F16MIX) ? 2 : 1;
    if (precision == PCD_PRECISION_F16MIX) {
        for (int l : kMixSinglePass) h->single_pass[l] = true;
        for (int l : kMixC8) h->c8[l] = true;
    }
    h->taps = std::getenv("PCD_TAPS") != nullptr;
    h->L.resize(L_COUNT);

#define FOLD(dst, conv, bn, co, ci) \
    HostMat dst;                    \
    if (!fold_conv_bn(tt, conv, bn, co, ci, &dst, &err)) return fail(err)

    // ---- time MLP (networks.py:737-741).  The reference only works for dim == time_dim (time_mlp emits `dim`, enc1 expects
    // 3 + time_dim input channels, :738-744); that width T is read off the checkpoint.  Nothing else in the network depends on it.
    {
        const pcd_named_tensor* t0 = tt.get("model.time_mlp.0.weight", &err);
        if (!t0) return fail(err);
        REQ(t0->ndim == 2 && t0->shape[0] == t0->shape[1], "model.time_mlp.0.weight must be square: the architecture needs dim == time_dim");
        REQ(t0->shape[0] >= 4 && t0->shape[0] <= 4096, "time_dim out of range (4..4096)");
        h->T = static_cast<int>(t0->shape[0]);
    }
    const int T = h->T;
    const float *tw0, *tb0, *tw2, *tb2;
    if (!fetch(tt, "model.time_mlp.0.weight", 1LL * T * T, &tw0, &err) || !fetch(tt, "model.time_mlp.0.bias", T, &tb0, &err) ||
        !fetch(tt, "model.time_mlp.2.weight", 1LL * T * T, &tw2, &err) || !fetch(tt, "model.time_mlp.2.bias", T, &tb2, &err))
        return fail(err);
    {
        const int half = T / 2;
        std::vector<float> w1t(1LL * T * T), w2t(1LL * T * T), b1(tb0, tb0 + T), b2(tb2, tb2 + T), fr(half);
        for (int o = 0; o < T; ++o)
            for (int k = 0; k < T; ++k) { w1t[1LL * k * T + o] = tw0[1LL * o * T + k]; w2t[1LL * k * T + o] = tw2[1LL * o * T + k]; }
        // networks.py:831-833 in fp32: emb = log(10000)/(half-1); f_j = exp(j * -emb)
        const float emb = std::log(10000.0f) / static_cast<float>(half - 1);
        for (int j = 0; j < half; ++j) fr[j] = std::exp(static_cast<float>(j) * -emb);
        if (dev_upload(h.get(), w1t, &h->W1T) || dev_upload(h.get(), w2t, &h->W2T) || dev_upload(h.get(), b1, &h->b1) ||
            dev_upload(h.get(), b2, &h->b2) || dev_upload(h.get(), fr, &h->freqs))
            return 1;
    }
    // ---- enc1.conv1: split [xyz | temb] columns (networks.py:797: cat([x, t_emb]))
    {
        const int cin = 3 + T;
        FOLD(e1c1, "model.enc1.conv1", "model.enc1.bn1", 64, cin);
        std::vector<float> wx(64 * 3), wtT(static_cast<size_t>(T) * 64);
        for (int c = 0; c < 64; ++c) {
            for (int k = 0; k < 3; ++k) wx[c * 3 + k] = e1c1.w[static_cast<size_t>(c) * cin + k];
            for (int k = 0; k < T; ++k) wtT[static_cast<size_t>(k) * 64 + c] = e1c1.w[static_cast<size_t>(c) * cin + 3 + k];
        }
        if (dev_upload(h.get(), wx, &h->Wx) || dev_upload(h.get(), wtT, &h->WtT) || dev_upload(h.get(), e1c1.b, &h->bt)) return 1;
    }
    struct Spec { int id; const char* conv; const char* bn; int co, ci; };
    const Spec plain[] = {
        {L_E1C2, "model.enc1.conv2", "model.enc1.bn2", 64, 64},       {L_E1C3, "model.enc1.conv3", "model.enc1.bn3", 128, 64},
        {L_E2C1, "model.enc2.conv1", "model.enc2.bn1", 128, 128},     {L_E2C2, "model.enc2.conv2", "model.enc2.bn2", 128, 128},
        {L_E2C3, "model.enc2.conv3", "model.enc2.bn3", 256, 128},     {L_E3C1, "model.enc3.conv1", "model.enc3.bn1", 256, 256},
        {L_E3C2, "model.enc3.conv2", "model.enc3.bn2", 256, 256},     {L_E3C3, "model.enc3.conv3", "model.enc3.bn3", 512, 256},
        {L_E4C1, "model.enc4.conv1", "model.enc4.bn1", 512, 512},     {L_E4C2, "model.enc4.conv2", "model.enc4.bn2", 512, 512},
        {L_E4C3, "model.enc4.conv3", "model.enc4.bn3", 1024, 512},    {L_G0, "model.global_feat.0", "model.global_feat.1", 2048, 1024},
        {L_G3, "model.global_feat.3", "model.global_feat.4", 4096, 2048},
        {L_D4C2, "model.dec4.conv2", "model.dec4.bn2", 1024, 1024},   {L_D4C3, "model.dec4.conv3", "model.dec4.bn3", 512, 1024},
        {L_D3C2, "model.dec3.conv2", "model.dec3.bn2", 512, 512},     {L_D3C3, "model.dec3.conv3", "model.dec3.bn3", 256, 512},
        {L_D2C2, "model.dec2.conv2", "model.dec2.bn2", 256, 256},     {L_D2C3, "model.dec2.conv3", "model.dec2.bn3", 128, 256},
        {L_D1C2, "model.dec1.conv2", "model.dec1.bn2", 128, 128},     {L_D1C3, "model.dec1.conv3", "model.dec1.bn3", 64, 128},
        {L_O0, "model.output.0", "model.output.1", 64, 64},
    };
    for (const Spec& s : plain) {
        HostMat m;
        if (!fold_conv_bn(tt, s.conv, s.bn, s.co, s.ci, &m, &err)) return fail(err);
        if (upload_layer(h.get(), m, &h->L[s.id], h->c8[s.id])) return 1;
    }
    // ---- decoder conv1 layers: cat([prev, refine(skip)]) (networks.py:811-814), refine pre-composed
    struct DecSpec { int id; const char* name; const char* refine; int co, kprev, ks; };
    const DecSpec decs[] = {{L_D4C1, "model.dec4", "model.refine4", 1024, 4096, 1024},
                            {L_D3C1, "model.dec3", "model.refine3", 512, 512, 512},
                            {L_D2C1, "model.dec2", "model.refine2", 256, 256, 256},
                            {L_D1C1, "model.dec1", "model.refine1", 128, 128, 128}};
    for (const DecSpec& d : decs) {
        HostMat full, ref;
        if (!fold_conv_bn(tt, std::string(d.name) + ".conv1", std::string(d.name) + ".bn1", d.co, d.kprev + d.ks, &full, &err))
            return fail(err);
        if (!fold_conv_bn(tt, d.refine, "", d.ks, d.ks, &ref, &err)) return fail(err);
        const int kf = d.kprev + d.ks;
        std::vector<float> wskip(1LL * d.co * d.ks), comp;
        for (int c = 0; c < d.co; ++c)
            for (int k = 0; k < d.ks; ++k) wskip[1LL * c * d.ks + k] = full.w[1LL * c * kf + d.kprev + k];
        if (compose_on_gpu(wskip, d.co, d.ks, ref.w, &comp)) return 1;
        std::vector<float> bias(d.co);
        for (int c = 0; c < d.co; ++c) {
            double s = full.b[c];
            for (int k = 0; k < d.ks; ++k) s += static_cast<double>(wskip[1LL * c * d.ks + k]) * ref.b[k];
            bias[c] = static_cast<float>(s);
        }
        HostMat m;
        if (d.id == L_D4C1) {
            // global-feature columns hoisted out (they multiply a per-sample constant, networks.py:808)
            std::vector<float> wg(1LL * d.co * d.kprev);
            for (int c = 0; c < d.co; ++c)
                std::memcpy(&wg[1LL * c * d.kprev], &full.w[1LL * c * kf], sizeof(float) * d.kprev);
            if (dev_upload(h.get(), wg, &h->Wg) || dev_upload(h.get(), bias, &h->bg)) return 1;
            m.cout = d.co; m.k = d.ks; m.w = comp; m.b.assign(d.co, 0.f);
        } else {
            m.cout = d.co; m.k = kf; m.w.resize(1LL * d.co * kf); m.b = bias;
            for (int c = 0; c < d.co; ++c) {
                std::memcpy(&m.w[1LL * c * kf], &full.w[1LL * c * kf], sizeof(float) * d.kprev);
                std::memcpy(&m.w[1LL * c * kf + d.kprev], &comp[1LL * c * d.ks], sizeof(float) * d.ks);
            }
        }
        if (upload_layer(h.get(), m, &h->L[d.id], h->c8[d.id])) return 1;
    }
    // ---- output.3 (bare conv, networks.py:816)
    {
        const float *w, *b;
        if (!fetch(tt, "model.output.3.weight", 3 * 64, &w, &err) || !fetch(tt, "model.output.3.bias", 3, &b, &err)) return fail(err);
        std::vector<float> vw(w, w + 192), vb(b, b + 3);
        if (dev_upload(h.get(), vw, &h->w3) || dev_upload(h.get(), vb, &h->b3)) return 1;
    }
    CU(cudaDeviceSynchronize());
    *out = h.release();
    return 0;
}

// ------------------------------------------------------------------------------------------
// per-(B, N) plan
// ------------------------------------------------------------------------------------------
struct Op {
    enum Kind { TIME, ENC1, GEMM, MEMSET_G, DBIAS, FINAL_SIMT, ADVANCE, TAPCOPY, CHAIN } kind;
    // CHAIN
    ChainMaps cmaps{};
    ChainParams cp{};
    int chain_id = 0;          // 0: enc1 + enc2, 1: dec1 + output
    double chain_flops = 0.0;
    // GEMM
    int layer = -1, epi = EPI_STORE, bn = 0, np = 1, cl = 1, out_planes = 1, two_sm = 0;
    CUtensorMap a0, a1, b, o;
    TcGemmParams tc{};
    SimtGemmParams st{};
    // TAPCOPY
    const void* src = nullptr; void* dst = nullptr; size_t bytes = 0;
};

struct Plan {
    int B = 0, N = 0, Npad = 0;
    long long M = 0;
    int elt = 2, planes = 1;
    bool c8 = false;     // this plan runs the handle's fp8-corrected layers as such (needs CTA pairs: an even number of 128-row blocks)
    int fmtX3 = 2, fmtX4 = 2, fmtD4 = 2;   // second-plane format of the tapped tensors (2 = 16-bit residual, 3 = e5m2 byte plane)
    void *X1 = nullptr, *X2 = nullptr, *X3 = nullptr, *X4 = nullptr, *T0 = nullptr, *T1 = nullptr;
    void *tapD4 = nullptr, *tapD1 = nullptr;
    float *temb = nullptr, *bias1 = nullptr, *gmax = nullptr, *biasd4 = nullptr, *dpartial = nullptr;
    float* xstage = nullptr;   // [B, N, 3] device staging of x for the host-buffer entry (allocated on first use)
    int dsplits = 1;
    float* sched = nullptr; int sched_cap = 0;
    float *bias1_steps = nullptr, *temb_steps = nullptr; int steps_cap = 0;    // the loop's time path, one row per reverse step
    int* step = nullptr;
    CallArgs* call = nullptr;
    std::vector<Op> ops;
    int kernels_per_step = 0;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    std::vector<void*> owned;
    ~Plan() {
        if (exec) cudaGraphExecDestroy(exec);
        if (graph) cudaGraphDestroy(graph);
        for (void* p : owned) cudaFree(p);
    }
};

static int plan_alloc(Plan* pl, void** out, size_t bytes) {
    CU(cudaMalloc(out, bytes));
    pl->owned.push_back(*out);
    return 0;
}

TcShape tc_shape(int epi, int np, long long M, int cout, int K, int num_sms) {
    TcShape s;
    if (epi == EPI_MAXPOOL) {
        s.bn = (np == 1 && M % 256 == 0) ? 256 : 128;
        s.cl = (cout / 128) % 2 == 0 ? 2 : 1;
    } else {
        s.cl = (M / 128) % 2 == 0 ? 2 : 1;
        // split precision (3 passes, 2 planes): 128-column tiles, or 256-column tiles on the pair MMA where each CTA stages only half
        // of the B tile (halves the L2->SM bytes per FLOP)
        const bool wide3 = np == 4 || (np == 3 && s.cl == 2 && cout >= 256 && K >= 512);
        s.bn = np >= 3 ? (wide3 ? 256 : (cout >= 128 ? 128 : cout)) : (cout >= 256 ? 256 : cout);
        // live activation bytes under the default order: one row block (128 rows x K x planes read) per CTA.  Measured per layer
        // (profiles/tile_order_ab_r2.jsonl): n fastest wins where that set is >= 38 MB and the layer has 2..4 weight tiles
        // (dec4.conv2 in f16mix: 3.68 -> 3.10 ms); with 8 weight tiles (global_feat.0) the default order stays ahead by 1-3 %.
        const int num_n = cout / s.bn;
        const double live_mb = static_cast<double>(num_sms) * 128.0 * K * 2.0 * (np >= 3 ? 2 : 1) / (1 << 20);
        s.tile_order = (num_n >= 2 && num_n <= 4 && live_mb > 30.0) ? 1 : 0;
    }
    // pairs run the pair MMA (cta_group::2) on layers with K >= 1024, TMA multicast + per-CTA MMAs elsewhere (measured: +5-6 % on
    // K >= 1024, -15 % on K <= 512 where per-tile hand-shakes dominate)
    s.two_sm = (s.cl == 2 && K >= 1024) ? 1 : 0;
    if (np >= 3 && s.bn == 256) s.two_sm = 1;
    return s;
}

static int add_gemm(pcd_denoiser* h, Plan* pl, int layer, const void* a0, int k0, const void* a1, int k1, void* dst,
                    int epi, const float* sample_bias, long long sample_bias_stride) {
    const DevLayer& L = h->L[layer];
    Op op; op.kind = Op::GEMM; op.layer = layer; op.epi = epi;
    if (k0 + k1 != L.k) return fail("internal: K mismatch for layer " + std::to_string(layer));
    const float* bias = sample_bias ? sample_bias : L.b;
    if (h->precision == PCD_PRECISION_FP32) {
        SimtGemmParams& p = op.st;
        p.A0 = static_cast<const float*>(a0); p.lda0 = k0; p.K0 = k0;
        p.A1 = static_cast<const float*>(a1); p.lda1 = k1; p.K1 = k1;
        p.W = L.w32; p.ldw = L.k; p.M = static_cast<int>(pl->M); p.Nout = L.cout;
        p.out = static_cast<float*>(dst); p.ldo = L.cout;
        p.bias = bias; p.bias_sample_stride = sample_bias_stride; p.rows_per_sample = pl->Npad; p.relu = 1;
        p.gmax = pl->gmax; p.ld_g = 4096; p.n_valid = pl->N;
        pl->ops.push_back(op);
        return 0;
    }
    TcGemmParams& p = op.tc;
    const int PLn = pl->planes;
    const long long Mrows = pl->M * PLn;        // hi plane rows [0, M), lo plane rows [M, 2M)
    op.np = layer_np(h, layer, pl->c8);   // a single-pass layer reads (and writes) hi planes only
    p.f16 = h->f16;
    // a STORE layer writes the second plane its consumers read: nothing when every consumer is single-pass (global_feat.0 ->
    // global_feat.3, and enc4.conv3 (x4) -> global_feat.0 + dec4.conv1 in f16mix), the 16-bit residual for split consumers, the
    // e5m2 byte plane for fp8-corrected consumers
    int fmt = out_format(h, layer, pl->c8);
    if (fmt == 1 && layer == L_E4C3 && h->taps) fmt = 2;      // the x4 tap shows the split value
    op.out_planes = (PLn == 2 && epi == EPI_STORE) ? fmt : 1;
    const bool np3_one_plane = op.np == 3 && op.out_planes == 1;   // only instantiated for the wide (256-column) pair-MMA tiles
    p.kb0 = k0 / 64; p.kb1 = k1 / 64;
    p.bias = bias; p.bias_sample_stride = sample_bias_stride; p.rows_per_sample = pl->Npad; p.relu = 1;
    p.gmax = pl->gmax; p.ld_g = 4096; p.n_valid = pl->N; p.num_samples = pl->B; p.call = pl->call;
    const TcShape sh = tc_shape(epi, op.np, pl->M, L.cout, k0 + k1, h->num_sms);
    op.bn = sh.bn; op.cl = sh.cl; op.two_sm = sh.two_sm; p.tile_order = sh.tile_order;
    if (epi == EPI_MAXPOOL) {
        // weights take the A role (128 channels per tile), points the B role
        p.num_m_blocks = L.cout / 128; p.num_n_blocks = static_cast<int>(pl->M / op.bn);
        p.a_plane_rows = PLn == 2 ? L.cout : 0; p.b_plane_rows = PLn == 2 ? static_cast<int>(pl->M) : 0; p.out_plane_rows = 0;
        if (make_tmap(&op.a0, L.w16, static_cast<long long>(L.cout) * PLn, L.k, L.k, 128)) return 1;
        op.a1 = op.a0;
        if (make_tmap(&op.b, a0, Mrows, k0, k0, op.bn / op.cl)) return 1;
        op.o = op.a0;
    } else {
        p.num_m_blocks = static_cast<int>(pl->M / 128);
        p.num_n_blocks = L.cout / op.bn;
        p.out = static_cast<__nv_bfloat16*>(dst); p.ldo = L.cout;
        p.a_plane_rows = PLn == 2 ? static_cast<int>(pl->M) : 0;
        p.b_plane_rows = PLn == 2 ? (op.np == 4 ? 2 * L.cout : L.cout) : 0;     // fp8-corrected layers read the weights' third plane
        p.out_plane_rows = PLn == 2 ? static_cast<int>(pl->M) : 0;
        if (make_tmap(&op.a0, a0, Mrows, k0, k0, 128)) return 1;
        if (k1 > 0) { if (make_tmap(&op.a1, a1, Mrows, k1, k1, 128)) return 1; }
        else op.a1 = op.a0;
        if (make_tmap(&op.b, L.w16, static_cast<long long>(L.cout) * L.wplanes, L.k, L.k, op.bn / op.cl)) return 1;
        // STORE layers: two epilogue warps per TMEM lane quarter (the 32 x 32 store map)
        p.epi_warps = epi == EPI_STORE ? 8 : 4;
        if (epi == EPI_STORE) { if (make_tmap_out32(&op.o, dst, Mrows, L.cout, L.cout)) return 1; }
        else op.o = op.a0;
    }
    if (np3_one_plane && op.bn != 256) op.out_planes = 2;
    if (layer == L_E3C3) pl->fmtX3 = op.out_planes;
    if (layer == L_E4C3) pl->fmtX4 = op.out_planes;
    if (layer == L_D4C3) pl->fmtD4 = op.out_planes;
    pl->ops.push_back(op);
    return 0;
}

// A fused chain (chain_tc.cu).  `layers` in execution order; ext0 / ext1: the HBM tensors the first layer streams (or nullptr);
// outs[i]: HBM destination of layer i (nullptr: none).
struct ChainSpec { int layer; int kb_ext0, kb_ext1; bool to_act; void* out; bool final; };
static int add_chain(pcd_denoiser* h, Plan* pl, int chain_id, const std::vector<ChainSpec>& layers, const void* ext0, int c0, const void* ext1,
                     int c1, bool first_from_x) {
    Op op; op.kind = Op::CHAIN; op.chain_id = chain_id;
    ChainParams& p = op.cp;
    const int PLn = pl->planes;
    const long long Mrows = pl->M * PLn;
    p.nlayers = static_cast<int>(layers.size());
    p.num_m_blocks = static_cast<int>(pl->M / 128); p.rows_per_sample = pl->Npad;
    p.a_plane_rows = PLn == 2 ? static_cast<int>(pl->M) : 0;
    p.first_from_x = first_from_x ? 1 : 0; p.Wx = h->Wx; p.bias1 = pl->bias1; p.call = pl->call;
    int nout = 0;
    for (size_t i = 0; i < layers.size(); ++i) {
        const ChainSpec& cs = layers[i];
        const DevLayer& L = h->L[cs.layer];
        ChainLayer& cl = p.L[i];
        cl.kb = L.k / 64; cl.kb_ext0 = cs.kb_ext0; cl.kb_ext1 = cs.kb_ext1; cl.n = L.cout; cl.np = PLn == 2 ? 3 : 1;
        cl.to_act = cs.to_act ? 1 : 0; cl.to_hbm = -1; cl.final = cs.final ? 1 : 0;
        cl.bias = L.b; cl.bias_sample_stride = 0;
        if (make_tmap(&op.cmaps.w[i], L.w16, static_cast<long long>(L.cout) * L.wplanes, L.k, L.k, L.cout < 128 ? L.cout : 128)) return 1;
        if (cs.out) {
            if (make_tmap_out32(&op.cmaps.out[nout], cs.out, Mrows, L.cout, L.cout)) return 1;
            cl.to_hbm = nout++;
        }
        op.chain_flops += 2.0 * static_cast<double>(pl->M) * L.k * L.cout;
    }
    if (first_from_x) op.chain_flops += 2.0 * static_cast<double>(pl->M) * 3 * 64;
    if (ext0 && make_tmap(&op.cmaps.ext[0], ext0, Mrows, c0, c0, 128)) return 1;
    if (ext1 && make_tmap(&op.cmaps.ext[1], ext1, Mrows, c1, c1, 128)) return 1;
    pl->ops.push_back(op);
    return 0;
}

// the chains run every layer as plain one-pass or three-pass layers with 16-bit residual planes: no single-pass or fp8-corrected
// f16mix layer inside them.  They are used for plans of at most 4 row tiles per SM (batch <= 37 at 2048 points), where launch /
// drain latency dominates.
static bool chain_ok(const pcd_denoiser* h, const Plan* pl, std::initializer_list<int> layers, int last_out_layer) {
    if (h->precision == PCD_PRECISION_FP32) return false;
    // Measured (profiles/chain_fused_ab_r2.jsonl, profiles/chain_fused_timing_r2.jsonl): batch 4 gains 8-9 % (11 launches become 2), batch 64
    // is neutral, batch 512 LOSES (f16mix: 0.97 -> 1.20 ms for enc1+enc2, bf16: 0.51 -> 0.93): inside a chain a tile's epilogue and its next
    // layer's MMAs are serial, while the per-layer kernels overlap them across tiles and already run at 73-89 % of the HBM rate.
    if (pl->M / 128 > 4LL * h->num_sms) return false;
    for (int l : layers)
        if (h->single_pass[l] || h->c8[l]) return false;
    if (pl->planes == 2 && last_out_layer >= 0 && out_format(h, last_out_layer, pl->c8) != 2) return false;
    return true;
}

static void add_tapcopy(Plan* pl, const void* src, void* dst, size_t bytes) {
    Op op; op.kind = Op::TAPCOPY; op.src = src; op.dst = dst; op.bytes = bytes;
    pl->ops.push_back(op);
}

static int build_plan(pcd_denoiser* h, int B, int N, Plan** out) {
    auto key = std::make_pair(B, N);
    if (Plan* hit = h->plans.find(key)) { *out = hit; return 0; }
    h->plans.make_room();
    auto pl = std::unique_ptr<Plan>(new Plan());
    pl->B = B; pl->N = N; pl->Npad = (N + 127) / 128 * 128;
    pl->M = static_cast<long long>(B) * pl->Npad;
    REQ(pl->M < (1LL << 31), "B * N too large for one call (shard the batch)");
    pl->elt = h->precision == PCD_PRECISION_FP32 ? 4 : 2;
    pl->planes = h->planes;
    // the fp8-corrected form exists on the pair MMA only: a plan whose row blocks do not pair up runs those layers as plain split layers
    pl->c8 = h->planes == 2 && (pl->M / 128) % 2 == 0;
    const size_t e = static_cast<size_t>(pl->elt) * pl->planes, M = static_cast<size_t>(pl->M);
    if (plan_alloc(pl.get(), &pl->X1, M * 128 * e) || plan_alloc(pl.get(), &pl->X2, M * 256 * e) ||
        plan_alloc(pl.get(), &pl->X3, M * 512 * e) || plan_alloc(pl.get(), &pl->X4, M * 1024 * e) ||
        plan_alloc(pl.get(), &pl->T0, M * 2048 * e) || plan_alloc(pl.get(), &pl->T1, M * 1024 * e))
        return 1;
    if (h->taps && (plan_alloc(pl.get(), &pl->tapD4, M * 512 * e) || plan_alloc(pl.get(), &pl->tapD1, M * 64 * e))) return 1;
    void* p = nullptr;
    if (plan_alloc(pl.get(), &p, sizeof(float) * B * h->T)) return 1; pl->temb = static_cast<float*>(p);
    if (plan_alloc(pl.get(), &p, sizeof(float) * B * 64)) return 1; pl->bias1 = static_cast<float*>(p);
    if (plan_alloc(pl.get(), &p, sizeof(float) * B * 4096)) return 1; pl->gmax = static_cast<float*>(p);
    if (plan_alloc(pl.get(), &p, sizeof(float) * B * 1024)) return 1; pl->biasd4 = static_cast<float*>(p);
    // dec4's per-sample bias GEMM ([B, 4096] x [4096, 1024]) is split the SAME number of ways along K for EVERY batch size: a split count chosen
    // from the batch (simt_pick_splits) changed the fp32 summation order between batch 256 and 512, so that a sample's result
    // depended on the batch it was in (1e-3 after 50 bf16 steps; tests/test_gpu_samplers.py::test_full_size_ddim50_properties)
    // 32 splits (K = 128 per CTA): the GEMM streams 16 MB of weights behind M = B rows, so at small batch its time is the length of the
    // per-CTA k loop (27 us of a 395 us step at batch 4 with 8 splits); at batch 512 the extra partial sums cost < 0.03 ms
    pl->dsplits = 32;
    if (pl->dsplits > 1) { if (plan_alloc(pl.get(), &p, sizeof(float) * pl->dsplits * B * 1024)) return 1; pl->dpartial = static_cast<float*>(p); }
    if (plan_alloc(pl.get(), &p, sizeof(int))) return 1; pl->step = static_cast<int*>(p);
    if (plan_alloc(pl.get(), &p, sizeof(CallArgs))) return 1; pl->call = static_cast<CallArgs*>(p);
    CU(cudaMemset(pl->step, 0, sizeof(int)));

    Op op;
    op = Op(); op.kind = Op::TIME; pl->ops.push_back(op);
    void *T0 = pl->T0, *T1 = pl->T1;
#define G(layer, a0, k0, a1, k1, dst) \
    if (add_gemm(h, pl.get(), layer, a0, k0, a1, k1, dst, EPI_STORE, nullptr, 0)) return 1
    // x1 (enc1.conv3) also feeds dec1.conv1 and x2 (enc2.conv3) enc3.conv1 / dec2.conv1: their second planes must be 16-bit residuals
    const bool chain_a = chain_ok(h, pl.get(), {L_E1C2, L_E1C3, L_E2C1, L_E2C2, L_E2C3}, L_E2C3) &&
                         (pl->planes == 1 || out_format(h, L_E1C3, pl->c8) == 2);
    if (chain_a) {
        if (add_chain(h, pl.get(), 0, {{L_E1C2, 0, 0, true, nullptr, false}, {L_E1C3, 0, 0, true, pl->X1, false}, {L_E2C1, 0, 0, true, nullptr, false},
                                       {L_E2C2, 0, 0, true, nullptr, false}, {L_E2C3, 0, 0, false, pl->X2, false}},
                      nullptr, 0, nullptr, 0, true))
            return 1;
    } else {
        op = Op(); op.kind = Op::ENC1; pl->ops.push_back(op);            // -> T0 [M,64]
        G(L_E1C2, T0, 64, nullptr, 0, T1);
        G(L_E1C3, T1, 64, nullptr, 0, pl->X1);
        G(L_E2C1, pl->X1, 128, nullptr, 0, T0);
        G(L_E2C2, T0, 128, nullptr, 0, T1);
        G(L_E2C3, T1, 128, nullptr, 0, pl->X2);
    }
    G(L_E3C1, pl->X2, 256, nullptr, 0, T0);
    G(L_E3C2, T0, 256, nullptr, 0, T1);
    G(L_E3C3, T1, 256, nullptr, 0, pl->X3);
    G(L_E4C1, pl->X3, 512, nullptr, 0, T0);
    G(L_E4C2, T0, 512, nullptr, 0, T1);
    G(L_E4C3, T1, 512, nullptr, 0, pl->X4);
    G(L_G0, pl->X4, 1024, nullptr, 0, T0);                          // [M,2048]
    op = Op(); op.kind = Op::MEMSET_G; pl->ops.push_back(op);
    if (add_gemm(h, pl.get(), L_G3, T0, 2048, nullptr, 0, nullptr, EPI_MAXPOOL, nullptr, 0)) return 1;
    op = Op(); op.kind = Op::DBIAS; pl->ops.push_back(op);          // biasd4[B,1024] = Wg * g + bg
    if (add_gemm(h, pl.get(), L_D4C1, pl->X4, 1024, nullptr, 0, T0, EPI_STORE, pl->biasd4, 1024)) return 1;
    G(L_D4C2, T0, 1024, nullptr, 0, T1);
    G(L_D4C3, T1, 1024, nullptr, 0, T0);                            // d4 out [M,512] in T0
    if (h->taps) add_tapcopy(pl.get(), T0, pl->tapD4, M * 512 * e);
    G(L_D3C1, T0, 512, pl->X3, 512, T1);
    G(L_D3C2, T1, 512, nullptr, 0, T0);
    G(L_D3C3, T0, 512, nullptr, 0, T1);                             // d3 out [M,256] in T1
    G(L_D2C1, T1, 256, pl->X2, 256, T0);
    G(L_D2C2, T0, 256, nullptr, 0, T1);
    G(L_D2C3, T1, 256, nullptr, 0, T0);                             // d2 out [M,128] in T0
    // d2 (dec2.conv3, in T0) and x1 are streamed by the chain's first layer: dec2.conv3 must write a 16-bit residual plane
    const bool chain_d = !h->taps && chain_ok(h, pl.get(), {L_D1C1, L_D1C2, L_D1C3, L_O0}, L_D2C3) &&
                         (pl->planes == 1 || out_format(h, L_E1C3, pl->c8) == 2);
    if (chain_d) {
        if (add_chain(h, pl.get(), 1, {{L_D1C1, 2, 2, true, nullptr, false}, {L_D1C2, 0, 0, true, nullptr, false}, {L_D1C3, 0, 0, true, nullptr, false},
                                       {L_O0, 0, 0, false, nullptr, true}},
                      T0, 128, pl->X1, 128, false))
            return 1;
    } else {
    G(L_D1C1, T0, 128, pl->X1, 128, T1);
    G(L_D1C2, T1, 128, nullptr, 0, T0);
    G(L_D1C3, T0, 128, nullptr, 0, T1);                             // d1 out [M,64] in T1
    if (h->taps) add_tapcopy(pl.get(), T1, pl->tapD1, M * 64 * e);
    if (h->precision == PCD_PRECISION_FP32) {
        G(L_O0, T1, 64, nullptr, 0, T0);
        op = Op(); op.kind = Op::FINAL_SIMT; pl->ops.push_back(op);
    } else {
        if (add_gemm(h, pl.get(), L_O0, T1, 64, nullptr, 0, nullptr, EPI_FINAL, nullptr, 0)) return 1;
    }
    }
#undef G
    op = Op(); op.kind = Op::ADVANCE; pl->ops.push_back(op);
    *out = h->plans.insert(key, std::move(pl));
    return 0;
}

static int run_step(pcd_denoiser* h, Plan* pl, cudaStream_t s, bool advance, std::vector<cudaEvent_t>* evs = nullptr) {
    int launched = 0;
    size_t ei = 0;
    for (const Op& op : pl->ops) {
        if (evs) CU(cudaEventRecord((*evs)[ei++], s));
        switch (op.kind) {
            case Op::TIME:
                // sampler calls (advance): the time path of all S steps was computed before the loop (pcd_sample_rows)
                if (advance) break;
                CU(launch_time_bias(pl->B, h->T, 0, pl->call, h->freqs, h->W1T, h->b1, h->W2T, h->b2, h->WtT, h->bt, pl->temb, pl->bias1, s));
                ++launched; break;
            case Op::ENC1:
                CU(launch_enc1_first(pl->elt, h->f16, pl->call, h->Wx, pl->bias1, 64, pl->T0,
                                     pl->planes == 2 ? static_cast<char*>(pl->T0) + pl->M * 64 * 2 : nullptr, pl->B, pl->N, pl->Npad, s));
                ++launched; break;
            case Op::GEMM:
                if (h->precision == PCD_PRECISION_FP32) CU(launch_gemm_simt(op.epi, op.st, s));
                else CU(launch_gemm_tc(op.bn, op.epi, op.np, op.out_planes, op.cl, op.two_sm, op.a0, op.a1, op.b, op.o, op.tc, h->num_sms, s));
                ++launched; break;
            case Op::CHAIN:
                CU(launch_chain_tc(pl->planes, h->f16, op.cmaps, op.cp, h->num_sms, s));
                ++launched; break;
            case Op::MEMSET_G:
                CU(launch_zero_f32(pl->gmax, static_cast<long long>(pl->B) * 4096, s));   // a kernel, not a memset node: keeps the
                ++launched;                                                               // programmatic-launch chain of the step unbroken
                break;
            case Op::DBIAS: {
                SimtGemmParams p{};
                p.A0 = pl->gmax; p.lda0 = 4096; p.K0 = 4096; p.A1 = nullptr; p.lda1 = 0; p.K1 = 0;
                p.W = h->Wg; p.ldw = 4096; p.M = pl->B; p.Nout = 1024; p.out = pl->biasd4; p.ldo = 1024;
                p.bias = h->bg; p.bias_sample_stride = 0; p.rows_per_sample = 1 << 30; p.relu = 0;
                p.partial = pl->dpartial; p.splits = pl->dsplits;
                // batches of at most 8: one CTA per (32 columns, k split) with the tiled kernel's accumulation order (bit-identical)
                if (skinny_splitk_ok(p)) { CU(launch_skinny_splitk(p, s)); }
                else { CU(launch_gemm_simt(EPI_STORE, p, s)); }
                ++launched;
                if (pl->dsplits > 1) { CU(launch_splitk_reduce(pl->dpartial, pl->dsplits, h->bg, pl->biasd4, pl->B, 1024, 0, s)); ++launched; }
                break;
            }
            case Op::FINAL_SIMT:
                CU(launch_final_simt(static_cast<const float*>(pl->T0), pl->M, pl->call, s));
                ++launched; break;
            case Op::ADVANCE:
                if (advance) { CU(launch_advance_step(pl->step, s)); ++launched; }
                break;
            case Op::TAPCOPY:
                CU(cudaMemcpyAsync(op.dst, op.src, op.bytes, cudaMemcpyDeviceToDevice, s));
                break;
        }
    }
    if (evs) CU(cudaEventRecord((*evs)[ei++], s));
    pl->kernels_per_step = launched;
    return 0;
}

static const char* kLayerNames[L_COUNT] = {
    "enc1.conv2", "enc1.conv3", "enc2.conv1", "enc2.conv2", "enc2.conv3", "enc3.conv1", "enc3.conv2", "enc3.conv3",
    "enc4.conv1", "enc4.conv2", "enc4.conv3", "global_feat.0", "global_feat.3+maxpool", "dec4.conv1", "dec4.conv2",
    "dec4.conv3", "dec3.conv1", "dec3.conv2", "dec3.conv3", "dec2.conv1", "dec2.conv2", "dec2.conv3", "dec1.conv1",
    "dec1.conv2", "dec1.conv3", "output.0+output.3+sampler"};

static std::string op_name(const pcd_denoiser* h, const Op& op) {
    switch (op.kind) {
        case Op::TIME: return "time_mlp+enc1_time_bias";
        case Op::ENC1: return "enc1.conv1(xyz)";
        case Op::GEMM: return (op.layer == L_O0 && h->precision == PCD_PRECISION_FP32) ? "output.0" : kLayerNames[op.layer];
        case Op::MEMSET_G: return "memset_g";
        case Op::DBIAS: return "dec4.global_bias";
        case Op::FINAL_SIMT: return "output.3+sampler";
        case Op::ADVANCE: return "advance_step";
        case Op::TAPCOPY: return "tap_copy";
        case Op::CHAIN: return op.chain_id == 0 ? "enc1.conv1-enc2.conv3 (fused chain)" : "dec1.conv1-output.3+sampler (fused chain)";
    }
    return "?";
}

static int set_call(Plan* pl, pcd_denoiser* h, const CallArgs& ca, cudaStream_t s) {
    // pageable -> device copy: the runtime stages the source before returning, so a stack object is safe
    CU(cudaMemcpyAsync(pl->call, &ca, sizeof(CallArgs), cudaMemcpyHostToDevice, s));
    (void)h;
    return 0;
}

extern "C" int pcd_denoiser_forward(pcd_denoiser* h, const float* x, const float* t, float* eps, int32_t B, int32_t N,
                                    void* stream) {
    REQ(h && x && t && eps, "null argument");
    REQ(B > 0 && N > 0, "B and N must be positive");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    Plan* pl = nullptr;
    if (build_plan(h, B, N, &pl)) return 1;
    CallArgs ca{};
    ca.s.x = const_cast<float*>(x); ca.s.eps_out = eps; ca.s.w3 = h->w3; ca.s.b3 = h->b3;
    ca.s.sched = nullptr; ca.s.sched_rows = 1; ca.s.step_ptr = pl->step; ca.s.noise = nullptr; ca.s.noise_step_stride = 0;
    ca.s.seed = 0; ca.s.sample_offset = 0; ca.s.N = N; ca.s.Npad = pl->Npad; ca.s.mode = 0;
    ca.t_in = t;
    if (set_call(pl, h, ca, s)) return 1;
    if (run_step(h, pl, s, false)) return 1;
    g_pcd_launches.fetch_add(pl->kernels_per_step, std::memory_order_relaxed);
    return 0;
}

extern "C" int pcd_denoiser_profile(pcd_denoiser* h, const float* x, const float* t, float* eps, int32_t B, int32_t N,
                                    float* ms_out, double* flops_out, char* names_out, int32_t name_stride, int32_t cap,
                                    int32_t* n_out, void* stream) {
    REQ(h && x && t && eps && ms_out && n_out, "null argument");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    Plan* pl = nullptr;
    if (build_plan(h, B, N, &pl)) return 1;
    CallArgs ca{};
    ca.s.x = const_cast<float*>(x); ca.s.eps_out = eps; ca.s.w3 = h->w3; ca.s.b3 = h->b3;
    ca.s.step_ptr = pl->step; ca.s.N = N; ca.s.Npad = pl->Npad; ca.s.mode = 0; ca.t_in = t;
    if (set_call(pl, h, ca, s)) return 1;
    std::vector<cudaEvent_t> evs(pl->ops.size() + 1);
    for (auto& e : evs) CU(cudaEventCreate(&e));
    int rc = run_step(h, pl, s, false, &evs);
    if (!rc) {
        cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) rc = fail(std::string("profile: ") + cudaGetErrorString(e));
    }
    int n = 0;
    if (!rc) {
        for (size_t i = 0; i < pl->ops.size() && n < cap; ++i) {
            const Op& op = pl->ops[i];
            if (op.kind == Op::ADVANCE || op.kind == Op::TAPCOPY) continue;
            float ms = 0.f;
            cudaEventElapsedTime(&ms, evs[i], evs[i + 1]);
            ms_out[n] = ms;
            if (flops_out) {
                double f = 0.0;   // algorithmic FLOPs of this launch (2 * M * K * Cout for the per-point GEMMs)
                if (op.kind == Op::GEMM) f = 2.0 * static_cast<double>(pl->M) * h->L[op.layer].k * h->L[op.layer].cout;
                if (op.kind == Op::GEMM && op.layer == L_O0) f += 2.0 * static_cast<double>(pl->M) * 64 * 3;
                if (op.kind == Op::ENC1) f = 2.0 * static_cast<double>(pl->M) * 3 * 64;
                if (op.kind == Op::DBIAS) f = 2.0 * static_cast<double>(pl->B) * 4096 * 1024;
                if (op.kind == Op::CHAIN) f = op.chain_flops + (op.chain_id == 1 ? 2.0 * static_cast<double>(pl->M) * 64 * 3 : 0.0);
                flops_out[n] = f;
            }
            if (names_out && name_stride > 0) {
                std::snprintf(names_out + static_cast<size_t>(n) * name_stride, name_stride, "%s", op_name(h, op).c_str());
            }
            ++n;
        }
    }
    for (auto& e : evs) cudaEventDestroy(e);
    *n_out = n;
    g_pcd_launches.fetch_add(pl->kernels_per_step, std::memory_order_relaxed);
    return rc;
}

static int ensure_graph(pcd_denoiser* h, Plan* pl) {
    if (pl->exec) return 0;
    cudaStream_t cs;
    CU(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
    CU(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
    int rc = run_step(h, pl, cs, true);
    cudaError_t e = cudaStreamEndCapture(cs, &pl->graph);
    cudaStreamDestroy(cs);
    if (rc) return 1;
    CU(e);
    CU(cudaGraphInstantiate(&pl->exec, pl->graph, 0));
    return 0;
}

extern "C" int pcd_sample_rows(pcd_denoiser* h, const float* sched, int32_t S, int32_t rows_per_step, float* x, const float* noise,
                               uint64_t seed, uint64_t sample_offset, int32_t B, int32_t N, void* stream) {
    REQ(h && sched && x, "null argument");
    REQ(B > 0 && N > 0 && S > 0, "B, N and S must be positive");
    REQ(rows_per_step == 1 || rows_per_step == B, "rows_per_step must be 1 (shared schedule) or B (one schedule row per sample)");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    Plan* pl = nullptr;
    if (build_plan(h, B, N, &pl)) return 1;
    const int rows = S * rows_per_step;
    if (rows > pl->sched_cap) {
        void* p = nullptr;
        if (plan_alloc(pl, &p, sizeof(float) * kSchedRow * rows)) return 1;
        pl->sched = static_cast<float*>(p); pl->sched_cap = rows;
    }
    CU(cudaMemcpyAsync(pl->sched, sched, sizeof(float) * kSchedRow * rows, cudaMemcpyHostToDevice, s));
    CU(cudaMemsetAsync(pl->step, 0, sizeof(int), s));
    CallArgs ca{};
    ca.s.x = x; ca.s.eps_out = nullptr; ca.s.w3 = h->w3; ca.s.b3 = h->b3;
    ca.s.sched = pl->sched; ca.s.sched_rows = rows_per_step; ca.s.step_ptr = pl->step; ca.s.noise = noise;
    ca.s.noise_step_stride = static_cast<long long>(B) * N * 3;
    ca.s.seed = seed; ca.s.sample_offset = sample_offset; ca.s.N = N; ca.s.Npad = pl->Npad; ca.s.mode = 1;
    ca.t_in = nullptr;
    if (S > pl->steps_cap) {
        void* p = nullptr;
        if (plan_alloc(pl, &p, sizeof(float) * 64 * S)) return 1;
        pl->bias1_steps = static_cast<float*>(p);
        if (plan_alloc(pl, &p, sizeof(float) * h->T * S)) return 1;
        pl->temb_steps = static_cast<float*>(p);
        pl->steps_cap = S;
    }
    ca.bias1_steps = pl->bias1_steps;
    if (set_call(pl, h, ca, s)) return 1;
    // t depends on the step only (every sample of a step shares it): timestep embedding + time MLP + the temb columns of
    // enc1.conv1 for ALL S steps in one launch, outside the per-step graph
    LAUNCH(launch_time_bias(S, h->T, 1, pl->call, h->freqs, h->W1T, h->b1, h->W2T, h->b2, h->WtT, h->bt, pl->temb_steps, pl->bias1_steps, s));
    const bool use_graph = std::getenv("PCD_NO_GRAPH") == nullptr;
    if (use_graph) {
        if (ensure_graph(h, pl)) return 1;
        for (int i = 0; i < S; ++i) CU(cudaGraphLaunch(pl->exec, s));
    } else {
        for (int i = 0; i < S; ++i)
            if (run_step(h, pl, s, true)) return 1;
    }
    g_pcd_launches.fetch_add(static_cast<long long>(pl->kernels_per_step) * S, std::memory_order_relaxed);
    return 0;
}

extern "C" int pcd_sample(pcd_denoiser* h, const float* sched, int32_t S, float* x, const float* noise, uint64_t seed,
                          uint64_t sample_offset, int32_t B, int32_t N, void* stream) {
    return pcd_sample_rows(h, sched, S, 1, x, noise, seed, sample_offset, B, N, stream);
}

extern "C" int pcd_sample_host(pcd_denoiser* h, const float* sched, int32_t S, const float* x_T_host, float* x_out_host,
                               const float* noise_host, uint64_t seed, uint64_t sample_offset, int32_t B, int32_t N,
                               void* stream) {
    return pcd_sample_host_rows(h, sched, S, 1, x_T_host, x_out_host, noise_host, seed, sample_offset, B, N, stream);
}

extern "C" int pcd_sample_host_rows(pcd_denoiser* h, const float* sched, int32_t S, int32_t rows_per_step, const float* x_T_host,
                                    float* x_out_host, const float* noise_host, uint64_t seed, uint64_t sample_offset, int32_t B,
                                    int32_t N, void* stream) {
    REQ(h && x_T_host && x_out_host, "null argument");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t bytes = sizeof(float) * 3 * static_cast<size_t>(B) * N;
    Plan* pl = nullptr;
    if (build_plan(h, B, N, &pl)) return 1;
    if (!pl->xstage) {   // plan-owned: no allocator traffic per call
        void* p = nullptr;
        if (plan_alloc(pl, &p, bytes)) return 1;
        pl->xstage = static_cast<float*>(p);
    }
    float *dx = pl->xstage, *dn = nullptr;
    CU(cudaMemcpyAsync(dx, x_T_host, bytes, cudaMemcpyHostToDevice, s));
    if (noise_host && S > 1) {
        CU(cudaMallocAsync(reinterpret_cast<void**>(&dn), bytes * (S - 1), s));
        CU(cudaMemcpyAsync(dn, noise_host, bytes * (S - 1), cudaMemcpyHostToDevice, s));
    }
    int rc = pcd_sample_rows(h, sched, S, rows_per_step, dx, dn, seed, sample_offset, B, N, stream);
    if (!rc) {
        cudaError_t e = cudaMemcpyAsync(x_out_host, dx, bytes, cudaMemcpyDeviceToHost, s);
        if (e != cudaSuccess) rc = fail(cudaGetErrorString(e));
    }
    if (dn) cudaFreeAsync(dn, s);
    cudaError_t e = cudaStreamSynchronize(s);
    if (!rc && e != cudaSuccess) rc = fail(std::string("pcd_sample_host: ") + cudaGetErrorString(e));
    return rc;
}

extern "C" int pcd_philox_normal(uint64_t seed, uint64_t sample_offset, int32_t step, float* out, int32_t B, int32_t N,
                                 void* stream) {
    REQ(out && B > 0 && N > 0, "bad argument");
    LAUNCH(launch_philox_fill(out, seed, sample_offset, step, B, N, static_cast<cudaStream_t>(stream)));
    return 0;
}

extern "C" int pcd_denoiser_tap(pcd_denoiser* h, const char* name, float* out_host, int64_t count) {
    REQ(h && name && out_host, "null argument");
    CU(cudaSetDevice(h->device));
    REQ(!h->plans.empty(), "no forward has run yet");
    Plan* pl = h->plans.last;                          // the plan of the most recent call
    REQ(pl != nullptr, "no forward has run yet");
    const std::string n(name);
    const void* src = nullptr; long long cnt = 0; bool act = true; int fmt = pl->planes == 2 ? 2 : 1, width = 0;
    if (n == "temb") { src = pl->temb; cnt = 1LL * pl->B * h->T; act = false; }
    else if (n == "g") { src = pl->gmax; cnt = 1LL * pl->B * 4096; act = false; }
    else if (n == "biasd4") { src = pl->biasd4; cnt = 1LL * pl->B * 1024; act = false; }
    else if (n == "x1") { src = pl->X1; cnt = pl->M * 128; }
    else if (n == "x2") { src = pl->X2; cnt = pl->M * 256; }
    else if (n == "x3") { src = pl->X3; cnt = pl->M * 512; fmt = pl->planes == 2 ? pl->fmtX3 : 1; width = 512; }
    else if (n == "x4") { src = pl->X4; cnt = pl->M * 1024; fmt = pl->planes == 2 ? pl->fmtX4 : 1; width = 1024; }
    else if (n == "d4") { src = pl->tapD4; cnt = pl->M * 512; fmt = pl->planes == 2 ? pl->fmtD4 : 1; width = 512; }
    else if (n == "d1") { src = pl->tapD1; cnt = pl->M * 64; }
    REQ(src != nullptr, "unknown tap (d4/d1 need PCD_TAPS=1 at create time): " + n);
    REQ(cnt == count, "tap size mismatch for " + n + ": expected " + std::to_string(cnt));
    CU(cudaDeviceSynchronize());
    if (!act || pl->elt == 4) {
        CU(cudaMemcpy(out_host, src, sizeof(float) * cnt, cudaMemcpyDeviceToHost));
    } else {
        float* tmp = nullptr;
        CU(cudaMalloc(&tmp, sizeof(float) * cnt));
        if (fmt == 3) LAUNCH(launch_16c8_to_f32(src, static_cast<const char*>(src) + cnt * 2, tmp, pl->M, width, 0));
        else LAUNCH(launch_16_to_f32(src, fmt == 2 ? static_cast<const char*>(src) + cnt * 2 : nullptr, tmp, cnt, h->f16, 0));
        CU(cudaMemcpy(out_host, tmp, sizeof(float) * cnt, cudaMemcpyDeviceToHost));
        cudaFree(tmp);
    }
    return 0;
}

extern "C" int pcd_denoiser_destroy(pcd_denoiser* h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    h->plans.clear();
    for (void* p : h->owned) cudaFree(p);
    delete h;
    return 0;
}

extern "C" int pcd_linear_bf16(const void* A0, int32_t K0, const void* A1, int32_t K1, const void* W, const float* bias,
                               void* out, int32_t M, int32_t Cout, int32_t relu, void* stream) {
    REQ(A0 && W && bias && out, "null argument");
    REQ(M > 0 && M % 128 == 0, "M must be a positive multiple of 128");
    REQ(K0 > 0 && K0 % 64 == 0 && K1 >= 0 && K1 % 64 == 0, "K0/K1 must be multiples of 64");
    REQ(Cout > 0 && Cout % 64 == 0 && (Cout <= 256 || Cout % 256 == 0) && Cout != 192, "Cout must be 64, 128 or a multiple of 256");
    int dev = 0; CU(cudaGetDevice(&dev));
    int sms = 0; CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int bn = Cout >= 256 ? 256 : Cout;
    CU(configure_gemm_tc());
    CUtensorMap a0, a1, b, o;
    if (make_tmap(&o, out, M, Cout, Cout, 32)) return 1;
    if (make_tmap(&a0, A0, M, K0, K0, 128)) return 1;
    if (K1 > 0) { REQ(A1 != nullptr, "A1 is null but K1 > 0"); if (make_tmap(&a1, A1, M, K1, K1, 128)) return 1; }
    else a1 = a0;
    const int cl = (M / 128) % 2 == 0 ? 2 : 1;
    if (make_tmap(&b, W, Cout, K0 + K1, K0 + K1, bn / cl)) return 1;
    TcGemmParams p{};
    p.num_m_blocks = M / 128; p.num_n_blocks = Cout / bn; p.kb0 = K0 / 64; p.kb1 = K1 / 64;
    p.out = static_cast<__nv_bfloat16*>(out); p.ldo = Cout; p.bias = bias; p.bias_sample_stride = 0;
    p.rows_per_sample = 1 << 30; p.relu = relu;
    const int two_sm = (cl == 2 && K0 + K1 >= 1024) ? 1 : 0;
    LAUNCH(launch_gemm_tc(bn, EPI_STORE, 1, 1, cl, two_sm, a0, a1, b, o, p, sms, static_cast<cudaStream_t>(stream)));
    return 0;
}

// ------------------------------------------------------------------------------------------
// Chamfer
// ------------------------------------------------------------------------------------------
extern "C" int pcd_chamfer_pairs(const float* x, const float* y, int32_t B, int32_t N, int32_t M, float scaling, float* cd,
                                 int32_t* idx_xy, int32_t* idx_yx, void* stream) {
    REQ(x && y && cd, "null argument");
    REQ(B > 0 && N > 0 && M > 0, "B, N, M must be positive");
    REQ(B <= 65535, "at most 65535 pairs per call");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    float4 *xn = nullptr, *yn = nullptr; float *dxy = nullptr, *dyx = nullptr;
    CU(cudaMallocAsync(reinterpret_cast<void**>(&xn), sizeof(float4) * B * N, s));
    CU(cudaMallocAsync(reinterpret_cast<void**>(&yn), sizeof(float4) * B * M, s));
    LAUNCH(launch_cloud_norm(x, B, N, xn, s));
    LAUNCH(launch_cloud_norm(y, B, M, yn, s));
    if (!idx_xy && !idx_yx && chamfer_fused_fits(N, M)) {
        // values only: one fused pass feeds both directional minima
        LAUNCH(launch_chamfer_fused(xn, yn, B, 0, N, M, scaling, cd, s));
    } else {
        CU(cudaMallocAsync(reinterpret_cast<void**>(&dxy), sizeof(float) * B * N, s));
        CU(cudaMallocAsync(reinterpret_cast<void**>(&dyx), sizeof(float) * B * M, s));
        LAUNCH(launch_chamfer_dir(xn, yn, B, N, M, dxy, idx_xy, s));
        LAUNCH(launch_chamfer_dir(yn, xn, B, M, N, dyx, idx_yx, s));
        LAUNCH(launch_chamfer_reduce(dxy, dyx, B, N, M, scaling, cd, s));
        cudaFreeAsync(dxy, s); cudaFreeAsync(dyx, s);
    }
    cudaFreeAsync(xn, s); cudaFreeAsync(yn, s);
    return 0;
}

extern "C" int pcd_chamfer_matrix(const float* G, int32_t nG, const float* R, int32_t nR, int32_t N, float scaling,
                                  float* out, void* stream) {
    REQ(G && R && out, "null argument");
    REQ(nG > 0 && nR > 0 && N > 0, "nG, nR, N must be positive");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    float4 *gn = nullptr, *rn = nullptr;
    if (G == R && nG == nR) {
        // a set against itself (the diagonal blocks of D_gg / D_rr in metrics.evaluate_sets): CD is bit-symmetric, so the upper
        // triangle is evaluated and mirrored -- same values as the full sweep for half the pairs, one normalisation pass
        CU(cudaMallocAsync(reinterpret_cast<void**>(&gn), sizeof(float4) * nG * N, s));
        LAUNCH(launch_cloud_norm(G, nG, N, gn, s));
        CU(launch_chamfer_matrix_self(gn, nG, N, scaling, out, s));
        g_pcd_launches.fetch_add(1, std::memory_order_relaxed);
        cudaFreeAsync(gn, s);
        return 0;
    }
    CU(cudaMallocAsync(reinterpret_cast<void**>(&gn), sizeof(float4) * nG * N, s));
    CU(cudaMallocAsync(reinterpret_cast<void**>(&rn), sizeof(float4) * nR * N, s));
    LAUNCH(launch_cloud_norm(G, nG, N, gn, s));
    LAUNCH(launch_cloud_norm(R, nR, N, rn, s));
    CU(launch_chamfer_matrix(gn, nG, rn, nR, N, scaling, out, s));
    g_pcd_launches.fetch_add(2, std::memory_order_relaxed);
    cudaFreeAsync(gn, s); cudaFreeAsync(rn, s);
    return 0;
}

// ------------------------------------------------------------------------------------------
// Sinkhorn EMD (metrics.py:94-158)
// ------------------------------------------------------------------------------------------
extern "C" int pcd_sinkhorn_emd(const float* x, const float* y, int32_t B, int32_t N, int32_t M, float epsilon, float thresh,
                                int32_t max_iter, float scaling, float* emd, int32_t* iters_out, void* stream) {
    REQ(B > 0 && N > 0 && M > 0, "B, N, M must be positive");   // before the null test: an empty batch has null buffers
    REQ(x && y && emd, "null argument");
    REQ(B <= 65535, "at most 65535 pairs per call");
    REQ(epsilon > 0.f && max_iter >= 0, "epsilon must be positive and max_iter non-negative");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int nblk = emd_row_blocks(N);
    float4 *xn = nullptr, *yn = nullptr;
    float* work = nullptr;   // alpha [B,N] | beta [B,M] | partial [B,nblk] | cmax | err[2*max_iter]
    const size_t nA = static_cast<size_t>(B) * N, nB = static_cast<size_t>(B) * M, nP = static_cast<size_t>(B) * nblk;
    const size_t nwork = nA + nB + nP + 1 + 2 * static_cast<size_t>(max_iter) + 2;
    CU(cudaMallocAsync(reinterpret_cast<void**>(&xn), sizeof(float4) * nA, s));
    CU(cudaMallocAsync(reinterpret_cast<void**>(&yn), sizeof(float4) * nB, s));
    CU(cudaMallocAsync(reinterpret_cast<void**>(&work), sizeof(float) * nwork, s));
    CU(cudaMemsetAsync(work, 0, sizeof(float) * nwork, s));   // duals start at 0 (metrics.py:130-131); cmax and err slots at 0
    float* alpha = work; float* beta = alpha + nA; float* partial = beta + nB;
    unsigned* cmax = reinterpret_cast<unsigned*>(partial + nP);
    unsigned* err = cmax + 1;
    int rc = 0;
    auto run = [&]() -> int {
        LAUNCH(launch_cloud_norm(x, B, N, xn, s));
        LAUNCH(launch_cloud_norm(y, B, M, yn, s));
        LAUNCH(launch_emd_cmax(xn, yn, B, N, M, cmax, s));
        const float lambda = static_cast<float>(1.0 / static_cast<double>(epsilon));       // lambda_val = 1 / epsilon (:127)
        const float log_mu = std::log(1.0f / static_cast<float>(N) + 1e-10f);              // log(mu + 1e-10) (:142)
        const float log_nu = std::log(1.0f / static_cast<float>(M) + 1e-10f);
        int it = 0;
        for (; it < max_iter; ++it) {
            LAUNCH(launch_sinkhorn_half(xn, yn, beta, alpha, B, N, M, cmax, lambda, epsilon, log_mu, err + 2 * it, s));
            LAUNCH(launch_sinkhorn_half(yn, xn, alpha, beta, B, M, N, cmax, lambda, epsilon, log_nu, err + 2 * it + 1, s));
            float e[2];
            CU(cudaMemcpyAsync(e, err + 2 * it, sizeof(e), cudaMemcpyDeviceToHost, s));
            CU(cudaStreamSynchronize(s));      // the reference's `if err < thresh: break` is the same host round trip (:148-151)
            if (e[0] < thresh && e[1] < thresh) { ++it; break; }
        }
        if (iters_out) *iters_out = it;
        LAUNCH(launch_sinkhorn_cost(xn, yn, alpha, beta, B, N, M, cmax, lambda, scaling, partial, emd, s));
        return 0;
    };
    rc = run();
    cudaFreeAsync(xn, s); cudaFreeAsync(yn, s); cudaFreeAsync(work, s);
    return rc;
}

// ------------------------------------------------------------------------------------------
// Exact EMD (metrics.py:49-92): auction assignment per pair, emd_exact.cu
// ------------------------------------------------------------------------------------------
extern "C" int pcd_emd_exact(const float* x, const float* y, int32_t B, int32_t N, int32_t M, float scaling, float* emd,
                             int32_t* assign_xy, void* stream) {
    REQ(x && y && emd, "null argument");
    REQ(B > 0 && N > 0 && M > 0, "B, N, M must be positive");
    REQ(B <= 65535, "at most 65535 pairs per call");
    REQ(emd_exact_fits(N, M), "exact EMD supports at most 4096 points per cloud (N = " + std::to_string(N) + ", M = " +
                                  std::to_string(M) + ")");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    float4 *xn = nullptr, *yn = nullptr;
    int* err = nullptr;
    CU(cudaMallocAsync(reinterpret_cast<void**>(&xn), sizeof(float4) * B * N, s));
    CU(cudaMallocAsync(reinterpret_cast<void**>(&yn), sizeof(float4) * B * M, s));
    CU(cudaMallocAsync(reinterpret_cast<void**>(&err), sizeof(int), s));
    auto run = [&]() -> int {
        CU(cudaMemsetAsync(err, 0, sizeof(int), s));
        LAUNCH(launch_cloud_norm(x, B, N, xn, s));
        LAUNCH(launch_cloud_norm(y, B, M, yn, s));
        LAUNCH(launch_emd_exact(xn, yn, B, N, M, scaling, emd, assign_xy, err, s));
        int e = 0;
        CU(cudaMemcpyAsync(&e, err, sizeof(int), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));      // the round-cap flag is the only thing read back
        REQ(e == 0, "exact EMD: an auction phase exceeded its round cap (the affected pairs are NaN)");
        return 0;
    };
    const int rc = run();
    cudaFreeAsync(xn, s); cudaFreeAsync(yn, s); cudaFreeAsync(err, s);
    return rc;
}
