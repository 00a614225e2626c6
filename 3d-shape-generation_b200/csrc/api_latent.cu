// C ABI of the latent-diffusion path: pcd_latent_* (include/pcd_b200.h).
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <memory>

#include "api_common.h"
#include "pcd_launch.h"
#include "pcd_types.h"

using namespace pcd;

namespace {

struct Lin {   // fp32 Linear on the device, weight [cout][cin]
    int cout = 0, cin = 0;
    float *w = nullptr, *b = nullptr;
    float *gamma = nullptr, *beta = nullptr;   // GroupNorm affine (nullptr: no norm)
};

struct LatentPlan {
    int B = 0;
    float *zbuf, *temb, *z1, *z2, *z3, *z4, *g0, *g1, *r, *d4, *d3, *d2, *d1, *o0, *eps;
    float* partial = nullptr;     // split-K workspace
    float* sched = nullptr; int sched_cap = 0;
    int* step = nullptr;
    LatentCall* call = nullptr;
    int kernels_per_step = 0;
    // persistent-kernel path (latent_mk.cu)
    float *emb = nullptr, *th = nullptr, *tembR = nullptr, *bias1 = nullptr;   // time rows [Rcap][256 / 256 / 256 / 128]
    int Rcap = 0;
    size_t partial_cap = 0;
    LtProgram* prog = nullptr;       // device copy of the reverse-step program
    LtProgram* dprog = nullptr;      // device copy of the SimplePointNetVAE.decode program
    float *da = nullptr, *db = nullptr, *dc = nullptr;
    unsigned* bar = nullptr;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    std::vector<void*> owned;
    ~LatentPlan() {
        if (exec) cudaGraphExecDestroy(exec);
        if (graph) cudaGraphDestroy(graph);
        for (void* p : owned) cudaFree(p);
    }
};

}  // namespace

struct pcd_latent {
    int num_sms = 148;
    int device = 0, latent_dim = 256, dim = 512, num_points = 0;
    float *freqs = nullptr, *W1T = nullptr, *b1 = nullptr, *W2T = nullptr, *b2 = nullptr;
    Lin enc1, enc2, enc3, enc4, gf0, gf3, dec4, dec3, dec2, dec1, out0, out2, ref1, ref2, ref3, ref4;
    Lin dec4c, dec3c, dec2c, dec1c;   // decK with refineK composed into its skip columns (persistent-kernel path)
    float *tw0 = nullptr, *tw2 = nullptr;   // time MLP weights [out][in]
    // tile-major, pre-swizzled copies streamed by the persistent kernel (latent_mk.cu: tile_weights_kernel)
    float *t_tw0 = nullptr, *t_tw2 = nullptr, *t_enc1t = nullptr, *t_enc3 = nullptr, *t_enc4 = nullptr, *t_gf0 = nullptr,
          *t_gf3 = nullptr, *t_dec4 = nullptr, *t_dec3 = nullptr, *t_dec2 = nullptr, *t_vd0 = nullptr, *t_vd2 = nullptr,
          *t_vd4 = nullptr, *t_vout = nullptr;
    int mk_grid = 0;                  // CTAs of the persistent kernel (0: unavailable)
    Lin vd0, vd2, vd4, vout;   // SimplePointNetVAE decoder
    float *out0T = nullptr, *out2T = nullptr;   // output.0 / output.2 weights transposed [in][out] for the row-per-CTA tail phase
    float *dec1cT = nullptr;                    // dec1 (refine1 composed) [384][128], transposed: the tail phase computes dec1 itself
    float *enc1zT = nullptr, *enc2T = nullptr;  // enc1's z columns [256][128] / enc2 [128][256], transposed for the row-per-CTA head phase
    bool has_model = true;    // false: decoder-only handle (no latent denoiser weights)
    bool has_vae = false;
    // FoldingDecoder (PointNetVAE.decode, networks.py:1449-1509), composed at load time (see folding.cu)
    struct Fold { Lin wz, wab, wbc; float *wg = nullptr, *wc2 = nullptr, *bc2 = nullptr; int kin = 0;
                  void* wab16 = nullptr; /* W_ab as fp16 hi / lo planes [2 * 512][512] for the tcgen05 path */ } fold[2];
    Lin upsample;
    float* grid = nullptr;     // [1024][2]
    bool has_folding = false;
    PlanCache<int, LatentPlan> plans;
    std::vector<void*> owned;
};

static int up(pcd_latent* h, const float* src, size_t n, float** out) {
    void* p = nullptr;
    CU(cudaMalloc(&p, n * sizeof(float)));
    h->owned.push_back(p);
    CU(cudaMemcpy(p, src, n * sizeof(float), cudaMemcpyHostToDevice));
    *out = static_cast<float*>(p);
    return 0;
}

static int load_lin(pcd_latent* h, const TensorTable& tt, const std::string& name, int cout, int cin, const std::string& gn,
                    Lin* L) {
    std::string err;
    const float *w, *b;
    if (!fetch(tt, name + ".weight", 1LL * cout * cin, &w, &err) || !fetch(tt, name + ".bias", cout, &b, &err)) return fail(err);
    L->cout = cout; L->cin = cin;
    if (up(h, w, 1LL * cout * cin, &L->w) || up(h, b, cout, &L->b)) return 1;
    if (!gn.empty()) {
        const float *g, *be;
        if (!fetch(tt, gn + ".weight", cout, &g, &err) || !fetch(tt, gn + ".bias", cout, &be, &err)) return fail(err);
        if (up(h, g, cout, &L->gamma) || up(h, be, cout, &L->beta)) return 1;
    }
    return 0;
}

// FoldingDecoder weights: conv(k=1) weights [cout, cin, 1].  fold f: layers 0/1/2 = FoldingLayer(256+kin, 512),
// (512, 512), (512, 3); every FoldingLayer is conv(.layer.0) -> ReLU -> conv(.layer.2) with nothing after it, so
//   W_ab = L1.0 * L0.2,  b_ab = L1.0 * b(L0.2) + b(L1.0)      (512 x 512)
//   W_bc = L2.0 * L1.2,  b_bc = L2.0 * b(L1.2) + b(L2.0)      (3 x 512)
// composed in double on the host.  The latent columns of L0.0 become a per-sample bias GEMM (wz).
static int load_folding(pcd_latent* h, const TensorTable& tt, int num_points) {
    std::string err;
    for (int f = 0; f < 2; ++f) {
        const std::string pre = std::string("vae.decoder.fold") + (f == 0 ? "1" : "2");
        const int kin = f == 0 ? 2 : 3, cin = 256 + kin;
        const float *a1, *ba1, *a2, *ba2, *b1, *bb1, *b2, *bb2, *c1, *bc1, *c2, *bc2;
        if (!fetch(tt, pre + ".0.layer.0.weight", 512LL * cin, &a1, &err) || !fetch(tt, pre + ".0.layer.0.bias", 512, &ba1, &err) ||
            !fetch(tt, pre + ".0.layer.2.weight", 512LL * 512, &a2, &err) || !fetch(tt, pre + ".0.layer.2.bias", 512, &ba2, &err) ||
            !fetch(tt, pre + ".1.layer.0.weight", 512LL * 512, &b1, &err) || !fetch(tt, pre + ".1.layer.0.bias", 512, &bb1, &err) ||
            !fetch(tt, pre + ".1.layer.2.weight", 512LL * 512, &b2, &err) || !fetch(tt, pre + ".1.layer.2.bias", 512, &bb2, &err) ||
            !fetch(tt, pre + ".2.layer.0.weight", 3LL * 512, &c1, &err) || !fetch(tt, pre + ".2.layer.0.bias", 3, &bc1, &err) ||
            !fetch(tt, pre + ".2.layer.2.weight", 9, &c2, &err) || !fetch(tt, pre + ".2.layer.2.bias", 3, &bc2, &err))
            return fail(err + " (FoldingDecoder with latent_dim = 256 expected)");
        pcd_latent::Fold& F = h->fold[f];
        F.kin = kin;
        std::vector<float> wz(512 * 256), wg(512 * kin);
        for (int c = 0; c < 512; ++c) {      // cat([z, grid]) / cat([z, fold1_out]): latent columns first (networks.py:1499,1503)
            for (int k = 0; k < 256; ++k) wz[c * 256 + k] = a1[c * cin + k];
            for (int k = 0; k < kin; ++k) wg[c * kin + k] = a1[c * cin + 256 + k];
        }
        F.wz.cout = 512; F.wz.cin = 256;
        if (up(h, wz.data(), wz.size(), &F.wz.w) || up(h, ba1, 512, &F.wz.b) || up(h, wg.data(), wg.size(), &F.wg)) return 1;
        std::vector<double> acc(512);
        std::vector<float> wab(512 * 512), bab(512), wbc(3 * 512), bbc(3);
        for (int o = 0; o < 512; ++o) {
            std::fill(acc.begin(), acc.end(), 0.0);
            double bs = bb1[o];
            for (int m = 0; m < 512; ++m) {
                const double w = b1[o * 512 + m];
                bs += w * ba2[m];
                const float* row = a2 + m * 512;
                for (int k = 0; k < 512; ++k) acc[k] += w * row[k];
            }
            for (int k = 0; k < 512; ++k) wab[o * 512 + k] = static_cast<float>(acc[k]);
            bab[o] = static_cast<float>(bs);
        }
        for (int o = 0; o < 3; ++o) {
            std::fill(acc.begin(), acc.end(), 0.0);
            double bs = bc1[o];
            for (int m = 0; m < 512; ++m) {
                const double w = c1[o * 512 + m];
                bs += w * bb2[m];
                const float* row = b2 + m * 512;
                for (int k = 0; k < 512; ++k) acc[k] += w * row[k];
            }
            for (int k = 0; k < 512; ++k) wbc[o * 512 + k] = static_cast<float>(acc[k]);
            bbc[o] = static_cast<float>(bs);
        }
        F.wab.cout = 512; F.wab.cin = 512; F.wbc.cout = 3; F.wbc.cin = 512;
        if (up(h, wab.data(), wab.size(), &F.wab.w) || up(h, bab.data(), 512, &F.wab.b) || up(h, wbc.data(), wbc.size(), &F.wbc.w) ||
            up(h, bbc.data(), 3, &F.wbc.b) || up(h, c2, 9, &F.wc2) || up(h, bc2, 3, &F.bc2))
            return 1;
        {
            void* p16 = nullptr;
            CU(cudaMalloc(&p16, sizeof(uint16_t) * 2 * 512 * 512)); h->owned.push_back(p16);
            F.wab16 = p16;
            CU(launch_f32_split_16(F.wab.w, p16, static_cast<char*>(p16) + sizeof(uint16_t) * 512 * 512, 512LL * 512, 1, nullptr));
        }
    }
    {
        // the 512 x 512 GEMMs of the folds run on the split-precision tcgen05 kernel
        cudaDeviceProp prop;
        CU(cudaGetDeviceProperties(&prop, h->device));
        REQ(prop.major == 10, "FoldingDecoder: the tcgen05 path requires an sm_100-class GPU (B200)");
        CU(configure_gemm_tc());
    }
    const float *wu, *bu, *grid;
    if (!fetch(tt, "vae.decoder.upsample.weight", 1024LL * num_points, &wu, &err) ||
        !fetch(tt, "vae.decoder.upsample.bias", num_points, &bu, &err))
        return fail(err);
    // the 32 x 32 folding grid is a plain attribute of the reference module (networks.py:1463-1467), not a parameter:
    // the host wrapper passes it as "vae.decoder.grid" [2, 1024] so that torch.linspace's exact bits are used
    if (!fetch(tt, "vae.decoder.grid", 2048, &grid, &err)) return fail(err);
    std::vector<float> g(2048);
    for (int n = 0; n < 1024; ++n) { g[n * 2] = grid[n]; g[n * 2 + 1] = grid[1024 + n]; }
    h->upsample.cout = num_points; h->upsample.cin = 1024;
    if (up(h, wu, 1024LL * num_points, &h->upsample.w) || up(h, bu, num_points, &h->upsample.b) || up(h, g.data(), 2048, &h->grid)) return 1;
    h->has_folding = true;
    return 0;
}

// decK(cat([prev, refineK(x_k)])) = Wd[:, :P] prev + (Wd[:, P:] Wr) x_k + (bd + Wd[:, P:] br): exact algebra, composed once
// on the device with double accumulation (networks.py:1080-1083); the four refine Linears leave the step.
static int compose_dec(pcd_latent* h, const Lin& dec, int P, const Lin& ref, Lin* out) {
    *out = dec;
    void* p = nullptr;
    CU(cudaMalloc(&p, sizeof(float) * dec.cout * dec.cin)); h->owned.push_back(p); out->w = static_cast<float*>(p);
    CU(cudaMalloc(&p, sizeof(float) * dec.cout)); h->owned.push_back(p); out->b = static_cast<float*>(p);
    CU(cudaMemcpy(out->w, dec.w, sizeof(float) * dec.cout * dec.cin, cudaMemcpyDeviceToDevice));
    if (dec.cin - P != ref.cout || ref.cin != ref.cout) return fail("latent: refine shape mismatch");
    CU(launch_compose_refine(dec.w, dec.cin, P, ref.w, ref.cout, dec.b, ref.b, out->w, out->b, dec.cout, nullptr));
    return 0;
}

// tile width of a layer in the persistent kernel: 128 columns where a CTA would otherwise walk many 64-column chunk jobs
// (global_feat.*, dec4, the VAE decoder's wide layers: half the chunk iterations per CTA), 64 elsewhere
static int lt_bn(int N, int K) { return (N % 128 == 0 && static_cast<long long>(N / 64) * (K / 32) >= 1024) ? 128 : 64; }

static int tile_w(pcd_latent* h, const float* W, int ldw, int col0, int N, int K, float** out) {
    void* p = nullptr;
    CU(cudaMalloc(&p, sizeof(float) * N * K)); h->owned.push_back(p);
    *out = static_cast<float*>(p);
    CU(launch_tile_weights(W, ldw, col0, N, K, lt_bn(N, K), *out, nullptr));
    return 0;
}

extern "C" int pcd_latent_destroy(pcd_latent* h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    h->plans.clear();
    for (void* p : h->owned) cudaFree(p);
    delete h;
    return 0;
}

extern "C" int pcd_latent_create(const pcd_named_tensor* tensors, int32_t n_tensors, int32_t num_points, int32_t device,
                                 pcd_latent** out) {
    REQ(tensors && out, "null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
        return fail("pcd: no CUDA device available -- this library has no CPU fallback");
    CU(cudaSetDevice(device));
    TensorTable tt;
    for (int i = 0; i < n_tensors; ++i) tt.m[tensors[i].name] = &tensors[i];
    std::unique_ptr<pcd_latent, int (*)(pcd_latent*)> h(new pcd_latent(), pcd_latent_destroy);
    h->device = device; h->num_points = num_points;
    CU(cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device));
    std::string err;
    pcd_latent* p = h.get();
    // a table without `model.*` builds a decoder-only handle (standalone `vae.decode`, networks.py:1219-1231 / 1579-1589)
    p->has_model = tt.m.count("model.time_mlp.0.weight") != 0;
    if (p->has_model) {
        // the kernels are specialised for the reference defaults latent_dim = time_dim = 256, dim = 512
        const float *tw0, *tb0, *tw2, *tb2;
        if (!fetch(tt, "model.time_mlp.0.weight", 256 * 256, &tw0, &err) || !fetch(tt, "model.time_mlp.0.bias", 256, &tb0, &err) ||
            !fetch(tt, "model.time_mlp.2.weight", 256 * 256, &tw2, &err) || !fetch(tt, "model.time_mlp.2.bias", 256, &tb2, &err))
            return fail(err + " (latent path supports latent_dim = time_dim = 256, dim = 512)");
        {
            std::vector<float> w1t(256 * 256), w2t(256 * 256), fr(128);
            for (int o = 0; o < 256; ++o)
                for (int k = 0; k < 256; ++k) { w1t[k * 256 + o] = tw0[o * 256 + k]; w2t[k * 256 + o] = tw2[o * 256 + k]; }
            const float emb = std::log(10000.0f) / 127.0f;
            for (int j = 0; j < 128; ++j) fr[j] = std::exp(static_cast<float>(j) * -emb);
            if (up(h.get(), tw0, 256 * 256, &h->tw0) || up(h.get(), tw2, 256 * 256, &h->tw2)) return 1;
            if (up(h.get(), w1t.data(), w1t.size(), &h->W1T) || up(h.get(), w2t.data(), w2t.size(), &h->W2T) ||
                up(h.get(), tb0, 256, &h->b1) || up(h.get(), tb2, 256, &h->b2) || up(h.get(), fr.data(), 128, &h->freqs))
                return 1;
        }
        if (load_lin(p, tt, "model.enc1.0", 128, 512, "model.enc1.1", &p->enc1) || load_lin(p, tt, "model.enc2.0", 256, 128, "model.enc2.1", &p->enc2) ||
            load_lin(p, tt, "model.enc3.0", 512, 256, "model.enc3.1", &p->enc3) || load_lin(p, tt, "model.enc4.0", 1024, 512, "model.enc4.1", &p->enc4) ||
            load_lin(p, tt, "model.global_feat.0", 2048, 1024, "model.global_feat.1", &p->gf0) ||
            load_lin(p, tt, "model.global_feat.3", 4096, 2048, "model.global_feat.4", &p->gf3) ||
            load_lin(p, tt, "model.dec4.0", 1024, 5120, "model.dec4.1", &p->dec4) || load_lin(p, tt, "model.dec3.0", 512, 1536, "model.dec3.1", &p->dec3) ||
            load_lin(p, tt, "model.dec2.0", 256, 768, "model.dec2.1", &p->dec2) || load_lin(p, tt, "model.dec1.0", 128, 384, "model.dec1.1", &p->dec1) ||
            load_lin(p, tt, "model.output.0", 128, 128, "", &p->out0) || load_lin(p, tt, "model.output.2", 256, 128, "", &p->out2) ||
            load_lin(p, tt, "model.refine1", 128, 128, "", &p->ref1) || load_lin(p, tt, "model.refine2", 256, 256, "", &p->ref2) ||
            load_lin(p, tt, "model.refine3", 512, 512, "", &p->ref3) || load_lin(p, tt, "model.refine4", 1024, 1024, "", &p->ref4))
            return 1;
    }
    if (tt.m.count("vae.output_layer.weight") && num_points > 0) {
        const int P3 = num_points * 3;
        if (load_lin(p, tt, "vae.decoder.0", 256, 256, "", &p->vd0) || load_lin(p, tt, "vae.decoder.2", 512, 256, "", &p->vd2) ||
            load_lin(p, tt, "vae.decoder.4", P3, 512, "", &p->vd4) || load_lin(p, tt, "vae.output_layer", P3, P3, "", &p->vout))
            return 1;
        p->has_vae = true;
    }
    if (tt.m.count("vae.decoder.fold1.0.layer.0.weight") && num_points > 0) {
        if (load_folding(p, tt, num_points)) return 1;
    }
    if (p->has_model) {
        {
            const float *w0, *w2;
            if (!fetch(tt, "model.output.0.weight", 128LL * 128, &w0, &err) || !fetch(tt, "model.output.2.weight", 256LL * 128, &w2, &err)) return fail(err);
            std::vector<float> t0(128 * 128), t2(128 * 256);
            for (int o = 0; o < 128; ++o) for (int k = 0; k < 128; ++k) t0[k * 128 + o] = w0[o * 128 + k];
            for (int o = 0; o < 256; ++o) for (int k = 0; k < 128; ++k) t2[k * 256 + o] = w2[o * 128 + k];
            if (up(p, t0.data(), t0.size(), &p->out0T) || up(p, t2.data(), t2.size(), &p->out2T)) return 1;
            const float *e1, *e2;
            if (!fetch(tt, "model.enc1.0.weight", 128LL * 512, &e1, &err) || !fetch(tt, "model.enc2.0.weight", 256LL * 128, &e2, &err)) return fail(err);
            std::vector<float> h1(256 * 128), h2(128 * 256);
            for (int o = 0; o < 128; ++o) for (int k = 0; k < 256; ++k) h1[k * 128 + o] = e1[o * 512 + k];      // cat([z, t_emb]): z first
            for (int o = 0; o < 256; ++o) for (int k = 0; k < 128; ++k) h2[k * 256 + o] = e2[o * 128 + k];
            if (up(p, h1.data(), h1.size(), &p->enc1zT) || up(p, h2.data(), h2.size(), &p->enc2T)) return 1;
        }
        if (compose_dec(p, p->dec4, 4096, p->ref4, &p->dec4c) || compose_dec(p, p->dec3, 1024, p->ref3, &p->dec3c) ||
            compose_dec(p, p->dec2, 512, p->ref2, &p->dec2c) || compose_dec(p, p->dec1, 256, p->ref1, &p->dec1c))
            return 1;
        {
            std::vector<float> w(128 * 384), wt(384 * 128);
            CU(cudaMemcpy(w.data(), p->dec1c.w, sizeof(float) * w.size(), cudaMemcpyDeviceToHost));     // synchronises with the compose kernel
            for (int o = 0; o < 128; ++o) for (int k = 0; k < 384; ++k) wt[k * 128 + o] = w[o * 384 + k];
            if (up(p, wt.data(), wt.size(), &p->dec1cT)) return 1;
        }
        if (tile_w(p, p->tw0, 256, 0, 256, 256, &p->t_tw0) || tile_w(p, p->tw2, 256, 0, 256, 256, &p->t_tw2) ||
            tile_w(p, p->enc1.w, 512, 256, 128, 256, &p->t_enc1t) || tile_w(p, p->enc3.w, 256, 0, 512, 256, &p->t_enc3) ||
            tile_w(p, p->enc4.w, 512, 0, 1024, 512, &p->t_enc4) || tile_w(p, p->gf0.w, 1024, 0, 2048, 1024, &p->t_gf0) ||
            tile_w(p, p->gf3.w, 2048, 0, 4096, 2048, &p->t_gf3) || tile_w(p, p->dec4c.w, 5120, 0, 1024, 5120, &p->t_dec4) ||
            tile_w(p, p->dec3c.w, 1536, 0, 512, 1536, &p->t_dec3) || tile_w(p, p->dec2c.w, 768, 0, 256, 768, &p->t_dec2))
            return 1;
    }
    if (p->has_vae && (num_points * 3) % 64 == 0) {
        const int P3 = num_points * 3;
        if (tile_w(p, p->vd0.w, 256, 0, 256, 256, &p->t_vd0) || tile_w(p, p->vd2.w, 256, 0, 512, 256, &p->t_vd2) ||
            tile_w(p, p->vd4.w, 512, 0, P3, 512, &p->t_vd4) || tile_w(p, p->vout.w, P3, 0, P3, P3, &p->t_vout))
            return 1;
    }
    {
        // the persistent kernel needs a cooperative launch of one CTA per SM; without it (or without room for its 187 KB of
        // shared memory) the handle keeps working on the launch-per-layer CUDA-graph path
        int coop = 0;
        CU(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device));
        if (!coop || latent_mk_grid(p->num_sms, &p->mk_grid) != cudaSuccess) { p->mk_grid = 0; cudaGetLastError(); }
    }
    CU(cudaDeviceSynchronize());
    *out = h.release();
    return 0;
}

static int lp_alloc(LatentPlan* pl, float** out, size_t n) {
    void* p = nullptr;
    CU(cudaMalloc(&p, n * sizeof(float)));
    pl->owned.push_back(p);
    *out = static_cast<float*>(p);
    return 0;
}

static int get_plan(pcd_latent* h, int B, LatentPlan** out) {
    if (LatentPlan* hit = h->plans.find(B)) { *out = hit; return 0; }
    h->plans.make_room();
    auto pl = std::unique_ptr<LatentPlan>(new LatentPlan());
    pl->B = B;
    const size_t b = B;
    if (lp_alloc(pl.get(), &pl->zbuf, b * 256) || lp_alloc(pl.get(), &pl->temb, b * 256) || lp_alloc(pl.get(), &pl->z1, b * 128) || lp_alloc(pl.get(), &pl->z2, b * 256) ||
        lp_alloc(pl.get(), &pl->z3, b * 512) || lp_alloc(pl.get(), &pl->z4, b * 1024) || lp_alloc(pl.get(), &pl->g0, b * 2048) ||
        lp_alloc(pl.get(), &pl->g1, b * 4096) || lp_alloc(pl.get(), &pl->r, b * 1024) || lp_alloc(pl.get(), &pl->d4, b * 1024) ||
        lp_alloc(pl.get(), &pl->d3, b * 512) || lp_alloc(pl.get(), &pl->d2, b * 256) || lp_alloc(pl.get(), &pl->d1, b * 128) ||
        lp_alloc(pl.get(), &pl->o0, b * 128) || lp_alloc(pl.get(), &pl->eps, b * 256) ||
        lp_alloc(pl.get(), &pl->partial, 32 * b * 1024 > 2 * b * 4096 ? 32 * b * 1024 : 2 * b * 4096))
        return 1;
    void* p = nullptr;
    CU(cudaMalloc(&p, sizeof(int))); pl->owned.push_back(p); pl->step = static_cast<int*>(p);
    CU(cudaMemset(pl->step, 0, sizeof(int)));
    CU(cudaMalloc(&p, sizeof(LatentCall))); pl->owned.push_back(p); pl->call = static_cast<LatentCall*>(p);
    *out = h->plans.insert(B, std::move(pl));
    return 0;
}

// out[B, cout] = act( [a0 | a1] W^T + b ), then optional GroupNorm(8)+ReLU in place.  Skinny problems (few
// 64x64 tiles) are split along K so all SMs stream weights; partial sums are reduced in a fixed order.
static int lin_op(pcd_latent* h, float* partial, size_t partial_cap, const Lin& L, const float* a0, int k0, const float* a1, int k1,
                  float* out, int B, bool relu, cudaStream_t s, int* launched) {
    if (k0 + k1 != L.cin) return fail("latent: K mismatch");
    int splits = partial ? simt_pick_splits(B, L.cout, L.cin, h->num_sms) : 1;
    while (splits > 1 && static_cast<size_t>(splits) * B * L.cout > partial_cap) splits /= 2;
    SimtGemmParams p{};
    p.A0 = a0; p.lda0 = k0; p.K0 = k0; p.A1 = a1; p.lda1 = k1; p.K1 = k1;
    p.W = L.w; p.ldw = L.cin; p.M = B; p.Nout = L.cout; p.out = out; p.ldo = L.cout;
    p.bias = L.b; p.bias_sample_stride = 0; p.rows_per_sample = 1 << 30; p.relu = (relu && !L.gamma) ? 1 : 0;
    p.partial = splits > 1 ? partial : nullptr; p.splits = splits;
    CU(launch_gemm_simt(EPI_STORE, p, s));
    ++*launched;
    if (L.gamma) {
        CU(launch_groupnorm_relu(out, partial, splits > 1 ? splits : 0, L.b, L.gamma, L.beta, B, L.cout, s));
        ++*launched;
    } else if (splits > 1) {
        CU(launch_splitk_reduce(partial, splits, L.b, out, B, L.cout, p.relu, s));
        ++*launched;
    }
    return 0;
}

static int run_latent_step(pcd_latent* h, LatentPlan* pl, const float* z_in, cudaStream_t s, bool advance) {
    int n = 0;
    const int B = pl->B;
    const size_t pcap = static_cast<size_t>(32) * B * 1024 > static_cast<size_t>(2) * B * 4096 ? static_cast<size_t>(32) * B * 1024 : static_cast<size_t>(2) * B * 4096;
#define lin_op(...) lin_op(h, pl->partial, pcap, __VA_ARGS__)
    CU(launch_latent_time(B, pl->call, h->freqs, h->W1T, h->b1, h->W2T, h->b2, pl->temb, s)); ++n;
    // cat([z, t_emb]) (networks.py:1068) is a two-source K-concatenated GEMM
    if (lin_op(h->enc1, z_in, 256, pl->temb, 256, pl->z1, B, true, s, &n)) return 1;
    if (lin_op(h->enc2, pl->z1, 128, nullptr, 0, pl->z2, B, true, s, &n)) return 1;
    if (lin_op(h->enc3, pl->z2, 256, nullptr, 0, pl->z3, B, true, s, &n)) return 1;
    if (lin_op(h->enc4, pl->z3, 512, nullptr, 0, pl->z4, B, true, s, &n)) return 1;
    if (lin_op(h->gf0, pl->z4, 1024, nullptr, 0, pl->g0, B, true, s, &n)) return 1;
    if (lin_op(h->gf3, pl->g0, 2048, nullptr, 0, pl->g1, B, true, s, &n)) return 1;
    if (lin_op(h->ref4, pl->z4, 1024, nullptr, 0, pl->r, B, false, s, &n)) return 1;
    if (lin_op(h->dec4, pl->g1, 4096, pl->r, 1024, pl->d4, B, true, s, &n)) return 1;   // cat([global, refine4(z4)]) :1080
    if (lin_op(h->ref3, pl->z3, 512, nullptr, 0, pl->r, B, false, s, &n)) return 1;
    if (lin_op(h->dec3, pl->d4, 1024, pl->r, 512, pl->d3, B, true, s, &n)) return 1;
    if (lin_op(h->ref2, pl->z2, 256, nullptr, 0, pl->r, B, false, s, &n)) return 1;
    if (lin_op(h->dec2, pl->d3, 512, pl->r, 256, pl->d2, B, true, s, &n)) return 1;
    if (lin_op(h->ref1, pl->z1, 128, nullptr, 0, pl->r, B, false, s, &n)) return 1;
    if (lin_op(h->dec1, pl->d2, 256, pl->r, 128, pl->d1, B, true, s, &n)) return 1;
    if (lin_op(h->out0, pl->d1, 128, nullptr, 0, pl->o0, B, true, s, &n)) return 1;
    if (lin_op(h->out2, pl->o0, 128, nullptr, 0, pl->eps, B, false, s, &n)) return 1;
    CU(launch_latent_update(pl->eps, pl->call, B, 256, s)); ++n;
    if (advance) { CU(launch_advance_step(pl->step, s)); ++n; }
#undef lin_op
    pl->kernels_per_step = n;
    return 0;
}

// ---- persistent-kernel path (latent_mk.cu) ------------------------------------------------------------------------------
static bool latent_legacy() { return std::getenv("PCD_LATENT_LEGACY") != nullptr; }

// K splits of a tiled Linear: fill the 148 CTAs of the persistent kernel (whole waves), at least two 32-wide chunks per split
// (one for the small layers), at most 16 splits and 4 N (>= 8192; 16384 for 128-column tiles) workspace floats per row.  Depends on the layer shape only -- never on the batch -- so a sample's
// result does not depend on the batch it is in.
static int pick_ks(int N, int K) {
    const int bn = lt_bn(N, K);
    const int tiles = N / bn, chunks = K / 32;
    int best = 1;
    double best_eff = -1.0;
    int cap = 4 * N > 8192 ? 4 * N : 8192;           // workspace floats per row (get_plan allocates 32768 per row)
    if (bn == 128 && cap < 16384) cap = 16384;
    for (int d = 1; d <= chunks && d <= 16; ++d) {
        // small layers (<= 12 chunks of K) may go down to ONE chunk per split: their phase time is a chain of latencies plus
        // ~0.75 us per chunk, and the extra partial sums are a few KB
        const int min_chunks = chunks <= 12 ? 1 : 2;
        if (chunks % d || (d > 1 && (chunks / d < min_chunks || d * N > cap))) continue;
        const int items = tiles * d;
        const double eff = static_cast<double>(items) / (((items + 147) / 148) * 148);
        if (eff > best_eff + 1e-9) { best_eff = eff; best = d; }
    }
    return best;
}

static LtOp lt_gemm(const float* A0, int K0, const float* A1, int K1, const float* Wtiled, int N, int ks, int epi, float* out,
                    const float* bias, int rows_mode) {
    LtOp o{};
    o.kind = LT_GEMM; o.rows_mode = rows_mode;
    o.A0 = A0; o.lda0 = K0; o.K0 = K0; o.A1 = A1; o.lda1 = K1; o.K1 = K1;
    o.W = Wtiled; o.kchunks = (K0 + K1) / 32; o.N = N; o.ks = ks; o.chunks_per_split = (K0 + K1) / 32 / ks;
    o.bn = epi == LT_PARTIAL ? lt_bn(N, K0 + K1) : 64;
    o.epi = epi; o.out = out; o.ldo = N; o.bias = bias; o.bias_mode = 0; o.bias_ld = 0;
    return o;
}

static LtOp lt_norm(const float* partial, int nsplit, const float* bias, const float* gamma, const float* beta, int act, int C,
                    float* out) {
    LtOp o{};
    o.kind = LT_NORM; o.partial = partial; o.nsplit = nsplit; o.bias = bias; o.gamma = gamma; o.beta = beta; o.act = act; o.C = C;
    o.out = out; o.ldo = C;
    return o;
}

// Linear (+ GroupNorm(8) + ReLU) = split-K tile jobs into the workspace, then the fixed-order reduce / normalise phase
static void lt_layer(LtProgram* P, int* n, const Lin& L, const float* Wtiled, const float* A0, int K0, const float* A1, int K1,
                     float* partial, float* out, int act) {
    const int ks = pick_ks(L.cout, L.cin);
    P->ops[(*n)++] = lt_gemm(A0, K0, A1, K1, Wtiled, L.cout, ks, LT_PARTIAL, partial, nullptr, 0);
    P->ops[(*n)++] = lt_norm(partial, ks, L.b, L.gamma, L.beta, act, L.cout, out);
}

static int mk_prepare(pcd_latent* h, LatentPlan* pl, int R) {
    if (!pl->bar) {
        void* p = nullptr;
        CU(cudaMalloc(&p, sizeof(unsigned) * kLtBarrierWords)); pl->owned.push_back(p); pl->bar = static_cast<unsigned*>(p);
        CU(cudaMalloc(&p, sizeof(LtProgram))); pl->owned.push_back(p); pl->prog = static_cast<LtProgram*>(p);
    }
    if (R <= pl->Rcap) return 0;
    CU(cudaDeviceSynchronize());     // an earlier launch may still be walking the program that is about to be rebuilt
    const size_t r = R;
    if (lp_alloc(pl, &pl->emb, r * 256) || lp_alloc(pl, &pl->th, r * 256) || lp_alloc(pl, &pl->tembR, r * 256) ||
        lp_alloc(pl, &pl->bias1, r * 128))
        return 1;
    pl->Rcap = R;
    LtProgram P{};
    int n = 0;
    // once per call, one row per time row: sinusoidal embedding -> time MLP (networks.py:977-981, 1064-1065) -> the t_emb half
    // of enc1 (cat([z, t_emb]), :1068) as a per-row bias:  bias1[r] = W_enc1[:, 256:] temb[r] + b_enc1
    LtOp e{};
    e.kind = LT_EMB; e.rows_mode = 1; e.out = pl->emb; e.bias = h->freqs;
    P.ops[n++] = e;
    P.ops[n++] = lt_gemm(pl->emb, 256, nullptr, 0, h->t_tw0, 256, 1, LT_BIAS_SILU, pl->th, h->b1, 1);
    P.ops[n++] = lt_gemm(pl->th, 256, nullptr, 0, h->t_tw2, 256, 1, LT_BIAS, pl->tembR, h->b2, 1);
    P.ops[n++] = lt_gemm(pl->tembR, 256, nullptr, 0, h->t_enc1t, 128, 1, LT_BIAS, pl->bias1, h->enc1.b, 1);
    P.n_pre = n;
    // every reverse step (the head reads the caller's z).  enc1 + enc2 as ONE rows-per-CTA phase (latent_mk.cu, head_phase), for every
    // batch size so that a row's arithmetic does not depend on the batch it is in
    {
        LtOp hd = lt_norm(nullptr, 0, pl->bias1, h->enc1.gamma, h->enc1.beta, 1, 128, pl->z1);
        hd.kind = LT_HEAD; hd.bias_mode = 1; hd.bias_ld = 128;
        hd.W2 = h->enc1zT; hd.W3 = h->enc2T; hd.b3 = h->enc2.b; hd.gamma2 = h->enc2.gamma; hd.beta2 = h->enc2.beta; hd.out2 = pl->z2;
        P.ops[n++] = hd;
    }
    lt_layer(&P, &n, h->enc3, h->t_enc3, pl->z2, 256, nullptr, 0, pl->partial, pl->z3, 1);
    lt_layer(&P, &n, h->enc4, h->t_enc4, pl->z3, 512, nullptr, 0, pl->partial, pl->z4, 1);
    lt_layer(&P, &n, h->gf0, h->t_gf0, pl->z4, 1024, nullptr, 0, pl->partial, pl->g0, 1);
    lt_layer(&P, &n, h->gf3, h->t_gf3, pl->g0, 2048, nullptr, 0, pl->partial, pl->g1, 1);
    lt_layer(&P, &n, h->dec4c, h->t_dec4, pl->g1, 4096, pl->z4, 1024, pl->partial, pl->d4, 1);   // cat([global, refine4(z4)]) :1080
    lt_layer(&P, &n, h->dec3c, h->t_dec3, pl->d4, 1024, pl->z3, 512, pl->partial, pl->d3, 1);
    lt_layer(&P, &n, h->dec2c, h->t_dec2, pl->d3, 512, pl->z2, 256, pl->partial, pl->d2, 1);
    // dec1 (from d2 and z1), its GroupNorm, output.0, output.2 and the update as ONE rows-per-CTA phase (latent_mk.cu, tail_phase), for
    // every batch size so that a row's arithmetic does not depend on the batch it is in
    {
        LtOp t = lt_norm(nullptr, 0, h->dec1c.b, h->dec1c.gamma, h->dec1c.beta, 1, 128, nullptr);
        t.kind = LT_TAIL; t.W2 = h->out0T; t.b2 = h->out0.b; t.W3 = h->out2T; t.b3 = h->out2.b;
        t.A0 = pl->d2; t.lda0 = 256; t.K0 = 256; t.A1 = pl->z1; t.lda1 = 128; t.K1 = 128; t.W = h->dec1cT;
        P.ops[n++] = t;
    }
    P.n_loop = n - P.n_pre;
    CU(cudaMemcpy(pl->prog, &P, sizeof(P), cudaMemcpyHostToDevice));
    return 0;
}

static bool mk_decode_ok(const pcd_latent* h) {
    const int P3 = h->num_points * 3;
    return h->has_vae && h->t_vout && h->mk_grid > 0 && !latent_legacy() && P3 % 64 == 0 && 1LL * pick_ks(P3, 512) * P3 <= 32768 &&
           1LL * pick_ks(P3, P3) * P3 <= 32768;
}

static int mk_decode(pcd_latent* h, const float* z, float* out, int B, cudaStream_t s) {
    LatentPlan* pl = nullptr;
    if (get_plan(h, B, &pl)) return 1;
    if (mk_prepare(h, pl, 1)) return 1;
    const int P3 = h->num_points * 3;
    if (!pl->dprog) {
        const size_t b = B;
        if (lp_alloc(pl, &pl->da, b * 256) || lp_alloc(pl, &pl->db, b * 512) || lp_alloc(pl, &pl->dc, b * P3)) return 1;
        void* p = nullptr;
        CU(cudaMalloc(&p, sizeof(LtProgram))); pl->owned.push_back(p); pl->dprog = static_cast<LtProgram*>(p);
        LtProgram P{};
        int n = 0;
        // SimplePointNetVAE.decode (networks.py:1144-1154, 1219-1231): 256 -> 256 -> 512 -> 3P (ReLU each) -> 3P
        P.ops[n++] = lt_gemm(nullptr, 256, nullptr, 0, h->t_vd0, 256, 1, LT_BIAS_RELU, pl->da, h->vd0.b, 0);
        P.ops[n++] = lt_gemm(pl->da, 256, nullptr, 0, h->t_vd2, 512, 1, LT_BIAS_RELU, pl->db, h->vd2.b, 0);
        lt_layer(&P, &n, h->vd4, h->t_vd4, pl->db, 512, nullptr, 0, pl->partial, pl->dc, 1);
        lt_layer(&P, &n, h->vout, h->t_vout, pl->dc, P3, nullptr, 0, pl->partial, nullptr, 0);    // out == nullptr: the caller's buffer
        P.n_pre = 0; P.n_loop = n;
        CU(cudaMemcpy(pl->dprog, &P, sizeof(P), cudaMemcpyHostToDevice));
    }
    LatentCall ca{};
    ca.z = const_cast<float*>(z); ca.eps_out = out; ca.B = B; ca.D = 256; ca.mode = 0;
    CU(cudaMemcpyAsync(pl->call, &ca, sizeof(ca), cudaMemcpyHostToDevice, s));
    LAUNCH(launch_latent_mk(pl->dprog, pl->call, 1, 1, 1, pl->bar, h->mk_grid, s));
    return 0;
}

extern "C" int pcd_latent_forward(pcd_latent* h, const float* z, const float* t, float* eps, int32_t B, void* stream) {
    REQ(h && z && t && eps && B > 0, "bad argument");
    REQ(h->has_model, "decoder-only handle: it was created without the latent denoiser's model.* tensors");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    LatentPlan* pl = nullptr;
    if (get_plan(h, B, &pl)) return 1;
    LatentCall ca{};
    ca.z = const_cast<float*>(z); ca.eps_out = eps; ca.t_in = t; ca.step_ptr = pl->step; ca.B = B; ca.D = 256; ca.mode = 0;
    CU(cudaMemcpyAsync(pl->call, &ca, sizeof(ca), cudaMemcpyHostToDevice, s));
    if (h->mk_grid > 0 && !latent_legacy()) {
        if (mk_prepare(h, pl, B)) return 1;
        LAUNCH(launch_latent_mk(pl->prog, pl->call, 1, B, 1, pl->bar, h->mk_grid, s));
        return 0;
    }
    if (run_latent_step(h, pl, z, s, false)) return 1;
    g_pcd_launches.fetch_add(pl->kernels_per_step, std::memory_order_relaxed);
    return 0;
}

extern "C" int pcd_latent_sample(pcd_latent* h, const float* sched, int32_t S, float* z, const float* noise, uint64_t seed,
                                 uint64_t sample_offset, int32_t B, void* stream) {
    return pcd_latent_sample_rows(h, sched, S, 1, z, noise, seed, sample_offset, B, stream);
}

extern "C" int pcd_latent_sample_rows(pcd_latent* h, const float* sched, int32_t S, int32_t rows_per_step, float* z,
                                      const float* noise, uint64_t seed, uint64_t sample_offset, int32_t B, void* stream) {
    REQ(h && sched && z && B > 0 && S > 0, "bad argument");
    REQ(rows_per_step == 1 || rows_per_step == B, "rows_per_step must be 1 (schedule shared by the batch) or B (one row per sample)");
    REQ(h->has_model, "decoder-only handle: it was created without the latent denoiser's model.* tensors");
    const int rows = rows_per_step;
    REQ(rows == 1 || (h->mk_grid > 0 && !latent_legacy()), "per-sample schedule rows need the persistent latent kernel");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    LatentPlan* pl = nullptr;
    if (get_plan(h, B, &pl)) return 1;
    if (S * rows > pl->sched_cap) {
        if (lp_alloc(pl, &pl->sched, static_cast<size_t>(kSchedRow) * S * rows)) return 1;
        pl->sched_cap = S * rows;
    }
    CU(cudaMemcpyAsync(pl->sched, sched, sizeof(float) * kSchedRow * S * rows, cudaMemcpyHostToDevice, s));
    if (h->mk_grid > 0 && !latent_legacy()) {
        // one cooperative launch runs all S steps in place on the caller's z
        if (mk_prepare(h, pl, S)) return 1;
        LatentCall ca{};
        ca.z = z; ca.sched = pl->sched; ca.sched_rows = rows; ca.noise = noise; ca.noise_step_stride = static_cast<long long>(B) * 256;
        ca.seed = seed; ca.sample_offset = sample_offset; ca.B = B; ca.D = 256; ca.mode = 1;
        CU(cudaMemcpyAsync(pl->call, &ca, sizeof(ca), cudaMemcpyHostToDevice, s));
        LAUNCH(launch_latent_mk(pl->prog, pl->call, S, S, 0, pl->bar, h->mk_grid, s));
        return 0;
    }
    CU(cudaMemsetAsync(pl->step, 0, sizeof(int), s));
    LatentCall ca{};
    // the loop runs on a plan-owned copy of z so the captured graph does not depend on the caller's pointer
    CU(cudaMemcpyAsync(pl->zbuf, z, sizeof(float) * B * 256, cudaMemcpyDeviceToDevice, s));
    ca.z = pl->zbuf; ca.t_in = nullptr; ca.sched = pl->sched; ca.step_ptr = pl->step; ca.noise = noise;
    ca.noise_step_stride = static_cast<long long>(B) * 256; ca.seed = seed; ca.sample_offset = sample_offset;
    ca.B = B; ca.D = 256; ca.mode = 1;
    CU(cudaMemcpyAsync(pl->call, &ca, sizeof(ca), cudaMemcpyHostToDevice, s));
    if (std::getenv("PCD_NO_GRAPH") == nullptr) {
        if (!pl->exec) {
            cudaStream_t cs;
            CU(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
            CU(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
            int rc = run_latent_step(h, pl, pl->zbuf, cs, true);
            cudaError_t e = cudaStreamEndCapture(cs, &pl->graph);
            cudaStreamDestroy(cs);
            if (rc) return 1;
            CU(e);
            CU(cudaGraphInstantiate(&pl->exec, pl->graph, 0));
        }
        for (int i = 0; i < S; ++i) CU(cudaGraphLaunch(pl->exec, s));
    } else {
        for (int i = 0; i < S; ++i)
            if (run_latent_step(h, pl, pl->zbuf, s, true)) return 1;
    }
    CU(cudaMemcpyAsync(z, pl->zbuf, sizeof(float) * B * 256, cudaMemcpyDeviceToDevice, s));
    g_pcd_launches.fetch_add(static_cast<long long>(pl->kernels_per_step) * S, std::memory_order_relaxed);
    return 0;
}

// FoldingDecoder.forward (networks.py:1484-1509) on rows = (sample, grid point)
// The folds on the tcgen05 split-precision GEMM (gemm_tc.cu, NP = 3, fp16 hi / lo planes): rows = B * 1024 is a multiple of 128,
// and its 8 B row blocks are always an even number for the CTA pairs.
static int folding_decode(pcd_latent* h, const float* z, float* out, int B, cudaStream_t s) {
    const long long rows = static_cast<long long>(B) * 1024;
    const int P = h->upsample.cout;
    REQ(2 * rows < (1LL << 31), "FoldingDecoder: too many latents per call (decode in chunks)");
    float *bz = nullptr, *o1 = nullptr, *cm = nullptr, *U = nullptr;
    void *h1 = nullptr, *h3 = nullptr;
    CU(cudaMallocAsync(reinterpret_cast<void**>(&bz), sizeof(float) * B * 512, s));
    CU(cudaMallocAsync(&h1, sizeof(uint16_t) * 2 * rows * 512, s));
    CU(cudaMallocAsync(&h3, sizeof(uint16_t) * 2 * rows * 512, s));
    CU(cudaMallocAsync(reinterpret_cast<void**>(&o1), sizeof(float) * rows * 3, s));
    CU(cudaMallocAsync(reinterpret_cast<void**>(&cm), sizeof(float) * rows * 3, s));
    CU(cudaMallocAsync(reinterpret_cast<void**>(&U), sizeof(float) * 3 * B * P, s));
    int n = 0;
    auto run = [&]() -> int {
        CUtensorMap ta, tb, to;
        if (make_tmap(&ta, h1, 2 * rows, 512, 512, 128) || make_tmap(&to, h3, 2 * rows, 512, 512, 32)) return 1;
        for (int f = 0; f < 2; ++f) {
            const pcd_latent::Fold& F = h->fold[f];
            // per-sample bias: the latent columns of the fold's first conv (z is repeated over the grid, :1496)
            if (lin_op(h, nullptr, 0, F.wz, z, 256, nullptr, 0, bz, B, false, s, &n)) return 1;
            CU(launch_fold_first(F.kin, f == 0 ? h->grid : o1, f == 0 ? 1024 : 0, F.wg, bz, rows, 1024, h1, s)); ++n;
            if (make_tmap(&tb, F.wab16, 2 * 512, 512, 512, 128)) return 1;       // CTA pair: each CTA stages half of the 256-column tile
            TcGemmParams p{};
            p.num_m_blocks = static_cast<int>(rows / 128); p.num_n_blocks = 2; p.kb0 = 8; p.kb1 = 0;
            p.a_plane_rows = static_cast<int>(rows); p.b_plane_rows = 512; p.out_plane_rows = static_cast<int>(rows);
            p.out = static_cast<__nv_bfloat16*>(h3); p.ldo = 512; p.bias = F.wab.b; p.bias_sample_stride = 0;
            p.rows_per_sample = 1 << 30; p.relu = 1; p.f16 = 1;
            CU(launch_gemm_tc(256, EPI_STORE, 3, 2, 2, 1, ta, ta, tb, to, p, h->num_sms, s)); ++n;
            CU(launch_fold_tail16(h3, F.wbc.w, F.wbc.b, F.wc2, F.bc2, rows, 1024, f == 1 ? 1 : 0, f == 1 ? cm : o1, s)); ++n;
        }
        // upsample = Linear(1024 -> num_points) ACROSS the point axis of [B, 3, 1024] (:1507-1508)
        if (lin_op(h, nullptr, 0, h->upsample, cm, 1024, nullptr, 0, U, 3 * B, false, s, &n)) return 1;
        CU(launch_fold_transpose(U, B, P, out, s)); ++n;
        return 0;
    };
    const int rc = run();
    cudaFreeAsync(bz, s); cudaFreeAsync(h1, s); cudaFreeAsync(h3, s); cudaFreeAsync(o1, s); cudaFreeAsync(cm, s); cudaFreeAsync(U, s);
    g_pcd_launches.fetch_add(n, std::memory_order_relaxed);
    return rc;
}

extern "C" int pcd_vae_decode(pcd_latent* h, const float* z, float* out, int32_t B, void* stream) {
    REQ(h && z && out && B > 0, "bad argument");
    REQ(h->has_vae || h->has_folding, "handle was created without decoder weights (SimplePointNetVAE: vae.decoder.*, "
                                      "vae.output_layer.*; PointNetVAE: vae.decoder.fold1/fold2/upsample.*)");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (h->has_folding) return folding_decode(h, z, out, B, s);
    if (mk_decode_ok(h)) return mk_decode(h, z, out, B, s);
    const int P3 = h->num_points * 3;
    float *a = nullptr, *b = nullptr, *c = nullptr;
    CU(cudaMallocAsync(reinterpret_cast<void**>(&a), sizeof(float) * B * 256, s));
    CU(cudaMallocAsync(reinterpret_cast<void**>(&b), sizeof(float) * B * 512, s));
    CU(cudaMallocAsync(reinterpret_cast<void**>(&c), sizeof(float) * B * P3, s));
    int n = 0;
    int rc = lin_op(h, nullptr, 0, h->vd0, z, 256, nullptr, 0, a, B, true, s, &n) || lin_op(h, nullptr, 0, h->vd2, a, 256, nullptr, 0, b, B, true, s, &n) ||
             lin_op(h, nullptr, 0, h->vd4, b, 512, nullptr, 0, c, B, true, s, &n) || lin_op(h, nullptr, 0, h->vout, c, P3, nullptr, 0, out, B, false, s, &n);
    cudaFreeAsync(a, s); cudaFreeAsync(b, s); cudaFreeAsync(c, s);
    g_pcd_launches.fetch_add(n, std::memory_order_relaxed);
    return rc;
}

extern "C" int pcd_latent_philox_normal(uint64_t seed, uint64_t sample_offset, int32_t step, float* out, int32_t B, int32_t D,
                                        void* stream) {
    REQ(out && B > 0 && D > 0, "bad argument");
    LAUNCH(launch_latent_philox_fill(out, seed, sample_offset, step, B, D, static_cast<cudaStream_t>(stream)));
    return 0;
}
