// Host-side helpers shared by api.cu and api_latent.cu.
#pragma once
#include <atomic>
#include <cstdlib>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/pcd_b200.h"

extern thread_local std::string g_pcd_err;
extern std::atomic<long long> g_pcd_launches;

inline int fail(const std::string& m) { g_pcd_err = m; return 1; }
#define CU(expr)                                                                                         \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess)                                                                           \
            return fail(std::string(#expr) + ": " + cudaGetErrorString(_e) + " @" + std::to_string(__LINE__)); \
    } while (0)
#define LAUNCH(expr)                                                                                     \
    do {                                                                                                 \
        CU(expr);                                                                                        \
        g_pcd_launches.fetch_add(1, std::memory_order_relaxed);                                          \
    } while (0)
#define REQ(cond, msg)                                                                                   \
    do {                                                                                                 \
        if (!(cond)) return fail(std::string("pcd: ") + msg);                                            \
    } while (0)

// TMA descriptors (defined in api.cu)
#include <cuda.h>
int make_tmap(CUtensorMap* tm, const void* base, long long rows, long long cols, long long ld, int box_rows);
int make_tmap5(CUtensorMap* tm, const void* base, int C, int W, int H, int D, long long nb, long long sw, long long sh,
               long long sd, long long sb, int bw, int bh, int bd, int bb, int es = 1);

int make_tmap_out32(CUtensorMap* tm, const void* base, long long rows, long long cols, long long ld);

// Tile shape of one tcgen05 GEMM launch (gemm_tc.cu) of a per-point layer: tile columns `bn`, cluster size `cl` (CTA pairs when the
// A-role blocks pair up), the pair MMA (`two_sm`) and the STORE tile order, from the epilogue, the MMA passes per k-step `np`, the
// point rows M, the output channels and K.  Shared by every handle that runs per-point layers (defined in api.cu).
struct TcShape { int bn = 0, cl = 1, two_sm = 0, tile_order = 0; };
TcShape tc_shape(int epi, int np, long long M, int cout, int K, int num_sms);

// Per-handle plan cache.  A plan owns the workspace of one problem shape (GBs at full batch), so only the `cap` most recently
// used shapes stay resident (PCD_MAX_PLANS, default 4); the least recently used one is destroyed -- after a device
// synchronisation, its kernels may still be in flight -- BEFORE the workspace of a new shape is allocated.
template <class Key, class PlanT>
struct PlanCache {
    std::map<Key, std::unique_ptr<PlanT>> m;
    std::map<Key, unsigned long long> stamp;
    unsigned long long tick = 0;
    PlanT* last = nullptr;       // most recently used plan (debug taps read it)
    static size_t cap() {
        const char* c = std::getenv("PCD_MAX_PLANS");
        const int n = c ? std::atoi(c) : 4;
        return n < 1 ? 1 : static_cast<size_t>(n);
    }
    PlanT* find(const Key& k) {
        auto it = m.find(k);
        if (it == m.end()) return nullptr;
        stamp[k] = ++tick;
        return last = it->second.get();
    }
    void make_room() {
        while (m.size() >= cap()) {
            auto victim = stamp.begin();
            for (auto it = stamp.begin(); it != stamp.end(); ++it)
                if (it->second < victim->second) victim = it;
            cudaDeviceSynchronize();
            if (last == m[victim->first].get()) last = nullptr;
            m.erase(victim->first);
            stamp.erase(victim);
        }
    }
    PlanT* insert(const Key& k, std::unique_ptr<PlanT> p) {
        stamp[k] = ++tick;
        last = p.get();
        m[k] = std::move(p);
        return last;
    }
    bool empty() const { return m.empty(); }
    void clear() { m.clear(); stamp.clear(); last = nullptr; }
};

struct TensorTable {
    std::map<std::string, const pcd_named_tensor*> m;
    const pcd_named_tensor* get(const std::string& name, std::string* err) const {
        auto it = m.find(name);
        if (it == m.end()) { *err = "state_dict entry missing: " + name; return nullptr; }
        return it->second;
    }
};

inline bool fetch(const TensorTable& tt, const std::string& name, long long n_expected, const float** out,
                  std::string* err) {
    const pcd_named_tensor* t = tt.get(name, err);
    if (!t) return false;
    if (t->dtype != PCD_DTYPE_F32) { *err = "expected float32 for " + name; return false; }
    long long n = 1;
    for (int i = 0; i < t->ndim; ++i) n *= t->shape[i];
    if (n != n_expected) {
        *err = "shape mismatch for " + name + ": got " + std::to_string(n) + " elements, expected " + std::to_string(n_expected);
        return false;
    }
    *out = static_cast<const float*>(t->data);
    return true;
}

struct HostMat {   // folded fp32 layer on the host
    int cout = 0, k = 0;
    std::vector<float> w;   // [cout][k]
    std::vector<float> b;   // [cout]
};

// conv (k=1) followed by eval-mode BatchNorm1d folded into one affine map in double (defined in api.cu); bn empty = bare conv
bool fold_conv_bn(const TensorTable& tt, const std::string& conv, const std::string& bn, int cout, int cin, HostMat* out,
                  std::string* err);
