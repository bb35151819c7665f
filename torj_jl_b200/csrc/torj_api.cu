// Host side of libtorj_cuda.so: the C ABI declared in include/torj_cuda.h.
// Plain CUDA runtime; no torch types, no CPU fallback (every entry point needs a CUDA device).
#include <cuda_runtime.h>

#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <cstdio>
#include <memory>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/torj_cuda.h"
#include "torj_kernels.cuh"

using namespace torj;

static thread_local std::string g_err;

#define CK(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess) {                                                                          \
            char buf_[512];                                                                               \
            snprintf(buf_, sizeof buf_, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            g_err = buf_;                                                                                 \
            return 1;                                                                                     \
        }                                                                                                 \
    } while (0)

#define FAIL(msg) do { g_err = (msg); return 2; } while (0)

// Owning array of size() T in device memory (dev_array) or page-locked host memory (pinned_array); it converts to its
// pointer. The destructor frees it, so whoever destroys an owner makes the owning device current first.
template <bool PINNED>
struct CudaFree {
    void operator()(void* p) const { PINNED ? cudaFreeHost(p) : cudaFree(p); }
};
template <class T, bool PINNED>
class cuda_array {
    std::unique_ptr<T, CudaFree<PINNED>> p_;
    size_t n_ = 0;

  public:
    operator T*() const { return p_.get(); }
    size_t size() const { return n_; }
    // Unchanged size: nothing. Otherwise wait for st (a kernel or copy on it may still use the old buffer), free, then
    // allocate. A failed allocation leaves the array empty.
    cudaError_t resize(size_t count, cudaStream_t st) {
        if (count == n_) return cudaSuccess;
        cudaError_t e = p_ ? cudaStreamSynchronize(st) : cudaSuccess;
        if (e != cudaSuccess) return e;
        p_.reset();
        n_ = 0;
        if (count == 0) return cudaSuccess;
        T* raw = nullptr;
        e = PINNED ? cudaHostAlloc(&raw, count * sizeof(T), cudaHostAllocDefault) : cudaMalloc(&raw, count * sizeof(T));
        if (e != cudaSuccess) return e;
        p_.reset(raw);
        n_ = count;
        return cudaSuccess;
    }
};
template <class T>
using dev_array = cuda_array<T, false>;
template <class T>
using pinned_array = cuda_array<T, true>;

struct torj_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    bool gl_set = false;
    int num_sms = 0;
    int64_t launches = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;  // bracket the last k_trace launch
    bool ev_valid = false;
    struct torj_bundle* ws = nullptr;  // workspace of the one-shot torj_trace call, kept between calls
    dev_array<double2> d_warm_tab;     // set_extv! tables of the warm-plasma model (reference src/general_absorption.jl:8-13)
    int exact_sum = 0;                 // torj_ctx_set_exact_sum: later traces book profiles exactly (torj_exactsum.cuh)
};

// The Gauss-Legendre table lives in ONE __constant__ symbol per device (like the reference's module globals,
// src/constants.jl:7-8); this registry remembers what each device holds so that a second context on the device inherits
// it, identical re-initialisations are free, and a different table is written only after the whole device is idle.
struct GLRegistry {
    std::mutex mu;
    std::vector<std::vector<double>> tab;  // per device: n nodes then n weights; empty = never set
};
static GLRegistry g_gl;

static std::atomic<uint64_t> g_plasma_serial{0};  // torj_multi_* creates plasmas from one host thread per device

struct torj_plasma {
    torj_ctx* ctx = nullptr;
    uint64_t id = 0;  // unique per created plasma (addresses can be recycled)
    DevTables T{};
    dev_array<double2> dA;  // [nodes][3]
    dev_array<DevTables> dT;  // T mirrored in global memory
    // host copy of the V(psi_N) spline (reference src/plasma.jl:42-44)
    std::vector<double> vol_c;
    int n_vol = 0;
    double vol_x0 = 0, vol_h = 1;
};

struct torj_bundle {
    torj_ctx* ctx = nullptr;
    int64_t n = 0;
    BundleDev B{};
    int per_ray_fm = 0;
    // per-ray device buffers
    dev_array<double> d_pos, d_dir, d_w, d_freq, d_u0, d_s0, d_psil, d_Pf, d_Pdep;
    dev_array<int> d_mode, d_status, d_npts;
    dev_array<double> d_ufinal;  // [7][n] state at retirement
    // deposition
    int n_psi = 0;
    dev_array<double> d_edges, d_bins, d_dV, d_profile;
    dev_array<unsigned long long> d_queue, d_counters;
    // segment hand-off (allocated on first use)
    dev_array<double> d_hand;
    dev_array<int> d_segdone, d_left;
    int h_left = 0;  // source of the copy into d_left (outlives the call)
    dev_array<int> d_life;                      // [n + 1]: predicted life of every ray in segments, then the maximum
    // trajectory window; d_tprof is sized by the trace's n_psi
    int64_t traj_first = 0, traj_count = 0;
    int traj_max = 0;
    dev_array<double> d_ts, d_txyz, d_tP, d_tdP, d_tprof;
    // what the device copies of psi_edges / dV were computed from (skips the re-upload when unchanged): the edges and the
    // plasma of every dV row (one row, or one per beam for a plasma set)
    std::vector<double> h_edges;
    std::vector<uint64_t> dV_plasmas;
    // beams
    int n_beams = 1, prof_rows = 0;
    dev_array<int> d_beam;
    // plasma set of the last torj_bundle_trace_plasmas (n_plasmas > 1): table bases then DevTables pointers, and the plasma
    // of every beam, as last uploaded
    std::vector<const void*> h_set;
    std::vector<int> h_beam_plasma;
    dev_array<const void*> d_set;
    dev_array<int> d_beam_plasma;
    int dV_rows = 1;  // rows of d_dV the last trace used
    // exact-sum mode (allocated on first use): the words of every bin and the status words, torj_xs_buffer_words(bins)
    dev_array<long long> d_xs;
    bool xs_last = false;  // the last trace booked exactly: results check the status words
    double w_max = 0.0;    // max |weight| of the host weights (infinite for a NaN); -1: weights made on the device
};

// Error paths: temporaries are owned by dev_array, objects under construction by a guard that destroys them unless the
// function reaches its end (every CK / FAIL returns early).
template <class T, void (*Destroy)(T*)>
struct Guard {
    T* p;
    explicit Guard(T* q) : p(q) {}
    ~Guard() { if (p) Destroy(p); }
    T* release() { T* q = p; p = nullptr; return q; }
    Guard(const Guard&) = delete;
    Guard& operator=(const Guard&) = delete;
};

static int set_device(const torj_ctx* c) {
    CK(cudaSetDevice(c->device));
    // Start every entry point from a clean error state: cudaGetLastError() after a kernel launch must report that launch,
    // not a non-sticky error some earlier, unrelated runtime call of this host thread (ours or the application's) left behind.
    (void)cudaGetLastError();
    return 0;
}

extern "C" {

const char* torj_last_error(void) { return g_err.c_str(); }
int torj_abi_version(void) { return TORJ_ABI_VERSION; }

void torj_options_default(torj_options* o) {
    o->scheme = 0;
    o->n_segments = 100;
    o->dtmax = 1e-4;
    o->abstol = 1e-6;
    o->reltol = 1e-6;
    o->psi_stop = 1.0;
    o->p_stop = 1e-6;
    o->te_min = 20.0;
    o->max_harmonic = 3;
    o->schedule = 0;
    o->absorption_model = 0;
    o->lanes_per_ray = 0;
    o->reserved_ = 0;
    o->max_steps_per_segment = 100000;
    o->alpha_floor = 1e-14;
}

static void fill_tableaux(Tableau t[2]) {
    memset(t, 0, 2 * sizeof(Tableau));
    double(*a)[7] = t[0].a;  // Tsit5
    a[1][0] = 0.161;
    a[2][0] = -0.008480655492356989; a[2][1] = 0.335480655492357;
    a[3][0] = 2.8971530571054935; a[3][1] = -6.359448489975075; a[3][2] = 4.3622954328695815;
    a[4][0] = 5.325864828439257; a[4][1] = -11.748883564062828; a[4][2] = 7.4955393428898365; a[4][3] = -0.09249506636175525;
    a[5][0] = 5.86145544294642; a[5][1] = -12.92096931784711; a[5][2] = 8.159367898576159; a[5][3] = -0.071584973281401;
    a[5][4] = -0.028269050394068383;
    a[6][0] = 0.09646076681806523; a[6][1] = 0.01; a[6][2] = 0.4798896504144996; a[6][3] = 1.379008574103742;
    a[6][4] = -3.290069515436081; a[6][5] = 2.324710524099774;
    const double bt[7] = {-0.00178001105222577714, -0.0008164344596567469, 0.007880878010261995, -0.1447110071732629,
                          0.5823571654525552, -0.45808210592918697, 0.015151515151515152};
    for (int i = 0; i < 7; ++i) t[0].bt[i] = bt[i];
    a = t[1].a;  // OwrenZen3
    a[1][0] = 12.0 / 23.0;
    a[2][0] = -68.0 / 375.0; a[2][1] = 368.0 / 375.0;
    a[3][0] = 31.0 / 144.0; a[3][1] = 529.0 / 1152.0; a[3][2] = 125.0 / 384.0;
    t[1].bt[0] = 25.0 / 144.0; t[1].bt[1] = -575.0 / 1152.0; t[1].bt[2] = 125.0 / 384.0;
}

// Warm-plasma model: quadrature tables of set_extv! (reference src/general_absorption.jl:8-13, src/constants.jl:1-4), the
// combination weights of dieltens_maxw_fr (:1069,1081-1082), fact (:240-257) and 1/exp(gammln(m + 3/2)) with the
// reference's own 6-term Lanczos gammln (:265-283) — restated here because ssbi (:298) takes its Gamma values from it.
static double ref_fact(int k) {
    double r = 1.0;
    for (int i = 2; i <= k; ++i) r *= (double)i;
    return r;
}
static double ref_gammln(double x) {
    const double stp = 2.5066282746310005;
    const double cof[6] = {76.18009172947146, -86.50532032941677, 24.01409824083091, -1.231739572450155, 0.1208650973866179e-2,
                           -0.5395239384953e-5};
    double y = x, tmp = x + 5.5;
    tmp = (x + 0.5) * std::log(tmp) - tmp;
    double ser = 1.000000000190015;
    for (int j = 0; j < 6; ++j) { y = y + 1.0; ser = ser + cof[j] / y; }
    return tmp + std::log(stp * ser / x);
}
static int upload_warm_constants(torj_ctx* c) {
    const int ntv = TORJ_WARM_NTV;
    const double tmax = 5.0, dt = 2.0 * tmax / (ntv - 1);
    std::vector<double2> tab(ntv);
    for (int i = 1; i <= ntv; ++i) {
        const double t = -tmax + (i - 1) * dt;
        tab[i - 1] = make_double2(t, std::exp(-(t * t)) * dt);
    }
    CK(c->d_warm_tab.resize(ntv, c->stream));
    CK(cudaMemcpyAsync(c->d_warm_tab, tab.data(), ntv * sizeof(double2), cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));  // tab is a local
    double comb[6][6][6], fal[6], fct[8], igam[8];
    memset(comb, 0, sizeof comb);
    for (int l = 1; l <= 5; ++l) {
        const int lm = l - 1;
        fal[l] = -std::pow(0.25, l) * ref_fact(2 * l) / (ref_fact(l) * ref_fact(l));
        for (int is = 0; is <= l; ++is) {
            const int k = l - is;
            const double asl = ((k % 2) ? -1.0 : 1.0) / (ref_fact(is + l) * ref_fact(l - is));
            const double bsl = asl * (is * is + (double)(2 * k * lm * (l + is)) / (2 * l - 1));
            double* cb = comb[is][l];
            cb[0] = (double)(is * is) * asl; cb[1] = (double)(is * l) * asl; cb[2] = bsl;
            cb[3] = (double)is * asl; cb[4] = (double)l * asl; cb[5] = asl;
        }
    }
    fal[0] = 0.0;
    for (int m = 0; m < 8; ++m) { fct[m] = ref_fact(m); igam[m] = 1.0 / std::exp(ref_gammln(m + 1.5)); }
    CK(cudaMemcpyToSymbol(cw_comb, comb, sizeof comb));
    double combs[7][4][6];
    memset(combs, 0, sizeof combs);
    for (int nq = -3; nq <= 3; ++nq)
        for (int l = 1; l <= 3; ++l) {
            const int is = nq < 0 ? -nq : nq;
            if (is > l) continue;
            for (int q = 0; q < 6; ++q) combs[nq + 3][l][q] = comb[is][l][q] * ((nq < 0 && (q == 1 || q == 3)) ? -1.0 : 1.0);
        }
    CK(cudaMemcpyToSymbol(cw_combs, combs, sizeof combs));
    CK(cudaMemcpyToSymbol(cw_fal, fal, sizeof fal));
    CK(cudaMemcpyToSymbol(cw_fact, fct, sizeof fct));
    CK(cudaMemcpyToSymbol(cw_igam, igam, sizeof igam));
    return 0;
}

int torj_ctx_create(int device, void* cuda_stream, torj_ctx** out) {
    if (!out) FAIL("torj_ctx_create: out is NULL");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_err = std::string("torj_ctx_create: no CUDA device (") + cudaGetErrorString(e) + "); libtorj_cuda has no CPU path";
        return 1;
    }
    if (device < 0 || device >= ndev) FAIL("torj_ctx_create: bad device index");
    CK(cudaSetDevice(device));
    torj_ctx* c = new torj_ctx();
    Guard<torj_ctx, torj_ctx_destroy> guard(c);
    c->device = device;
    if (cuda_stream) {
        c->stream = (cudaStream_t)cuda_stream;
    } else {
        CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        c->own_stream = true;
    }
    CK(cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, device));
    CK(cudaEventCreate(&c->ev0));
    CK(cudaEventCreate(&c->ev1));
    Tableau t[2];
    fill_tableaux(t);
    // cudaMemcpyToSymbol, not the stream: every context writes the same constants, so a running kernel never sees a change
    CK(cudaMemcpyToSymbol(c_tab, t, sizeof t));
    // Bessel series coefficients c[n][k] = (-1)^k n!/(k!(n+k)!)
    double bc[5][TORJ_BESS_K];
    for (int n = 0; n < 5; ++n) {
        bc[n][0] = 1.0;
        for (int k = 1; k < TORJ_BESS_K; ++k) bc[n][k] = -bc[n][k - 1] / ((double)k * (double)(n + k));
    }
    CK(cudaMemcpyToSymbol(c_bess, bc, sizeof bc));
    double bd[5][TORJ_BESS_K];
    for (int n = 0; n < 5; ++n)
        for (int k = 0; k < TORJ_BESS_K; ++k) bd[n][k] = (double)(n + 2 * k) * bc[n][k];
    CK(cudaMemcpyToSymbol(c_bessd, bd, sizeof bd));
    if (int rc = upload_warm_constants(c)) return rc;
    {
        std::lock_guard<std::mutex> lk(g_gl.mu);
        if ((int)g_gl.tab.size() > device && !g_gl.tab[device].empty()) c->gl_set = true;  // inherited (see GLRegistry)
    }
    *out = guard.release();
    return 0;
}

void torj_ctx_destroy(torj_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->ws) torj_bundle_destroy(c->ws);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    delete c;
}

int torj_ctx_sync(torj_ctx* c) {
    if (set_device(c)) return 1;
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int64_t torj_ctx_launch_count(const torj_ctx* c) { return c->launches; }

int torj_ctx_set_exact_sum(torj_ctx* c, int32_t on) {
    if (!c) FAIL("torj_ctx_set_exact_sum: ctx is NULL");
    if (on != 0 && on != 1) FAIL("torj_ctx_set_exact_sum: on must be 0 (floating-point atomics) or 1 (exact sum)");
    c->exact_sum = on;
    return 0;
}

int torj_ctx_last_trace_ms(torj_ctx* c, double* ms) {
    if (!c->ev_valid) FAIL("torj_ctx_last_trace_ms: no trace launched yet");
    if (set_device(c)) return 1;
    CK(cudaEventSynchronize(c->ev1));
    float t = 0.f;
    CK(cudaEventElapsedTime(&t, c->ev0, c->ev1));
    *ms = (double)t;
    return 0;
}

int torj_abs_init(torj_ctx* c, int32_t n, const double* nodes, const double* weights) {
    if (n < 1 || n > TORJ_MAX_GL) FAIL("torj_abs_init: need 1 <= n <= 64");
    if (!nodes || !weights) FAIL("torj_abs_init: NULL nodes / weights");
    if (set_device(c)) return 1;
    // the rule must be symmetric, t[k] = -t[n-1-k], w[k] = w[n-1-k] — every Gauss-Legendre rule is (gausslegendre(N), reference
    // src/absorption.jl:4): the kernel evaluates the Bessel functions of a node pair once
    for (int k = 0; k < n; ++k)
        if (std::fabs(nodes[k] + nodes[n - 1 - k]) > 1e-13 || std::fabs(weights[k] - weights[n - 1 - k]) > 1e-13)
            FAIL("torj_abs_init: nodes / weights are not a symmetric rule (expected FastGaussQuadrature.gausslegendre(N))");
    std::vector<double> want(nodes, nodes + n);
    want.insert(want.end(), weights, weights + n);
    std::lock_guard<std::mutex> lk(g_gl.mu);
    if ((int)g_gl.tab.size() <= c->device) g_gl.tab.resize(c->device + 1);
    if (g_gl.tab[c->device] == want) {  // the device already holds exactly this table
        c->gl_set = true;
        return 0;
    }
    GLNodes g;
    memset(&g, 0, sizeof g);
    g.n = n;
    for (int i = 0; i < n; ++i) {
        g.t[i] = nodes[i];
        g.sq[i] = std::sqrt(1.0 - nodes[i] * nodes[i]);
        g.wp[i] = (2 * i == n - 1) ? 0.5 * weights[i] : weights[i];
    }
    CK(cudaDeviceSynchronize());  // no kernel of ANY context on this device may be reading the old table
    CK(cudaMemcpyToSymbol(c_gl, &g, sizeof g));  // not a stream copy: the whole device is idle (above)
    g_gl.tab[c->device] = want;
    c->gl_set = true;
    return 0;
}

// ---- B-spline prefilter (host): rows (1/6, 2/3, 1/6), natural ends c0-2c1+c2 = 0 -> c[1]=y[0], c[n]=y[n-1]
static void prefilter_line(const double* y, size_t ys, int n, double* c, size_t cs) {
    std::vector<double> sol(n), cp(n), dp(n);
    sol[0] = y[0];
    sol[n - 1] = y[(size_t)(n - 1) * ys];
    if (n > 2) {
        const double a = 1.0 / 6.0, b = 2.0 / 3.0;
        int m = n - 2;
        cp[0] = a / b;
        dp[0] = (y[ys] - a * sol[0]) / b;
        for (int k = 1; k < m; ++k) {
            double r = y[(size_t)(k + 1) * ys];
            if (k == m - 1) r -= a * sol[n - 1];
            double den = b - a * cp[k - 1];
            cp[k] = a / den;
            dp[k] = (r - a * dp[k - 1]) / den;
        }
        if (m == 1) dp[0] = (y[ys] - a * sol[0] - a * sol[n - 1]) / b;
        sol[m] = dp[m - 1];
        for (int k = m - 2; k >= 0; --k) sol[k + 1] = dp[k] - cp[k] * sol[k + 2];
    }
    for (int k = 0; k < n; ++k) c[(size_t)(k + 1) * cs] = sol[k];
    c[0] = 2.0 * sol[0] - sol[1];
    c[(size_t)(n + 1) * cs] = 2.0 * sol[n - 1] - sol[n - 2];
}

int torj_bspline_prefilter_1d(int32_t n, const double* data, double* coef) {
    if (n < 2) FAIL("torj_bspline_prefilter_1d: n < 2");
    prefilter_line(data, 1, n, coef, 1);
    return 0;
}

int torj_bspline_prefilter_2d(int32_t nR, int32_t nZ, const double* data, double* coef) {
    if (nR < 2 || nZ < 2) FAIL("torj_bspline_prefilter_2d: need at least 2 points per axis");
    size_t sr = (size_t)nR + 2;
    std::vector<double> tmp(sr * nZ);
    for (int j = 0; j < nZ; ++j) prefilter_line(data + (size_t)j * nR, 1, nR, tmp.data() + (size_t)j * sr, 1);
    for (size_t i = 0; i < sr; ++i) prefilter_line(tmp.data() + i, sr, nZ, coef + i, sr);
    return 0;
}

// The DevTables of a plasma whose node data are in p->dA, on grid g, and their copy p->dT
static int plasma_tables(torj_plasma* p, const torj_grid* g, double psi_prof_max) {
    cudaStream_t st = p->ctx->stream;
    DevTables& T = p->T;
    T.A = p->dA;
    T.nR = g->nR; T.nZ = g->nZ; T.row = g->nR + 2;
    T.r0 = g->R_first; T.z0 = g->Z_first;
    double hr = (g->R_last - g->R_first) / (double)(g->nR - 1), hz = (g->Z_last - g->Z_first) / (double)(g->nZ - 1);
    T.inv_hr = 1.0 / hr; T.inv_hz = 1.0 / hz;
    T.rlast = g->R_first + hr * (g->nR - 1); T.zlast = g->Z_first + hz * (g->nZ - 1);
    T.psi_prof_max = psi_prof_max;
    CK(p->dT.resize(1, st));
    CK(cudaMemcpyAsync(p->dT, &T, sizeof(DevTables), cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));  // a plasma set hands dT to the kernels of any context on the device
    return 0;
}

int torj_plasma_create(torj_ctx* c, const torj_grid* g, const double* coef_psi, const double* coef_lnne,
                       const double* coef_lnTe, const double* coef_BR, const double* coef_BZ, const double* coef_Bphi,
                       const double* vol_coef, int32_t n_vol, double vol_psi0, double vol_dpsi, double psi_prof_max,
                       torj_plasma** out) {
    if (!c || !g || !out) FAIL("torj_plasma_create: NULL argument");
    if (g->nR < 2 || g->nZ < 2 || n_vol < 2) FAIL("torj_plasma_create: grid too small");
    if ((double)(g->nR + 2) * (double)(g->nZ + 2) >= 2147483648.0) FAIL("torj_plasma_create: grid too large (2^31 nodes)");
    if (set_device(c)) return 1;
    torj_plasma* p = new torj_plasma();
    Guard<torj_plasma, torj_plasma_destroy> guard(p);
    p->ctx = c;
    p->id = ++g_plasma_serial;
    size_t nodes = (size_t)(g->nR + 2) * (g->nZ + 2);
    std::vector<double2> hA(3 * nodes);
    for (size_t k = 0; k < nodes; ++k) {
        hA[3 * k] = make_double2(coef_BR[k], coef_BZ[k]);
        hA[3 * k + 1] = make_double2(coef_Bphi[k], coef_lnne[k]);
        hA[3 * k + 2] = make_double2(coef_lnTe[k], coef_psi[k]);
    }
    CK(p->dA.resize(3 * nodes, c->stream));
    CK(cudaMemcpyAsync(p->dA, hA.data(), 3 * nodes * sizeof(double2), cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (int rc = plasma_tables(p, g, psi_prof_max)) return rc;
    p->vol_c.assign(vol_coef, vol_coef + n_vol + 2);
    p->n_vol = n_vol; p->vol_x0 = vol_psi0; p->vol_h = vol_dpsi;
    *out = guard.release();
    return 0;
}

// natural cubic spline through (x, y), x strictly increasing, resampled on the uniform range x[0]..x[n-1] with n
// points: IMAS.interp1d(x, y, :cubic).(range(x[1], x[end], length(x))) of reference src/plasma.jl:17-18,42-43
static void resample_uniform(const double* x, const double* y, int n, std::vector<double>& xr, std::vector<double>& yr) {
    std::vector<double> m2(n, 0.0);  // second derivatives, natural ends
    if (n > 2) {
        std::vector<double> cp(n), dp(n);
        for (int i = 1; i < n - 1; ++i) {
            double h0 = x[i] - x[i - 1], h1 = x[i + 1] - x[i];
            double diag = 2.0 * (h0 + h1), rhs = 6.0 * ((y[i + 1] - y[i]) / h1 - (y[i] - y[i - 1]) / h0);
            if (i == 1) { cp[i] = h1 / diag; dp[i] = rhs / diag; }
            else { double den = diag - h0 * cp[i - 1]; cp[i] = h1 / den; dp[i] = (rhs - h0 * dp[i - 1]) / den; }
        }
        m2[n - 2] = dp[n - 2];
        for (int i = n - 3; i >= 1; --i) m2[i] = dp[i] - cp[i] * m2[i + 1];
    }
    xr.resize(n); yr.resize(n);
    int seg = 0;
    for (int q = 0; q < n; ++q) {
        double t = (q == n - 1) ? x[n - 1] : x[0] + (x[n - 1] - x[0]) * (double)q / (double)(n - 1);
        xr[q] = t;
        while (seg < n - 2 && t >= x[seg + 1]) ++seg;
        double h = x[seg + 1] - x[seg], A = (x[seg + 1] - t) / h, B = (t - x[seg]) / h;
        yr[q] = A * y[seg] + B * y[seg + 1] + ((A * A * A - A) * m2[seg] + (B * B * B - B) * m2[seg + 1]) * h * h / 6.0;
    }
}

static std::vector<double> thomas_pivots(int n) {  // cp[k] of the (1/6, 2/3, 1/6) system with n-2 unknowns
    std::vector<double> cp(std::max(n, 2));
    const double a = 1.0 / 6.0, b = 2.0 / 3.0;
    cp[0] = a / b;
    for (int k = 1; k < n; ++k) cp[k] = a / (b - a * cp[k - 1]);
    return cp;
}

int torj_plasma_create_from_data(torj_ctx* c, const torj_grid* g, const double* psi_norm, const double* psi_prof,
                                 const double* ne_prof, const double* Te_prof, int32_t n_prof, const double* BR,
                                 const double* BZ, const double* Bphi, const double* psi_1d, const double* vol_1d,
                                 int32_t n_1d, torj_plasma** out) {
    if (!c || !g || !out) FAIL("torj_plasma_create_from_data: NULL argument");
    if (g->nR < 2 || g->nZ < 2 || n_prof < 4 || n_1d < 2) FAIL("torj_plasma_create_from_data: grid or profile too small");
    if ((double)(g->nR + 2) * (double)(g->nZ + 2) >= 2147483648.0) FAIL("torj_plasma_create_from_data: grid too large (2^31 nodes)");
    for (int i = 1; i < n_prof; ++i) if (!(psi_prof[i] > psi_prof[i - 1])) FAIL("torj_plasma_create_from_data: psi_prof must increase");
    if (set_device(c)) return 1;
    cudaStream_t st = c->stream;
    const int nR = g->nR, nZ = g->nZ, sr = nR + 2;
    const size_t npts = (size_t)nR * nZ, nodes = (size_t)sr * (nZ + 2);
    // ---- 1-D host work (tiny): resample, log, prefilter (src/plasma.jl:16-19,42-44)
    std::vector<double> xr, yr, c1[2];
    double x0[2], hh[2];
    const double* profs[2] = {ne_prof, Te_prof};
    for (int q = 0; q < 2; ++q) {
        resample_uniform(psi_prof, profs[q], n_prof, xr, yr);
        for (auto& v : yr) v = std::log(v);
        c1[q].resize(n_prof + 2);
        prefilter_line(yr.data(), 1, n_prof, c1[q].data(), 1);
        x0[q] = xr[0]; hh[q] = (xr[n_prof - 1] - xr[0]) / (double)(n_prof - 1);
    }
    std::vector<double> vr, vv, vc(n_1d + 2);
    resample_uniform(psi_1d, vol_1d, n_1d, vr, vv);
    prefilter_line(vv.data(), 1, n_1d, vc.data(), 1);
    double psi_prof_max = psi_prof[0];
    for (int i = 1; i < n_prof; ++i) psi_prof_max = std::max(psi_prof_max, psi_prof[i]);
    // ---- device: node data of six fields, R pass, Z pass, pack
    dev_array<double> o_raw, o_tmp, o_coef, o_c1, o_cpR, o_cpZ;
    CK(o_raw.resize(6 * npts, st));
    CK(o_tmp.resize((size_t)sr * nZ, st));
    CK(o_coef.resize(6 * nodes, st));
    CK(o_c1.resize(2 * (size_t)(n_prof + 2), st));
    std::vector<double> cpR = thomas_pivots(nR), cpZ = thomas_pivots(nZ);
    CK(o_cpR.resize(cpR.size(), st));
    CK(o_cpZ.resize(cpZ.size(), st));
    double *d_raw = o_raw, *d_tmp = o_tmp, *d_coef = o_coef, *d_c1 = o_c1, *d_cpR = o_cpR,
           *d_cpZ = o_cpZ;
    const double* src[6] = {psi_norm, nullptr, nullptr, BR, BZ, Bphi};  // field order: psi, lnne, lnTe, BR, BZ, Bphi
    for (int f = 0; f < 6; ++f)
        if (src[f]) CK(cudaMemcpyAsync(d_raw + f * npts, src[f], npts * sizeof(double), cudaMemcpyHostToDevice, st));
    for (int q = 0; q < 2; ++q)
        CK(cudaMemcpyAsync(d_c1 + q * (n_prof + 2), c1[q].data(), (n_prof + 2) * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_cpR, cpR.data(), cpR.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_cpZ, cpZ.data(), cpZ.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    for (int q = 0; q < 2; ++q) {
        k_profile_to_grid<<<(unsigned)((npts + 255) / 256), 256, 0, st>>>(d_raw, (long long)npts, d_c1 + q * (n_prof + 2), n_prof,
                                                                       x0[q], hh[q], d_raw + (1 + q) * npts);
        c->launches++;
    }
    for (int f = 0; f < 6; ++f) {
        // R pass: nZ lines of nR points (contiguous) -> tmp[(nR+2) x nZ]; Z pass: nR+2 columns of nZ points -> coef
        k_prefilter_lines<<<(nZ + 127) / 128, 128, 0, st>>>(d_raw + f * npts, d_tmp, nR, nZ, nR, 1, sr, 1, d_cpR);
        k_prefilter_lines<<<(sr + 127) / 128, 128, 0, st>>>(d_tmp, d_coef + f * nodes, nZ, sr, 1, sr, 1, sr, d_cpZ);
        c->launches += 2;
    }
    CK(cudaGetLastError());
    torj_plasma* p = new torj_plasma();
    Guard<torj_plasma, torj_plasma_destroy> guard(p);
    p->ctx = c;
    p->id = ++g_plasma_serial;
    CK(p->dA.resize(3 * nodes, st));
    k_pack_tables<<<(unsigned)((nodes + 255) / 256), 256, 0, st>>>(d_coef, d_coef + nodes, d_coef + 2 * nodes, d_coef + 3 * nodes,
                                                                 d_coef + 4 * nodes, d_coef + 5 * nodes, (long long)nodes, p->dA);
    c->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    if (int rc = plasma_tables(p, g, psi_prof_max)) return rc;
    p->vol_c = vc;
    p->n_vol = n_1d; p->vol_x0 = vr[0]; p->vol_h = (vr[n_1d - 1] - vr[0]) / (double)(n_1d - 1);
    *out = guard.release();
    return 0;
}

void torj_plasma_destroy(torj_plasma* p) {
    if (!p) return;
    cudaSetDevice(p->ctx->device);
    delete p;
}

// V(psi_N): 1-D cubic B-spline with Line extrapolation (reference src/plasma.jl:44,109,113)
static double volume_at(const torj_plasma* p, double x) {
    const int n = p->n_vol;
    double xl = p->vol_x0 + p->vol_h * (n - 1);
    double xc = std::min(std::max(x, p->vol_x0), xl);
    double u = (xc - p->vol_x0) / p->vol_h + 1.0;
    int i = (int)std::floor(u);
    i = std::min(std::max(i, 1), n - 1);
    double d = u - i, e = 1.0 - d;
    double w[4] = {e * e * e / 6.0, 2.0 / 3.0 - d * d + d * d * d / 2.0, 2.0 / 3.0 - e * e + e * e * e / 2.0, d * d * d / 6.0};
    double dw[4] = {-e * e / 2.0 / p->vol_h, (-2.0 * d + 1.5 * d * d) / p->vol_h, (2.0 * e - 1.5 * e * e) / p->vol_h,
                    d * d / 2.0 / p->vol_h};
    double v = 0, dv = 0;
    for (int k = 0; k < 4; ++k) { v += w[k] * p->vol_c[i - 1 + k]; dv += dw[k] * p->vol_c[i - 1 + k]; }
    if (xc != x) v += (x - xc) * dv;
    return v;
}

typedef void (*trace_kernel_t)(TraceArgs);
extern "C++" {  // (inside the extern "C" block)
template <bool SET, bool XS>
static trace_kernel_t pick_trace_kernel_set(int scheme, bool high, int model, int lpr) {
    const bool z3 = scheme == 1;
    if (model == 1) return lpr == 32 ? (z3 ? k_trace<1, false, 1, 32, SET, XS> : k_trace<0, false, 1, 32, SET, XS>)
                                     : (z3 ? k_trace<1, false, 1, 1, SET, XS> : k_trace<0, false, 1, 1, SET, XS>);
    if (lpr == 32) return high ? (z3 ? k_trace<1, true, 0, 32, SET, XS> : k_trace<0, true, 0, 32, SET, XS>) : (z3 ? k_trace<1, false, 0, 32, SET, XS> : k_trace<0, false, 0, 32, SET, XS>);
    if (lpr == 8) return high ? (z3 ? k_trace<1, true, 0, 8, SET, XS> : k_trace<0, true, 0, 8, SET, XS>) : (z3 ? k_trace<1, false, 0, 8, SET, XS> : k_trace<0, false, 0, 8, SET, XS>);
    if (lpr == 4) return high ? (z3 ? k_trace<1, true, 0, 4, SET, XS> : k_trace<0, true, 0, 4, SET, XS>) : (z3 ? k_trace<1, false, 0, 4, SET, XS> : k_trace<0, false, 0, 4, SET, XS>);
    if (lpr == 2) return high ? (z3 ? k_trace<1, true, 0, 2, SET, XS> : k_trace<0, true, 0, 2, SET, XS>) : (z3 ? k_trace<1, false, 0, 2, SET, XS> : k_trace<0, false, 0, 2, SET, XS>);
    return high ? (z3 ? k_trace<1, true, 0, 1, SET, XS> : k_trace<0, true, 0, 1, SET, XS>) : (z3 ? k_trace<1, false, 0, 1, SET, XS> : k_trace<0, false, 0, 1, SET, XS>);
}
}
// set: the plasma-set instantiations (torj_bundle_trace_plasmas with more than one plasma)
// xs: the exact-sum instantiations (a template parameter: a never-taken out-of-line call in the float kernels measured 0.7 %
// on the bench beam and on the warm model at one lane per ray, profiles/README.md)
static trace_kernel_t pick_trace_kernel(int scheme, bool high, int model, int lpr, bool set, bool xs) {
    if (xs) return set ? pick_trace_kernel_set<true, true>(scheme, high, model, lpr) : pick_trace_kernel_set<false, true>(scheme, high, model, lpr);
    return set ? pick_trace_kernel_set<true, false>(scheme, high, model, lpr) : pick_trace_kernel_set<false, false>(scheme, high, model, lpr);
}

static SolverOpts to_sopts(const torj_options* o, double s_max) {
    torj_options d;
    torj_options_default(&d);
    if (o) d = *o;
    SolverOpts s;
    s.n_segments = d.n_segments; s.max_steps = d.max_steps_per_segment; s.s_max = s_max; s.dtmax = d.dtmax;
    s.abstol = d.abstol; s.reltol = d.reltol; s.psi_stop = d.psi_stop; s.p_stop = d.p_stop; s.te_min = d.te_min;
    s.max_harmonic = d.max_harmonic;
    s.alpha_floor = d.alpha_floor;
    return s;
}

int torj_probe(torj_ctx* c, const torj_plasma* p, const torj_options* opt, int64_t n, const double* x, const double* N,
               double freq_hz, int32_t mode, double* out) {
    if (!c->gl_set) FAIL("The weights and abscissae for the absorption were never initialized. Call `abs_Al_init` before using the absorption.");
    if (set_device(c)) return 1;
    SolverOpts so = to_sopts(opt, 1.0);
    dev_array<double> o_x, o_N, o_out;
    CK(o_x.resize(3 * (size_t)n, c->stream));
    CK(o_N.resize(3 * (size_t)n, c->stream));
    CK(o_out.resize(11 * (size_t)n, c->stream));
    double *dx = o_x, *dN = o_N, *dout = o_out;
    CK(cudaMemcpyAsync(dx, x, 3 * n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(dN, N, 3 * n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    const int model = opt ? opt->absorption_model : 0;
    if (model != 0 && model != 1) FAIL("torj_probe: absorption_model must be 0 (Albajar) or 1 (warm)");
    k_probe<<<(unsigned)((n + 127) / 128), 128, TORJ_WARM_H * 128 * sizeof(double), c->stream>>>(
        p->T, n, dx, dN, freq_hz, mode, so.te_min, so.max_harmonic, so.alpha_floor, model, c->d_warm_tab, dout);
    c->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, dout, 11 * n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int torj_rhs(torj_ctx* c, const torj_plasma* p, const torj_options* opt, int64_t n, const double* u, double freq_hz,
             int32_t mode, double* du) {
    if (!c->gl_set) FAIL("The weights and abscissae for the absorption were never initialized. Call `abs_Al_init` before using the absorption.");
    if (set_device(c)) return 1;
    SolverOpts so = to_sopts(opt, 1.0);
    dev_array<double> o_u, o_du;
    CK(o_u.resize(7 * (size_t)n, c->stream));
    CK(o_du.resize(7 * (size_t)n, c->stream));
    double *d_u = o_u, *d_du = o_du;
    CK(cudaMemcpyAsync(d_u, u, 7 * n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    const int model = opt ? opt->absorption_model : 0;
    if (model != 0 && model != 1) FAIL("torj_rhs: absorption_model must be 0 (Albajar) or 1 (warm)");
    k_rhs<<<(unsigned)((n + 127) / 128), 128, TORJ_WARM_H * 128 * sizeof(double), c->stream>>>(
        p->T, n, d_u, freq_hz, mode, so.te_min, so.max_harmonic, so.alpha_floor, model, c->d_warm_tab, d_du);
    c->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(du, d_du, 7 * n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int torj_warm_alpha(torj_ctx* c, int64_t n, const double* omega, const double* X, const double* Y, const double* N_r,
                    const double* theta, const double* te, const double* v_g_perp, int32_t imod, double* N_warm,
                    double* alpha, int32_t* lrm, int32_t* ierr) {
    if (!c || n < 1 || !omega || !X || !Y || !N_r || !theta || !te || !v_g_perp) FAIL("torj_warm_alpha: bad argument");
    if (set_device(c)) return 1;
    std::vector<double> in(7 * (size_t)n), out(5 * (size_t)n);
    const double* src[7] = {omega, X, Y, N_r, theta, te, v_g_perp};
    for (int q = 0; q < 7; ++q) memcpy(in.data() + q * n, src[q], n * sizeof(double));
    dev_array<double> o_in, o_out;
    CK(o_in.resize(in.size(), c->stream));
    CK(o_out.resize(out.size(), c->stream));
    CK(cudaMemcpyAsync(o_in, in.data(), in.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    k_warm_alpha<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(n, o_in, imod, c->d_warm_tab, o_out);
    c->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out.data(), o_out, out.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    for (int64_t i = 0; i < n; ++i) {
        if (N_warm) N_warm[i] = out[i];
        if (alpha) alpha[i] = out[n + i];
        if (lrm) lrm[i] = (int32_t)out[2 * n + i];
        if (ierr) ierr[i] = (int32_t)out[3 * n + i];
    }
    return 0;
}

// ---- bundle ---------------------------------------------------------------------------------------------------
static int bundle_upload(torj_bundle* b, const double* pos, const double* dir, const double* weight,
                         const double* freq_hz, const int32_t* mode) {
    torj_ctx* c = b->ctx;
    const int64_t n = b->n;
    size_t nf = b->per_ray_fm ? (size_t)n : 1;
    CK(cudaMemcpyAsync(b->d_pos, pos, 3 * n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(b->d_dir, dir, 3 * n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(b->d_w, weight, n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    b->w_max = 0.0;
    for (int64_t i = 0; i < n; ++i) b->w_max = std::isnan(weight[i]) ? INFINITY : std::max(b->w_max, std::fabs(weight[i]));
    CK(cudaMemcpyAsync(b->d_freq, freq_hz, nf * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(b->d_mode, mode, nf * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));  // host buffers may be released by the caller on return
    return 0;
}

// A new bundle of n rays on c (the current device): its per-ray device arrays and the BundleDev that points at them
static int bundle_new(torj_ctx* c, int64_t n, int32_t per_ray_fm, torj_bundle** out) {
    torj_bundle* b = new torj_bundle();
    Guard<torj_bundle, torj_bundle_destroy> guard(b);
    b->ctx = c; b->n = n; b->per_ray_fm = per_ray_fm;
    const size_t nr = (size_t)n, nf = per_ray_fm ? nr : 1;
    cudaStream_t st = c->stream;
    CK(b->d_pos.resize(3 * nr, st));
    CK(b->d_dir.resize(3 * nr, st));
    CK(b->d_w.resize(nr, st));
    CK(b->d_freq.resize(nf, st));
    CK(b->d_mode.resize(nf, st));
    CK(b->d_u0.resize(7 * nr, st));
    CK(b->d_s0.resize(nr, st));
    CK(b->d_psil.resize(nr, st));
    CK(b->d_Pf.resize(nr, st));
    CK(b->d_Pdep.resize(nr, st));
    CK(b->d_status.resize(nr, st));
    CK(b->d_npts.resize(nr, st));
    CK(b->d_queue.resize(1, st));
    CK(b->d_counters.resize(8, st));
    CK(b->d_ufinal.resize(7 * nr, st));
    BundleDev& B = b->B;
    B.n_rays = n; B.pos = b->d_pos; B.dir = b->d_dir; B.weight = b->d_w; B.freq = b->d_freq; B.mode = b->d_mode;
    B.per_ray_fm = per_ray_fm; B.u0 = b->d_u0; B.s0 = b->d_s0; B.psi_launch = b->d_psil; B.status = b->d_status;
    B.P_final = b->d_Pf; B.P_dep = b->d_Pdep; B.n_points = b->d_npts;
    *out = guard.release();
    return 0;
}

int torj_bundle_create(torj_ctx* c, int64_t n, const double* pos, const double* dir, const double* weight,
                       const double* freq_hz, const int32_t* mode, int32_t per_ray_fm, torj_bundle** out) {
    if (!c || !out || n < 1) FAIL("torj_bundle_create: bad argument");
    if (set_device(c)) return 1;
    torj_bundle* b = nullptr;
    if (int rc = bundle_new(c, n, per_ray_fm, &b)) return rc;
    Guard<torj_bundle, torj_bundle_destroy> guard(b);
    if (bundle_upload(b, pos, dir, weight, freq_hz, mode)) return 1;
    *out = guard.release();
    return 0;
}

// Bundle generated on the device from launcher parameters: launch_peripheral_rays (reference src/launch.jl:24-132) for
// n_launchers beams at once; ray k of launcher L is ray L*n_per+k, its beam index is L, frequency and mode are per ray.
// gh_nodes/gh_weights: Gauss-Hermite rule of order 2*N_rings+2 (FastGaussQuadrature.gausshermite, src/launch.jl:72).
int torj_bundle_create_from_launchers(torj_ctx* c, int32_t n_launchers, const double* x0, const double* N0, const double* w,
                                      const double* inv_Rc, const double* f, const int32_t* mode, int32_t N_rings,
                                      int32_t min_azimuthal_points, int32_t normalize_weight_sum, const double* gh_nodes,
                                      const double* gh_weights, torj_bundle** out, int64_t* n_rays_out) {
    if (!c || !out || n_launchers < 1) FAIL("torj_bundle_create_from_launchers: bad argument");
    if (N_rings < 2) FAIL("N_rings < 2 which is the minimum");  // ArgumentError of src/launch.jl:27-29
    if (set_device(c)) return 1;
    // ring radii in units of w/sqrt(2): v[N_rings+2:end] of the ascending rule, first N_rings used (src/launch.jl:72-83)
    std::vector<double> ru(N_rings), rwu(N_rings);
    std::vector<int> start(N_rings + 1, 0);
    double wsum = 0.0;
    for (int i = 0; i < N_rings; ++i) {
        ru[i] = gh_nodes[N_rings + 1 + i];
        rwu[i] = gh_weights[N_rings + 1 + i];
        long nth = std::max(1L, (long)std::nearbyint((double)min_azimuthal_points * ru[i] / ru[0]));
        start[i + 1] = start[i] + (int)nth;
    }
    // sum of the launcher's weights, accumulated ray by ray in launch order like `sum(ray_weights)` does
    for (int i = 0; i < N_rings; ++i) {
        int nth = start[i + 1] - start[i];
        double wt = ru[i] * rwu[i] * (2.0 * M_PI / (double)nth);
        for (int j = 0; j < nth; ++j) wsum += wt;
    }
    const int n_per = start[N_rings];
    const int64_t n = (int64_t)n_launchers * n_per;
    // an empty bundle shell with device arrays, then the generator kernel fills pos/dir/weight/freq/mode/beam
    torj_bundle* b = nullptr;
    if (int rc = bundle_new(c, n, 1, &b)) return rc;
    Guard<torj_bundle, torj_bundle_destroy> guard(b);
    b->w_max = -1.0;  // weights of order 1 made on the device; an exact booking out of range is refused there
    cudaStream_t st = c->stream;
    CK(b->d_beam.resize(n, st));
    b->n_beams = n_launchers;
    // launcher parameters to the device
    const size_t nl = n_launchers;
    dev_array<double> o_par; dev_array<int> o_ipar;
    CK(o_par.resize(9 * nl + 2 * N_rings, st));
    CK(o_ipar.resize(nl + N_rings + 1, st));
    double* d_par = o_par; int* d_ipar = o_ipar;
    CK(cudaMemcpyAsync(d_par, x0, 3 * nl * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_par + 3 * nl, N0, 3 * nl * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_par + 6 * nl, w, nl * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_par + 7 * nl, inv_Rc, nl * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_par + 8 * nl, f, nl * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_par + 9 * nl, ru.data(), N_rings * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_par + 9 * nl + N_rings, rwu.data(), N_rings * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_ipar, mode, nl * sizeof(int), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_ipar + nl, start.data(), (N_rings + 1) * sizeof(int), cudaMemcpyHostToDevice, st));
    LaunchArgs A;
    A.n_launchers = n_launchers; A.n_rings = N_rings; A.n_per = n_per;
    A.x0 = d_par; A.N0 = d_par + 3 * nl; A.w = d_par + 6 * nl; A.inv_Rc = d_par + 7 * nl; A.f = d_par + 8 * nl;
    A.r_unit = d_par + 9 * nl; A.rw_unit = d_par + 9 * nl + N_rings;
    A.mode = d_ipar; A.ring_start = d_ipar + nl;
    A.wsum_unit = wsum; A.normalize = normalize_weight_sum;
    A.pos = b->d_pos; A.dir = b->d_dir; A.weight = b->d_w; A.freq = b->d_freq; A.mode_out = b->d_mode; A.beam = b->d_beam;
    k_launch_rays<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(A);
    c->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    *out = guard.release();
    if (n_rays_out) *n_rays_out = n;
    return 0;
}

// copy the generated (or uploaded) launch arrays back: pos/dir [3][n], weight [n] (any pointer may be NULL)
int torj_bundle_rays(torj_bundle* b, double* pos, double* dir, double* weight) {
    torj_ctx* c = b->ctx;
    if (set_device(c)) return 1;
    if (pos) CK(cudaMemcpyAsync(pos, b->d_pos, 3 * b->n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if (dir) CK(cudaMemcpyAsync(dir, b->d_dir, 3 * b->n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if (weight) CK(cudaMemcpyAsync(weight, b->d_w, b->n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

void torj_bundle_destroy(torj_bundle* b) {
    if (!b) return;
    cudaSetDevice(b->ctx->device);
    cudaStreamSynchronize(b->ctx->stream);
    delete b;
}

int torj_bundle_set_window(torj_bundle* b, int64_t first, int64_t count, int32_t max_pts) {
    if (count > 0 && max_pts > 0 && (first < 0 || first + count > b->n)) FAIL("torj_bundle_set_window: window outside the bundle");
    if (set_device(b->ctx)) return 1;
    cudaStream_t st = b->ctx->stream;
    b->traj_first = 0; b->traj_count = 0; b->traj_max = 0;  // a failing allocation below leaves an EMPTY window, not a dangling one
    const size_t m = (count > 0 && max_pts > 0) ? (size_t)count * max_pts : 0;
    CK(b->d_ts.resize(m, st));
    CK(b->d_txyz.resize(3 * m, st));
    CK(b->d_tP.resize(m, st));
    CK(b->d_tdP.resize(m, st));
    CK(b->d_tprof.resize(0, st));  // until a trace sizes it for its n_psi
    if (m == 0) return 0;
    b->traj_first = first; b->traj_count = count; b->traj_max = max_pts;
    return 0;
}

int torj_bundle_set_beams(torj_bundle* b, int32_t n_beams, const int32_t* beam_id) {
    torj_ctx* c = b->ctx;
    if (n_beams < 1) FAIL("torj_bundle_set_beams: n_beams < 1");
    if (set_device(c)) return 1;
    CK(cudaStreamSynchronize(c->stream));
    if (n_beams == 1 || !beam_id) {
        b->n_beams = 1;
        return 0;
    }
    for (int64_t i = 0; i < b->n; ++i)
        if (beam_id[i] < 0 || beam_id[i] >= n_beams) FAIL("torj_bundle_set_beams: beam_id out of range");
    CK(b->d_beam.resize(b->n, c->stream));  // allocated on first use
    CK(cudaMemcpyAsync(b->d_beam, beam_id, b->n * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));  // beam_id belongs to the caller
    b->n_beams = n_beams;
    return 0;
}

}  // extern "C"

// The refusals of a plasma set (torj_bundle_trace_plasmas / torj_trace_plasmas); n_beams: the bundle's beams
static int check_plasma_set(const char* fn, const torj_ctx* c, int32_t n_pl, const torj_plasma* const* pls,
                            const int32_t* beam_plasma, int n_beams) {
    char msg[256];
    if (n_pl < 1) { snprintf(msg, sizeof msg, "%s: n_plasmas must be >= 1", fn); FAIL(msg); }
    if (!pls) { snprintf(msg, sizeof msg, "%s: plasmas is NULL", fn); FAIL(msg); }
    for (int k = 0; k < n_pl; ++k) {
        if (!pls[k]) { snprintf(msg, sizeof msg, "%s: plasmas[%d] is NULL", fn, k); FAIL(msg); }
        if (pls[k]->ctx->device != c->device) {
            snprintf(msg, sizeof msg, "%s: plasmas[%d] is on device %d, the bundle's context on device %d", fn, k,
                     pls[k]->ctx->device, c->device);
            FAIL(msg);
        }
        const DevTables &T0 = pls[0]->T, &T = pls[k]->T;
        if (T.nR != T0.nR || T.nZ != T0.nZ || T.row != T0.row || memcmp(&T.r0, &T0.r0, sizeof(double)) ||
            memcmp(&T.z0, &T0.z0, sizeof(double)) || memcmp(&T.inv_hr, &T0.inv_hr, sizeof(double)) ||
            memcmp(&T.inv_hz, &T0.inv_hz, sizeof(double)) || memcmp(&T.rlast, &T0.rlast, sizeof(double)) ||
            memcmp(&T.zlast, &T0.zlast, sizeof(double))) {
            snprintf(msg, sizeof msg, "%s: plasmas[%d] is on another (R,Z) grid than plasmas[0]; a set shares one grid", fn, k);
            FAIL(msg);
        }
    }
    if (n_pl == 1) return 0;
    if (n_beams < 2) {
        snprintf(msg, sizeof msg, "%s: %d plasmas need beams (torj_bundle_set_beams): a profile row belongs to one plasma", fn, n_pl);
        FAIL(msg);
    }
    if (!beam_plasma) { snprintf(msg, sizeof msg, "%s: beam_plasma is NULL", fn); FAIL(msg); }
    for (int q = 0; q < n_beams; ++q)
        if (beam_plasma[q] < 0 || beam_plasma[q] >= n_pl) {
            snprintf(msg, sizeof msg, "%s: beam_plasma[%d] = %d is outside [0, %d)", fn, q, beam_plasma[q], n_pl);
            FAIL(msg);
        }
    return 0;
}

static int finalize(torj_bundle* b);

// torj_bundle_trace (one plasma) and torj_bundle_trace_plasmas: beam q through pls[beam_plasma[q]] when n_pl > 1
static int bundle_trace(torj_bundle* b, int32_t n_pl, const torj_plasma* const* pls, const int32_t* beam_plasma,
                        const torj_options* opt, double s_max, int32_t n_psi, const double* psi_edges) {
    torj_ctx* c = b->ctx;
    const torj_plasma* p = pls[0];  // the set's grid; its tables alone with one plasma
    const bool set = n_pl > 1;
    if (!c->gl_set) FAIL("The weights and abscissae for the absorption were never initialized. Call `abs_Al_init` before using the absorption.");
    if (n_psi < 2) FAIL("torj_bundle_trace: need at least 2 psi levels");
    for (int j = 1; j < n_psi; ++j) if (!(psi_edges[j] > psi_edges[j - 1])) FAIL("torj_bundle_trace: psi_dP_dV must be strictly increasing");
    torj_options od;
    torj_options_default(&od);
    if (opt) od = *opt;
    if (od.scheme != 0 && od.scheme != 1) FAIL("torj_bundle_trace: scheme must be 0 (Tsit5) or 1 (OwrenZen3)");
    if (od.n_segments < 1) FAIL("torj_bundle_trace: n_segments must be >= 1");
    if (!(od.alpha_floor >= 0.0)) FAIL("torj_bundle_trace: alpha_floor must be >= 0");
    if (od.max_harmonic < 1 || od.max_harmonic > 16) FAIL("torj_bundle_trace: max_harmonic must be in 1..16 (1 = no absorption)");
    if (!(od.dtmax > 0.0) || !(od.abstol > 0.0) || !(od.reltol > 0.0)) FAIL("torj_bundle_trace: dtmax, abstol and reltol must be > 0");
    if (od.schedule < 0 || od.schedule > 3)
        FAIL("torj_bundle_trace: schedule must be 0 (automatic), 1 (whole rays), 2 (segment hand-off) or 3 (hand-off without tail stages)");
    if ((od.schedule == 2 || od.schedule == 3) && od.n_segments > TORJ_SEG_MAX)
        FAIL("torj_bundle_trace: the segment hand-off (schedule 2 or 3) takes n_segments <= 16000; schedules 0 and 1 trace whole rays above that");
    if (od.max_steps_per_segment < 1) FAIL("torj_bundle_trace: max_steps_per_segment < 1");
    if (od.absorption_model != 0 && od.absorption_model != 1) FAIL("torj_bundle_trace: absorption_model must be 0 (Albajar) or 1 (warm)");
    if (od.lanes_per_ray != 0 && od.lanes_per_ray != 1 && od.lanes_per_ray != 2 && od.lanes_per_ray != 4 && od.lanes_per_ray != 8 &&
        od.lanes_per_ray != 32)
        FAIL("torj_bundle_trace: lanes_per_ray must be 0 (automatic), 1, 2, 4, 8 or 32");
    if (od.absorption_model == 1 && od.lanes_per_ray > 1 && od.lanes_per_ray < 32)
        FAIL("torj_bundle_trace: the warm model runs with 1 or 32 lanes per ray");
    if (od.absorption_model == 1 && od.max_harmonic > 3) FAIL("torj_bundle_trace: max_harmonic > 3 belongs to the Albajar model; the warm model takes its harmonics from larmornumber");
    if (!(s_max > 0.0)) FAIL("torj_bundle_trace: s_max must be > 0");
    const bool xs = c->exact_sum != 0;
    if (xs && b->w_max > TORJ_XS_WMAX)
        FAIL("torj_bundle_trace: exact sum mode takes ray weights of magnitude <= 2^40 (and no NaN)");
    if (set_device(c)) return 1;
    cudaStream_t st = c->stream;
    if (b->n_psi != n_psi || b->prof_rows != b->n_beams) {
        b->n_psi = 0; b->prof_rows = 0;  // a failing allocation below leaves the bundle untraced
        b->h_edges.clear();
        CK(b->d_edges.resize(n_psi, st));
        CK(b->d_bins.resize((size_t)b->n_beams * (n_psi + 2), st));
        CK(b->d_dV.resize((size_t)b->n_beams * n_psi, st));  // one row, or one per beam for a plasma set
        CK(b->d_profile.resize((size_t)b->n_beams * (n_psi + 2), st));
        b->n_psi = n_psi;
        b->prof_rows = b->n_beams;
    }
    if (b->traj_count > 0) CK(b->d_tprof.resize((size_t)b->traj_count * n_psi, st));
    const int dV_rows = set ? b->n_beams : 1;
    std::vector<uint64_t> row_plasma(dV_rows);
    for (int q = 0; q < dV_rows; ++q) row_plasma[q] = pls[set ? beam_plasma[q] : 0]->id;
    if (b->dV_plasmas != row_plasma || (int)b->h_edges.size() != n_psi ||
        memcmp(b->h_edges.data(), psi_edges, n_psi * sizeof(double)) != 0) {
        std::vector<double> dV((size_t)dV_rows * n_psi, 1.0);
        for (int q = 0; q < dV_rows; ++q) {
            const torj_plasma* pq = pls[set ? beam_plasma[q] : 0];
            for (int j = 0; j + 1 < n_psi; ++j) dV[(size_t)q * n_psi + j] = volume_at(pq, psi_edges[j + 1]) - volume_at(pq, psi_edges[j]);
        }
        CK(cudaMemcpyAsync(b->d_edges, psi_edges, n_psi * sizeof(double), cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(b->d_dV, dV.data(), dV.size() * sizeof(double), cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));  // dV is a local; psi_edges belongs to the caller
        b->h_edges.assign(psi_edges, psi_edges + n_psi);
        b->dV_plasmas = row_plasma;
    }
    b->dV_rows = dV_rows;
    PlasmaSetDev P{nullptr, nullptr, nullptr, nullptr};
    if (set) {
        std::vector<const void*> hs(2 * (size_t)n_pl);
        for (int k = 0; k < n_pl; ++k) { hs[k] = pls[k]->dA; hs[n_pl + k] = pls[k]->dT; }
        std::vector<int> hb(beam_plasma, beam_plasma + b->n_beams);
        if (hs != b->h_set || hb != b->h_beam_plasma) {
            CK(cudaStreamSynchronize(st));  // an earlier trace may still read them
            b->h_set.clear(); b->h_beam_plasma.clear();  // until the copies below have completed
            CK(b->d_set.resize(hs.size(), st));
            CK(b->d_beam_plasma.resize(hb.size(), st));
            CK(cudaMemcpyAsync(b->d_set, hs.data(), hs.size() * sizeof(void*), cudaMemcpyHostToDevice, st));
            CK(cudaMemcpyAsync(b->d_beam_plasma, hb.data(), hb.size() * sizeof(int), cudaMemcpyHostToDevice, st));
            CK(cudaStreamSynchronize(st));  // hs and hb are locals
            b->h_set = hs; b->h_beam_plasma = hb;
        }
        const void** d_set = b->d_set;
        P.A = reinterpret_cast<const double2* const*>(d_set);
        P.T = reinterpret_cast<const DevTables* const*>(d_set + n_pl);
        P.beam_plasma = b->d_beam_plasma; P.beam_id = b->d_beam;
    }
    CK(cudaMemsetAsync(b->d_bins, 0, (size_t)b->n_beams * (n_psi + 2) * sizeof(double), st));
    const size_t xs_words = torj_xs_buffer_words((size_t)b->n_beams * (n_psi + 2));
    b->xs_last = false;
    if (xs) {
        CK(b->d_xs.resize(xs_words, st));
        CK(cudaMemsetAsync(b->d_xs, 0, xs_words * sizeof(long long), st));
    }
    CK(cudaMemsetAsync(b->d_queue, 0, sizeof(unsigned long long), st));
    CK(cudaMemsetAsync(b->d_counters, 0, 8 * sizeof(unsigned long long), st));
    if (b->traj_count > 0) CK(cudaMemsetAsync(b->d_tprof, 0, (size_t)b->traj_count * n_psi * sizeof(double), st));

    SolverOpts so = to_sopts(&od, s_max);
    k_ray_init<<<(unsigned)((b->n + 127) / 128), 128, 0, st>>>(p->T, b->B, so, P);
    c->launches++;
    CK(cudaGetLastError());

    TraceArgs a;
    a.T = p->T; a.B = b->B; a.O = so; a.P = P;
    a.J.first = b->traj_first; a.J.count = b->traj_count; a.J.max_pts = b->traj_max;
    a.J.s = b->d_ts; a.J.xyz = b->d_txyz; a.J.P = b->d_tP; a.J.dP = b->d_tdP; a.J.prof = b->d_tprof;
    a.n_psi = n_psi; a.n_beams = b->n_beams; a.beam_id = b->d_beam; a.psi_edges = b->d_edges; a.bins = b->d_bins; a.next_ray = b->d_queue; a.counters = b->d_counters;
    a.warm_tab = c->d_warm_tab; a.u_final = b->d_ufinal;
    a.xs = xs ? b->d_xs + TORJ_XS_STAT : nullptr;
    const int model = od.absorption_model;
    // Several lanes per ray when the bundle cannot fill the GPU with one thread per ray — then the time is one ray's
    // latency, and splitting the quadrature nodes over the lanes of a group shortens exactly that. Measured
    // (profiles/r02_lanes_per_ray.json), ms for 1 / 2 / 4 / 8 lanes: cold 4 keV beam of 1 025 rays 54.9 / 53.2 / 51.9 / 52.1;
    // 10 keV scans of 1 025 rays 215 / 183 / 151 / 150, 4 100 rays 293 / 241 / 211 / 231, 8 200 rays 290 / 248 / 242 / 303,
    // 16 400 rays 316 / 304 / 332 / 620 (32 lanes fit only 1 184 rays at a time: 4 100 rays 576). Hence: the widest group
    // that still fits all rays at once, 8 lanes only while that leaves every scheduler a single warp. The warm model, whose
    // alpha is ~100x the rest of the RHS and warp-cooperative either way, takes a warp per ray up to half the lanes.
    const int64_t lanes_guess = (int64_t)c->num_sms * TORJ_MINB * TORJ_TPB;
    int lpr = od.lanes_per_ray;
    if (lpr == 0) {
        if (model == 1) lpr = (b->n <= lanes_guess / 2) ? 32 : 1;
        else lpr = (b->n * 8 <= lanes_guess / 2) ? 8 : (b->n * 4 <= lanes_guess) ? 4 : (b->n * 2 <= lanes_guess) ? 2 : 1;
    }
    // k_trace's dynamic shared memory: stage derivatives, parked scalars and, for the warm model at one lane per ray, its stash
    size_t smem = (size_t)(TORJ_K_WORDS + TORJ_PARK_SLOTS * TORJ_TPB) * sizeof(double);
    if (model == 1 && lpr == 1) smem += (size_t)TORJ_WARM_H * TORJ_TPB * sizeof(double);
    int bps = 0;
    int64_t warps = (b->n * lpr + 31) / 32;
    int64_t blocks_needed = (warps + (TORJ_TPB / 32) - 1) / (TORJ_TPB / 32);
    // harmonics above the third, the warm model and the warp-per-ray mapping run in their own instantiations, so the
    // default kernels do not carry the code
    void (*kern)(TraceArgs);
    const bool high = od.max_harmonic > 3;
    kern = pick_trace_kernel(od.scheme, high, model, lpr, set, xs);
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, TORJ_TPB, smem));
    if (bps < 1) FAIL("torj_bundle_trace: trace kernel does not fit on an SM");
    int64_t grid = std::min<int64_t>((int64_t)c->num_sms * bps, blocks_needed);  // persistent: resident CTAs only
    // Segment hand-off whenever the bundle exceeds the resident lanes. It removes the partly filled last wave (65 543
    // rays on 37 888 lanes: 1.73 ray-times instead of 2) and keeps the lanes of a warp in step: with whole rays per lane
    // a bundle of rays of very different lengths (the 1 M-ray angle sweep) drifts apart and some lane pays for the full
    // absorption coefficient on every trip (measured 3.1 s -> 2.4 s). Below one wave there is nothing to balance.
    const int64_t lanes = (int64_t)c->num_sms * bps * TORJ_TPB / lpr;  // rays in flight
    int interleave = od.schedule == 2 || od.schedule == 3 || (od.schedule == 0 && b->n > lanes);
    if (od.n_segments < 2 || od.n_segments > TORJ_SEG_MAX || b->n > 0x7fffffff) interleave = 0;  // TORJ_SEG_MAX: the hand-off word's 15-bit fields
    a.interleave = interleave; a.hand = nullptr; a.seg_done = nullptr; a.rays_left = nullptr;
    if (interleave) {
        CK(b->d_hand.resize((size_t)b->n * TORJ_HAND_D, st));
        CK(b->d_segdone.resize((size_t)b->n, st));
        CK(b->d_left.resize(1, st));
        b->h_left = (int)b->n;
        CK(cudaMemsetAsync(b->d_segdone, 0, (size_t)b->n * sizeof(int), st));
        CK(cudaMemcpyAsync(b->d_left, &b->h_left, sizeof(int), cudaMemcpyHostToDevice, st));
        a.hand = b->d_hand; a.seg_done = b->d_segdone; a.rays_left = b->d_left;
    }
    a.life = nullptr; a.lmax = nullptr;
    CK(cudaEventRecord(c->ev0, st));
    // Life-ordered rounds (hand-off schedule, Albajar model): breadth-first rounds make all rays advance together, so the
    // few longest-lived rays finish alone while the GPU idles — a fixed ~67 ms on the 1 M-ray sweep whatever the number of
    // GPUs (profiles/). A pilot march predicts every ray's life; the rounds are shifted so that all rays END together and
    // the long ones start first, while idle lanes run ahead in the queue and start the short ones early.
    if (interleave && model == 0 && od.schedule != 3) {
        CK(b->d_life.resize((size_t)b->n + 1, st));
        CK(cudaMemsetAsync(b->d_life + b->n, 0, sizeof(int), st));
        k_predict_life<<<(unsigned)((b->n + 127) / 128), 128, 0, st>>>(p->T, b->B, so, P, TORJ_LIFE_HARM_COST, b->d_life,
                                                                      b->d_life + b->n);
        c->launches++;
        CK(cudaGetLastError());
        a.life = b->d_life; a.lmax = b->d_life + b->n;
    }
    kern<<<(unsigned)grid, TORJ_TPB, smem, st>>>(a);
    c->launches++;
    CK(cudaGetLastError());
    CK(cudaEventRecord(c->ev1, st));
    c->ev_valid = true;
    b->xs_last = xs;
    return finalize(b);
}

// bins (or, after an exact-sum trace, the words) -> d_profile, normalised by the dV rows of the last trace
static int finalize(torj_bundle* b) {
    torj_ctx* c = b->ctx;
    const unsigned grid = (unsigned)(((size_t)b->n_beams * (b->n_psi + 2) + 127) / 128);
    if (b->xs_last)
        k_finalize_exact<<<grid, 128, 0, c->stream>>>(b->d_xs + TORJ_XS_STAT, b->d_dV, b->n_psi, b->n_beams, (int)(b->dV_rows > 1), b->d_profile);
    else
        k_finalize<<<grid, 128, 0, c->stream>>>(b->d_bins, b->d_dV, b->n_psi, b->n_beams, (int)(b->dV_rows > 1), b->d_profile);
    c->launches++;
    CK(cudaGetLastError());
    return 0;
}

extern "C" {

int torj_bundle_trace(torj_bundle* b, const torj_plasma* p, const torj_options* opt, double s_max, int32_t n_psi,
                      const double* psi_edges) {
    return bundle_trace(b, 1, &p, nullptr, opt, s_max, n_psi, psi_edges);
}

int torj_bundle_trace_plasmas(torj_bundle* b, int32_t n_plasmas, const torj_plasma* const* plasmas, const int32_t* beam_plasma,
                              const torj_options* opt, double s_max, int32_t n_psi, const double* psi_edges) {
    if (!b) FAIL("torj_bundle_trace_plasmas: bundle is NULL");
    if (int rc = check_plasma_set("torj_bundle_trace_plasmas", b->ctx, n_plasmas, plasmas, beam_plasma, b->n_beams)) return rc;
    return bundle_trace(b, n_plasmas, plasmas, beam_plasma, opt, s_max, n_psi, psi_edges);
}

void* torj_bundle_device_profile(torj_bundle* b) { return b->d_profile; }

}  // extern "C"

// The refusals of the exact-word pair: the words exist only after a trace that booked them
static int check_exact_words(const torj_bundle* b, const char* fn) {
    char msg[256];
    if (!b) { snprintf(msg, sizeof msg, "%s: bundle is NULL", fn); FAIL(msg); }
    if (b->n_psi == 0) { snprintf(msg, sizeof msg, "%s: nothing traced yet", fn); FAIL(msg); }
    if (!b->xs_last) {
        snprintf(msg, sizeof msg, "%s: the last trace did not book exact sums (torj_ctx_set_exact_sum(ctx, 1) before it)", fn);
        FAIL(msg);
    }
    return 0;
}

extern "C" {

int torj_bundle_device_exact_words(torj_bundle* b, void** words, int64_t* n_words) {
    if (int rc = check_exact_words(b, "torj_bundle_device_exact_words")) return rc;
    if (!words || !n_words) FAIL("torj_bundle_device_exact_words: words and n_words must not be NULL");
    *words = static_cast<long long*>(b->d_xs);
    *n_words = (int64_t)b->d_xs.size();
    return 0;
}

int torj_bundle_finalize_exact(torj_bundle* b) {
    if (int rc = check_exact_words(b, "torj_bundle_finalize_exact")) return rc;
    if (set_device(b->ctx)) return 1;
    return finalize(b);
}

int torj_bundle_results(torj_bundle* b, double* dP_dV, double* deposited_power, double* P_final, double* P_dep,
                        int32_t* n_points, int32_t* status, torj_counters* counters) {
    torj_ctx* c = b->ctx;
    if (set_device(c)) return 1;
    cudaStream_t st = c->stream;
    if (b->n_psi == 0) FAIL("torj_bundle_results: nothing traced yet");
    const size_t row = (size_t)b->n_psi + 2;
    std::vector<double> prof(row * b->n_beams);
    CK(cudaMemcpyAsync(prof.data(), b->d_profile, prof.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (P_final) CK(cudaMemcpyAsync(P_final, b->d_Pf, b->n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (P_dep) CK(cudaMemcpyAsync(P_dep, b->d_Pdep, b->n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (n_points) CK(cudaMemcpyAsync(n_points, b->d_npts, b->n * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (status) CK(cudaMemcpyAsync(status, b->d_status, b->n * sizeof(int), cudaMemcpyDeviceToHost, st));
    unsigned long long cn[8];
    CK(cudaMemcpyAsync(cn, b->d_counters, sizeof cn, cudaMemcpyDeviceToHost, st));
    long long xst[TORJ_XS_STAT] = {0, 0};
    if (b->xs_last)
        CK(cudaMemcpyAsync(xst, b->d_xs, sizeof xst, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (!torj_xs_valid(xst[0], xst[1])) {
        char msg[256];
        if (xst[1])
            snprintf(msg, sizeof msg, "torj_bundle_results: exact sum: %lld bookings outside the accumulator's range (|w dP| >= 2^64 "
                     "or NaN); the profile is NaN", xst[1]);
        else
            snprintf(msg, sizeof msg, "torj_bundle_results: exact sum: %lld bookings exceed the accumulator's bound of 2^34; "
                     "the profile is NaN", xst[0]);
        FAIL(msg);
    }
    for (int q = 0; q < b->n_beams; ++q) {
        if (dP_dV) memcpy(dP_dV + (size_t)q * b->n_psi, prof.data() + q * row, b->n_psi * sizeof(double));
        if (deposited_power) deposited_power[q] = prof[q * row + b->n_psi];
    }
    if (counters) {
        counters->n_acc = (int64_t)cn[0]; counters->n_rej = (int64_t)cn[1]; counters->n_rhs = (int64_t)cn[2];
        counters->n_alpha = (int64_t)cn[3]; counters->n_harm = (int64_t)cn[4]; counters->n_rays_ok = (int64_t)cn[5];
        counters->n_harm_pruned = (int64_t)cn[6];
        counters->n_alpha_skipped = (int64_t)cn[7];
    }
    return 0;
}

int torj_bundle_trajectories(torj_bundle* b, double* s, double* xyz, double* P, double* dP_ds, double* dP_dV_ray) {
    torj_ctx* c = b->ctx;
    if (b->traj_count <= 0) FAIL("torj_bundle_trajectories: no trajectory window set");
    if (set_device(c)) return 1;
    cudaStream_t st = c->stream;
    size_t m = (size_t)b->traj_count * b->traj_max;
    if (s) CK(cudaMemcpyAsync(s, b->d_ts, m * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (xyz) CK(cudaMemcpyAsync(xyz, b->d_txyz, 3 * m * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (P) CK(cudaMemcpyAsync(P, b->d_tP, m * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (dP_ds) CK(cudaMemcpyAsync(dP_ds, b->d_tdP, m * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (dP_dV_ray && b->d_tprof)
        CK(cudaMemcpyAsync(dP_dV_ray, b->d_tprof, (size_t)b->traj_count * b->n_psi * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (dP_dV_ray) {  // shell power -> dP/dV per ray (reference src/plasma.jl:141), with the volume of the ray's plasma
        std::vector<double> dV((size_t)b->dV_rows * b->n_psi);
        std::vector<int> beam(b->dV_rows > 1 ? b->traj_count : 0);
        CK(cudaMemcpyAsync(dV.data(), b->d_dV, dV.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (!beam.empty())
            CK(cudaMemcpyAsync(beam.data(), b->d_beam + b->traj_first, beam.size() * sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));  // dV and beam are locals
        for (int64_t r = 0; r < b->traj_count; ++r) {
            double* row = dP_dV_ray + (size_t)r * b->n_psi;
            const double* dVr = dV.data() + (beam.empty() ? 0 : (size_t)beam[r] * b->n_psi);
            for (int j = 0; j + 1 < b->n_psi; ++j) row[j] /= dVr[j];
            row[b->n_psi - 1] = 0.0;
        }
    }
    return 0;
}

int torj_bundle_final_state(torj_bundle* b, double* u_final, double* R, double* phi, double* tau) {
    torj_ctx* c = b->ctx;
    if (b->n_psi == 0) FAIL("torj_bundle_final_state: nothing traced yet");
    if (set_device(c)) return 1;
    const int64_t n = b->n;
    std::vector<double> u(7 * (size_t)n);
    std::vector<int> st(n);
    CK(cudaMemcpyAsync(u.data(), b->d_ufinal, u.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(st.data(), b->d_status, n * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    const double nan = std::nan("");
    for (int64_t i = 0; i < n; ++i) {
        const bool never_traced = st[i] == TORJ_RAY_CUTOFF_AT_ENTRY || st[i] == TORJ_RAY_INIT_FAILED;
        if (never_traced) for (int q = 0; q < 7; ++q) u[(size_t)q * n + i] = nan;
        const double x = u[i], y = u[n + i], P = u[6 * (size_t)n + i];
        if (R) R[i] = std::hypot(x, y);
        if (phi) phi[i] = std::atan2(y, x);
        if (tau) tau[i] = -std::log(P);
    }
    if (u_final) memcpy(u_final, u.data(), u.size() * sizeof(double));
    return 0;
}

int torj_bundle_trajectories_cyl(torj_bundle* b, double* R, double* phi, double* tau) {
    if (b->traj_count <= 0) FAIL("torj_bundle_trajectories_cyl: no trajectory window set");
    const size_t m = (size_t)b->traj_count * b->traj_max;
    std::vector<double> xyz(3 * m), P(m);
    if (int rc = torj_bundle_trajectories(b, nullptr, xyz.data(), P.data(), nullptr, nullptr)) return rc;
    std::vector<int> np(b->n);
    CK(cudaMemcpyAsync(np.data(), b->d_npts, b->n * sizeof(int), cudaMemcpyDeviceToHost, b->ctx->stream));
    CK(cudaStreamSynchronize(b->ctx->stream));  // np is a local
    for (int64_t r = 0; r < b->traj_count; ++r) {
        const int cnt = std::min<int>(std::max(np[b->traj_first + r], 0), b->traj_max);
        const double* x = xyz.data() + (size_t)r * 3 * b->traj_max;
        for (int k = 0; k < b->traj_max; ++k) {
            const size_t o = (size_t)r * b->traj_max + k;
            const bool ok = k < cnt;
            if (R) R[o] = ok ? std::hypot(x[k], x[b->traj_max + k]) : 0.0;
            if (phi) phi[o] = ok ? std::atan2(x[b->traj_max + k], x[k]) : 0.0;
            if (tau) tau[o] = ok ? -std::log(P[o]) : 0.0;
        }
    }
    return 0;
}

}  // extern "C"

static void drop_workspace(torj_ctx* c) {  // a workspace in an unknown state is not kept
    torj_bundle_destroy(c->ws);
    c->ws = nullptr;
}

// The rays and beams of a one-shot call, or of one device's shard of it
struct JobRays {
    int64_t n_rays;
    const double *pos, *dir, *weight, *freq_hz;
    const int32_t* mode;
    int32_t per_ray_fm, n_beams;
    const int32_t* beam_id;
};

// A one-shot call (torj_trace*, torj_multi_trace*): its arguments after the plasma ones, in the C ABI's order
struct HostJob : JobRays {
    const torj_options* opt;  // psi levels, options and s_max
    double s_max;
    int32_t n_psi;
    const double* psi_edges;
    double *dP_dV, *deposited_power, *P_final, *P_dep;  // outputs
    int32_t *n_points, *status;
    int64_t traj_first, traj_count;  // trajectory window
    int32_t traj_max_pts;
    double *traj_s, *traj_xyz, *traj_P, *traj_dP_ds, *traj_dP_dV_ray;
    torj_counters* counters;
    int trace_oneshot(torj_ctx* c, int32_t n_pl, const torj_plasma* const* pls, const int32_t* beam_plasma) const;
    int multi_trace(torj_multi* m, const char* fn, bool set_api, int32_t n_pl, const torj_mplasma* const* mps,
                    const int32_t* beam_plasma);
};
#define TORJ_HOST_JOB                                                                                              \
    HostJob {                                                                                                      \
        {n_rays, pos, dir, weight, freq_hz, mode, per_ray_fm, n_beams, beam_id}, opt, s_max, n_psi, psi_edges, dP_dV, \
            deposited_power, P_final, P_dep, n_points, status, traj_first, traj_count, traj_max_pts, traj_s, traj_xyz,  \
            traj_P, traj_dP_ds, traj_dP_dV_ray, counters                                                           \
    }

// The one-shot calls (torj_trace*, torj_multi_trace*) trace through the context's workspace c->ws with the rays r, the
// trajectory window [traj_first, traj_first + traj_count) and j's psi levels and options. The workspace of the previous
// call is reused when the bundle shape is unchanged (no cudaMalloc/cudaFree on the repeated-call path of make_beam scans).
static int workspace_trace(torj_ctx* c, int32_t n_pl, const torj_plasma* const* pls, const int32_t* beam_plasma,
                           const HostJob& j, const JobRays& r, int64_t traj_first, int64_t traj_count) {
    torj_bundle* b = c->ws;
    if (b && (b->n != r.n_rays || b->per_ray_fm != r.per_ray_fm)) {
        drop_workspace(c);
        b = nullptr;
    }
    int rc = 0;
    if (!b) {
        rc = torj_bundle_create(c, r.n_rays, r.pos, r.dir, r.weight, r.freq_hz, r.mode, r.per_ray_fm, &b);
        if (rc) return rc;
        c->ws = b;
    } else {
        if (set_device(c)) return 1;
        rc = bundle_upload(b, r.pos, r.dir, r.weight, r.freq_hz, r.mode);
        if (rc) return rc;
    }
    if (traj_count != b->traj_count || traj_first != b->traj_first || (traj_count > 0 && j.traj_max_pts != b->traj_max))
        rc = torj_bundle_set_window(b, traj_first, traj_count, j.traj_max_pts);
    if (!rc) rc = torj_bundle_set_beams(b, r.n_beams, r.beam_id);
    if (!rc) rc = bundle_trace(b, n_pl, pls, beam_plasma, j.opt, j.s_max, j.n_psi, j.psi_edges);
    return rc;
}

// torj_trace (one plasma) and torj_trace_plasmas
int HostJob::trace_oneshot(torj_ctx* c, int32_t n_pl, const torj_plasma* const* pls, const int32_t* beam_plasma) const {
    int rc = workspace_trace(c, n_pl, pls, beam_plasma, *this, *this, traj_first, traj_count);
    torj_bundle* b = c->ws;
    if (!rc) rc = torj_bundle_results(b, dP_dV, deposited_power, P_final, P_dep, n_points, status, counters);
    if (!rc && traj_count > 0) rc = torj_bundle_trajectories(b, traj_s, traj_xyz, traj_P, traj_dP_ds, traj_dP_dV_ray);
    if (rc) drop_workspace(c);
    return rc;
}

extern "C" {

int torj_trace(torj_ctx* c, const torj_plasma* p, const torj_options* opt, int64_t n_rays, const double* pos,
               const double* dir, const double* weight, const double* freq_hz, const int32_t* mode, int32_t per_ray_fm,
               double s_max, int32_t n_psi, const double* psi_edges, int32_t n_beams, const int32_t* beam_id, double* dP_dV,
               double* deposited_power, double* P_final, double* P_dep, int32_t* n_points, int32_t* status, int64_t traj_first,
               int64_t traj_count, int32_t traj_max_pts, double* traj_s, double* traj_xyz, double* traj_P, double* traj_dP_ds,
               double* traj_dP_dV_ray, torj_counters* counters) {
    return TORJ_HOST_JOB.trace_oneshot(c, 1, &p, nullptr);
}

int torj_trace_plasmas(torj_ctx* c, int32_t n_plasmas, const torj_plasma* const* plasmas, const int32_t* beam_plasma,
                       const torj_options* opt, int64_t n_rays, const double* pos, const double* dir, const double* weight,
                       const double* freq_hz, const int32_t* mode, int32_t per_ray_fm, double s_max, int32_t n_psi,
                       const double* psi_edges, int32_t n_beams, const int32_t* beam_id, double* dP_dV, double* deposited_power,
                       double* P_final, double* P_dep, int32_t* n_points, int32_t* status, int64_t traj_first, int64_t traj_count,
                       int32_t traj_max_pts, double* traj_s, double* traj_xyz, double* traj_P, double* traj_dP_ds,
                       double* traj_dP_dV_ray, torj_counters* counters) {
    if (!c) FAIL("torj_trace_plasmas: ctx is NULL");
    // refused before the workspace is touched; the bundle's beams are those torj_bundle_set_beams will set
    if (int rc = check_plasma_set("torj_trace_plasmas", c, n_plasmas, plasmas, beam_plasma, (beam_id && n_beams > 1) ? n_beams : 1))
        return rc;
    return TORJ_HOST_JOB.trace_oneshot(c, n_plasmas, plasmas, beam_plasma);
}

// ---- single-process multi-GPU front end (what a Julia make_beam on an 8-GPU box calls) -------------------------
// NCCL is loaded at run time (dlopen of libnccl.so.2: a process that already holds a copy, e.g. PyTorch's, keeps using
// that one) — nccl.h supplies only the types. Without the library the front end still works through the host sum.
}  // extern "C" (C++ helpers of the multi-GPU front end follow)

struct NcclApi {
    void* h = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
static NcclApi& nccl_api() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* nm : names) {
            api.h = dlopen(nm, RTLD_NOW | RTLD_LOCAL);
            if (api.h) break;
        }
        if (!api.h) return;
        api.CommInitAll = (decltype(api.CommInitAll))dlsym(api.h, "ncclCommInitAll");
        api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.h, "ncclCommDestroy");
        api.AllReduce = (decltype(api.AllReduce))dlsym(api.h, "ncclAllReduce");
        api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.h, "ncclGetErrorString");
        api.ok = api.CommInitAll && api.CommDestroy && api.AllReduce && api.GetErrorString;
    });
    return api;
}

// One persistent host thread per device: jobs are closures run in order; run() hands one job to every worker and waits.
struct MultiWorker {
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::function<void()> job;
    bool has_job = false, quit = false, done = true;
    void loop() {
        for (;;) {
            std::function<void()> j;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return has_job || quit; });
                if (quit && !has_job) return;
                j = std::move(job);
                has_job = false;
            }
            j();
            {
                std::lock_guard<std::mutex> lk(mu);
                done = true;
            }
            cv.notify_all();
        }
    }
    void submit(std::function<void()> j) {
        {
            std::lock_guard<std::mutex> lk(mu);
            job = std::move(j);
            has_job = true;
            done = false;
        }
        cv.notify_all();
    }
    void wait() {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return done; });
    }
};

// Pinned host staging of one device's shard, grown on demand and kept between calls
struct MultiStage {
    size_t cap = 0;
    pinned_array<double> pos, dir, w, freq, Pf, Pd;
    pinned_array<int> mode, beam, np, st;
    std::vector<int64_t> gidx;  // global ray index of local ray j
    cudaError_t reserve(size_t n, cudaStream_t s) {
        if (n <= cap) return cudaSuccess;
        cap = 0;
        cudaError_t e;
        if ((e = pos.resize(3 * n, s)) || (e = dir.resize(3 * n, s)) || (e = w.resize(n, s)) || (e = freq.resize(n, s)) ||
            (e = Pf.resize(n, s)) || (e = Pd.resize(n, s)) || (e = mode.resize(n, s)) || (e = beam.resize(n, s)) ||
            (e = np.resize(n, s)) || (e = st.resize(n, s)))
            return e;
        cap = n;
        return cudaSuccess;
    }
};

struct torj_multi {
    std::vector<torj_ctx*> ctx;
    std::vector<std::unique_ptr<MultiWorker>> worker;
    std::vector<std::unique_ptr<MultiStage>> stage;  // freed with its device current
    std::vector<ncclComm_t> comm;  // empty when NCCL is unavailable
    int sharding = 0;              // 0 contiguous, 1 block-cyclic
    int64_t block = 1;
    int reduction = 0;             // 0 NCCL all-reduce (host sum when unavailable), 1 host sum in device order
    int used_nccl = 0;
    template <class F>
    void run(int used, F&& f) {  // f(d) on worker d for d < used, all concurrently
        for (int d = 0; d < used; ++d) worker[d]->submit([&f, d] { f(d); });
        for (int d = 0; d < used; ++d) worker[d]->wait();
    }
};
struct torj_mplasma {
    std::vector<torj_plasma*> p;
};

extern "C" {

int torj_multi_create(int32_t n_devices, torj_multi** out) {
    if (!out) FAIL("torj_multi_create: out is NULL");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_err = std::string("torj_multi_create: no CUDA device (") + cudaGetErrorString(e) + "); libtorj_cuda has no CPU path";
        return 1;
    }
    if (n_devices <= 0 || n_devices > ndev) n_devices = ndev;
    torj_multi* m = new torj_multi();
    Guard<torj_multi, torj_multi_destroy> guard(m);
    for (int d = 0; d < n_devices; ++d) {
        torj_ctx* c = nullptr;
        if (int rc = torj_ctx_create(d, nullptr, &c)) return rc;
        m->ctx.push_back(c);
    }
    for (int d = 0; d < n_devices; ++d) {
        m->stage.emplace_back(new MultiStage());
        m->worker.emplace_back(new MultiWorker());
        MultiWorker* w = m->worker.back().get();
        w->th = std::thread([w] { w->loop(); });
    }
    if (n_devices > 1 && nccl_api().ok) {  // one communicator per device, created once (SURVEY.md §5 / §8(e))
        std::vector<int> devs(n_devices);
        for (int d = 0; d < n_devices; ++d) devs[d] = d;
        m->comm.resize(n_devices);
        ncclResult_t r = nccl_api().CommInitAll(m->comm.data(), n_devices, devs.data());
        if (r != ncclSuccess) m->comm.clear();  // fall back to the host sum; torj_multi_used_nccl reports it
    }
    *out = guard.release();
    return 0;
}

void torj_multi_destroy(torj_multi* m) {
    if (!m) return;
    for (auto& w : m->worker) {
        {
            std::lock_guard<std::mutex> lk(w->mu);
            w->quit = true;
        }
        w->cv.notify_all();
        if (w->th.joinable()) w->th.join();
    }
    for (size_t d = 0; d < m->comm.size(); ++d) nccl_api().CommDestroy(m->comm[d]);
    for (size_t d = 0; d < m->stage.size(); ++d) {
        if (d < m->ctx.size()) cudaSetDevice(m->ctx[d]->device);
        m->stage[d].reset();
    }
    for (auto* c : m->ctx) torj_ctx_destroy(c);
    delete m;
}

int32_t torj_multi_device_count(const torj_multi* m) { return (int32_t)m->ctx.size(); }
int32_t torj_multi_used_nccl(const torj_multi* m) { return m->used_nccl; }

int torj_multi_configure(torj_multi* m, int32_t sharding, int64_t block_rays, int32_t reduction) {
    if (sharding != 0 && sharding != 1) FAIL("torj_multi_configure: sharding must be 0 (contiguous) or 1 (block-cyclic)");
    if (sharding == 1 && block_rays < 1) FAIL("torj_multi_configure: block_rays < 1");
    if (reduction != 0 && reduction != 1) FAIL("torj_multi_configure: reduction must be 0 (NCCL all-reduce) or 1 (host sum)");
    m->sharding = sharding; m->block = std::max<int64_t>(1, block_rays); m->reduction = reduction;
    return 0;
}

int torj_multi_set_exact_sum(torj_multi* m, int32_t on) {
    if (!m) FAIL("torj_multi_set_exact_sum: torj_multi is NULL");
    if (on != 0 && on != 1) FAIL("torj_multi_set_exact_sum: on must be 0 (floating-point atomics) or 1 (exact sum)");
    for (auto* c : m->ctx) c->exact_sum = on;
    return 0;
}

int torj_multi_abs_init(torj_multi* m, int32_t n, const double* nodes, const double* weights) {
    for (auto* c : m->ctx)
        if (int rc = torj_abs_init(c, n, nodes, weights)) return rc;
    return 0;
}

int torj_multi_last_trace_ms(torj_multi* m, int32_t device, double* ms) {
    if (device < 0 || device >= (int)m->ctx.size()) FAIL("torj_multi_last_trace_ms: device outside the torj_multi");
    return torj_ctx_last_trace_ms(m->ctx[device], ms);
}

int torj_multi_plasma_create_from_data(torj_multi* m, const torj_grid* g, const double* psi_norm, const double* psi_prof,
                                       const double* ne_prof, const double* Te_prof, int32_t n_prof, const double* BR,
                                       const double* BZ, const double* Bphi, const double* psi_1d, const double* vol_1d,
                                       int32_t n_1d, torj_mplasma** out) {
    if (!out) FAIL("torj_multi_plasma_create_from_data: out is NULL");
    torj_mplasma* mp = new torj_mplasma();
    for (auto* c : m->ctx) {  // the tables (3.2 MB for 257x257) are replicated on every device
        torj_plasma* p = nullptr;
        int rc = torj_plasma_create_from_data(c, g, psi_norm, psi_prof, ne_prof, Te_prof, n_prof, BR, BZ, Bphi, psi_1d, vol_1d,
                                              n_1d, &p);
        if (rc) { for (auto* q : mp->p) torj_plasma_destroy(q); delete mp; return rc; }
        mp->p.push_back(p);
    }
    *out = mp;
    return 0;
}

void torj_multi_plasma_destroy(torj_mplasma* mp) {
    if (!mp) return;
    for (auto* p : mp->p) torj_plasma_destroy(p);
    delete mp;
}

// The rays of shard d of `used`: contiguous block, or the blocks d, d+used, d+2 used, ... of `block` rays each.
static void shard_indices(int64_t n_rays, int used, int d, int sharding, int64_t block, std::vector<int64_t>& idx) {
    idx.clear();
    if (sharding == 0) {
        const int64_t base = n_rays / used, rem = n_rays % used;
        const int64_t lo = d * base + std::min<int64_t>(d, rem), n = base + (d < rem ? 1 : 0);
        idx.resize(n);
        for (int64_t j = 0; j < n; ++j) idx[j] = lo + j;
    } else {
        const int64_t nb = (n_rays + block - 1) / block;
        for (int64_t bk = d; bk < nb; bk += used)
            for (int64_t g = bk * block; g < std::min(n_rays, (bk + 1) * block); ++g) idx.push_back(g);
    }
}

// torj_multi_trace (one plasma, called "plasma" in the refusals: set_api false) and torj_multi_trace_plasmas.
// Every refusal comes before phase A, so a refused call enqueues nothing and leaves the devices' workspaces as they were.
// Phase A on device d: gather the shard into pinned staging, upload, enqueue ray init + trace + finalize through the set's
// copies on d. Phase B: (NCCL all-reduce of the device profile buffers, in place, one call per device thread;) results to
// the host.
int HostJob::multi_trace(torj_multi* m, const char* fn, bool set_api, int32_t n_pl, const torj_mplasma* const* mps,
                         const int32_t* beam_plasma) {
    const int nd = (int)m->ctx.size();
    char msg[256];
    const bool have = n_pl >= 1 && mps;
    for (int k = 0; have && k < n_pl; ++k) {  // every device holds its own copy of a plasma, made by this torj_multi
        const torj_mplasma* mp = mps[k];
        if (!mp) continue;  // check_plasma_set names it
        char who[32] = "plasma";
        if (set_api) snprintf(who, sizeof who, "plasmas[%d]", k);
        if ((int)mp->p.size() != nd) { snprintf(msg, sizeof msg, "%s: %s was created on a different device set", fn, who); FAIL(msg); }
        for (int d = 0; d < nd; ++d)
            if (mp->p[d]->ctx != m->ctx[d]) {
                snprintf(msg, sizeof msg, "%s: %s belongs to another torj_multi (its copy on device %d has another context)", fn,
                         who, d);
                FAIL(msg);
            }
    }
    if (n_beams < 1 || !beam_id) n_beams = 1;
    std::vector<std::vector<const torj_plasma*>> sets(nd, std::vector<const torj_plasma*>(have ? n_pl : 0, nullptr));
    for (int d = 0; d < nd; ++d) {
        for (int k = 0; have && k < n_pl; ++k) sets[d][k] = mps[k] ? mps[k]->p[d] : nullptr;
        if (int rc = check_plasma_set(fn, m->ctx[d], n_pl, have ? sets[d].data() : nullptr, beam_plasma, n_beams)) return rc;
    }
    if (n_rays < 1) { snprintf(msg, sizeof msg, "%s: n_rays < 1", fn); FAIL(msg); }
    if (traj_count < 0 || (traj_count > 0 && (traj_first < 0 || traj_first + traj_count > n_rays))) {
        snprintf(msg, sizeof msg, "%s: trajectory window outside the bundle", fn);
        FAIL(msg);
    }
    int used = (int)std::min<int64_t>(nd, n_rays);
    if (m->sharding == 1) used = (int)std::min<int64_t>(used, (n_rays + m->block - 1) / m->block);
    std::vector<int> rcs(used, 0);
    std::vector<std::string> errs(used);
    std::vector<torj_counters> cnts(used);
    std::vector<int64_t> wlo(used, 0), wcnt(used, 0);  // local trajectory window of each shard
    const size_t prow = (size_t)n_psi + 2;
    const bool want_nccl = m->reduction == 0 && used == nd && (int)m->comm.size() == nd && nd > 1;
    std::vector<std::vector<double>> prof(used);

    // ---- phase A
    m->run(used, [&](int d) {
        torj_ctx* c = m->ctx[d];
        MultiStage& S = *m->stage[d];
        auto fail = [&](int rc) { rcs[d] = rc; errs[d] = g_err; };  // g_err is thread-local
        if (set_device(c)) return fail(1);
        shard_indices(n_rays, used, d, m->sharding, m->block, S.gidx);
        const int64_t n = (int64_t)S.gidx.size();
        if (cudaError_t e = S.reserve((size_t)n, c->stream)) { g_err = std::string("pinned staging: ") + cudaGetErrorString(e); return fail(1); }
        for (int64_t j = 0; j < n; ++j) {
            const int64_t g = S.gidx[j];
            for (int q = 0; q < 3; ++q) { S.pos[q * n + j] = pos[q * n_rays + g]; S.dir[q * n + j] = dir[q * n_rays + g]; }
            S.w[j] = weight[g];
            if (per_ray_fm) { S.freq[j] = freq_hz[g]; S.mode[j] = mode[g]; }
            if (n_beams > 1) S.beam[j] = beam_id[g];
        }
        if (!per_ray_fm) { S.freq[0] = freq_hz[0]; S.mode[0] = mode[0]; }
        // local trajectory window: the local rays whose global index falls into [traj_first, traj_first + traj_count)
        int64_t lo = n, cntw = 0;
        if (traj_count > 0)
            for (int64_t j = 0; j < n; ++j)
                if (S.gidx[j] >= traj_first && S.gidx[j] < traj_first + traj_count) { lo = std::min(lo, j); ++cntw; }
        wlo[d] = cntw ? lo : 0; wcnt[d] = cntw;  // contiguous in local order for both shardings
        if (int rc = workspace_trace(c, n_pl, sets[d].data(), beam_plasma, *this,
                                     {n, S.pos, S.dir, S.w, S.freq, S.mode, per_ray_fm, n_beams, S.beam}, wlo[d], wcnt[d]))
            fail(rc);
    });
    bool all_ok = true;
    for (int d = 0; d < used; ++d) all_ok = all_ok && rcs[d] == 0;

    // Exact sum: the devices' words are summed as integers (status words included), before any conversion, so the profile
    // is that of one device tracing the whole bundle. Without NCCL on the host; device 0 then converts the sum.
    const bool xs = m->ctx[0]->exact_sum != 0;
    const bool do_nccl = all_ok && want_nccl;
    if (all_ok && xs && !do_nccl && used > 1) {
        const size_t nw = m->ctx[0]->ws->d_xs.size();
        std::vector<std::vector<unsigned long long>> hw(used, std::vector<unsigned long long>(nw));
        m->run(used, [&](int d) {
            torj_ctx* c = m->ctx[d];
            auto fail = [&](int rc) { rcs[d] = rc; errs[d] = g_err; };
            if (set_device(c)) return fail(1);
            cudaError_t e = cudaMemcpyAsync(hw[d].data(), c->ws->d_xs, nw * sizeof(long long), cudaMemcpyDeviceToHost, c->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
            if (e != cudaSuccess) { g_err = std::string("exact sum: ") + cudaGetErrorString(e); return fail(1); }
        });
        for (int d = 0; d < used; ++d) all_ok = all_ok && rcs[d] == 0;
        if (all_ok) {
            for (int d = 1; d < used; ++d)
                for (size_t k = 0; k < nw; ++k) hw[0][k] += hw[d][k];  // two's complement: a signed sum, in any order
            torj_ctx* c0 = m->ctx[0];
            torj_bundle* b0 = c0->ws;
            int rc = set_device(c0);
            if (!rc) {
                cudaError_t e = cudaMemcpyAsync(b0->d_xs, hw[0].data(), nw * sizeof(long long), cudaMemcpyHostToDevice, c0->stream);
                if (e == cudaSuccess) e = cudaStreamSynchronize(c0->stream);
                if (e != cudaSuccess) { g_err = std::string("exact sum: ") + cudaGetErrorString(e); rc = 1; }
            }
            if (!rc) rc = finalize(b0);
            if (rc) { rcs[0] = rc; errs[0] = g_err; all_ok = false; }
        }
    }

    // ---- phase B (the collective only when every device got through phase A: a missing rank would hang the others)
    const bool one = do_nccl || xs;  // every device's (or device 0's) profile is the whole bundle's
    if (all_ok) m->run(used, [&](int d) {
        torj_ctx* c = m->ctx[d];
        torj_bundle* b = c->ws;
        MultiStage& S = *m->stage[d];
        auto fail = [&](int rc) { rcs[d] = rc; errs[d] = g_err; };
        if (set_device(c)) return fail(1);
        const int64_t n = b->n;
        if (do_nccl && xs) {
            ncclResult_t r = nccl_api().AllReduce(b->d_xs, b->d_xs, b->d_xs.size(), ncclInt64, ncclSum, m->comm[d], c->stream);
            if (r != ncclSuccess) { g_err = std::string("ncclAllReduce: ") + nccl_api().GetErrorString(r); return fail(3); }
            if (int rc = finalize(b)) return fail(rc);
        } else if (do_nccl) {
            ncclResult_t r = nccl_api().AllReduce(b->d_profile, b->d_profile, (size_t)n_beams * prow, ncclDouble, ncclSum,
                                                  m->comm[d], c->stream);
            if (r != ncclSuccess) { g_err = std::string("ncclAllReduce: ") + nccl_api().GetErrorString(r); return fail(3); }
        }
        memset(&cnts[d], 0, sizeof(torj_counters));
        prof[d].assign((size_t)n_beams * prow, 0.0);
        std::vector<double> pr((size_t)n_beams * n_psi), dp(n_beams);
        int rc = torj_bundle_results(b, (!one || d == 0) ? pr.data() : nullptr, (!one || d == 0) ? dp.data() : nullptr,
                                     P_final ? static_cast<double*>(S.Pf) : nullptr, P_dep ? static_cast<double*>(S.Pd) : nullptr,
                                     n_points ? static_cast<int*>(S.np) : nullptr, status ? static_cast<int*>(S.st) : nullptr,
                                     &cnts[d]);
        if (rc) return fail(rc);
        for (int q = 0; q < n_beams; ++q) {
            memcpy(prof[d].data() + q * prow, pr.data() + (size_t)q * n_psi, n_psi * sizeof(double));
            prof[d][q * prow + n_psi] = dp[q];
        }
        for (int64_t j = 0; j < n; ++j) {
            const int64_t g = S.gidx[j];
            if (P_final) P_final[g] = S.Pf[j];
            if (P_dep) P_dep[g] = S.Pd[j];
            if (n_points) n_points[g] = S.np[j];
            if (status) status[g] = S.st[j];
        }
        if (wcnt[d] > 0) {
            const size_t M = (size_t)traj_max_pts, wc = (size_t)wcnt[d];
            std::vector<double> ts(traj_s ? wc * M : 0), tx(traj_xyz ? 3 * wc * M : 0), tp(traj_P ? wc * M : 0),
                td(traj_dP_ds ? wc * M : 0), tv(traj_dP_dV_ray ? wc * n_psi : 0);
            rc = torj_bundle_trajectories(b, traj_s ? ts.data() : nullptr, traj_xyz ? tx.data() : nullptr,
                                          traj_P ? tp.data() : nullptr, traj_dP_ds ? td.data() : nullptr,
                                          traj_dP_dV_ray ? tv.data() : nullptr);
            if (rc) return fail(rc);
            for (size_t k = 0; k < wc; ++k) {
                const size_t o = (size_t)(S.gidx[wlo[d] + k] - traj_first);
                if (traj_s) memcpy(traj_s + o * M, ts.data() + k * M, M * sizeof(double));
                if (traj_xyz) memcpy(traj_xyz + o * 3 * M, tx.data() + k * 3 * M, 3 * M * sizeof(double));
                if (traj_P) memcpy(traj_P + o * M, tp.data() + k * M, M * sizeof(double));
                if (traj_dP_ds) memcpy(traj_dP_ds + o * M, td.data() + k * M, M * sizeof(double));
                if (traj_dP_dV_ray) memcpy(traj_dP_dV_ray + o * n_psi, tv.data() + k * n_psi, n_psi * sizeof(double));
            }
        }
    });
    for (int d = 0; d < used; ++d)
        if (rcs[d]) {
            for (int q = 0; q < used; ++q) drop_workspace(m->ctx[q]);
            g_err = "device " + std::to_string(d) + ": " + errs[d];
            return rcs[d];
        }
    m->used_nccl = do_nccl ? 1 : 0;
    for (int q = 0; q < n_beams; ++q) {
        for (int j = 0; j < n_psi + 1; ++j) {
            double sum = 0.0;
            if (one) sum = prof[0][q * prow + j];  // device 0 holds the whole bundle's profile
            else for (int d = 0; d < used; ++d) sum += prof[d][q * prow + j];  // device order (each device's own sums are not ordered)
            if (j < n_psi) { if (dP_dV) dP_dV[(size_t)q * n_psi + j] = sum; }
            else if (deposited_power) deposited_power[q] = sum;
        }
    }
    if (counters) {
        memset(counters, 0, sizeof(torj_counters));
        for (int d = 0; d < used; ++d) {
            counters->n_acc += cnts[d].n_acc; counters->n_rej += cnts[d].n_rej; counters->n_rhs += cnts[d].n_rhs;
            counters->n_alpha += cnts[d].n_alpha; counters->n_harm += cnts[d].n_harm; counters->n_rays_ok += cnts[d].n_rays_ok;
            counters->n_harm_pruned += cnts[d].n_harm_pruned; counters->n_alpha_skipped += cnts[d].n_alpha_skipped;
        }
    }
    return 0;
}

int torj_multi_trace(torj_multi* m, const torj_mplasma* mp, const torj_options* opt, int64_t n_rays, const double* pos,
                     const double* dir, const double* weight, const double* freq_hz, const int32_t* mode, int32_t per_ray_fm,
                     double s_max, int32_t n_psi, const double* psi_edges, int32_t n_beams, const int32_t* beam_id,
                     double* dP_dV, double* deposited_power, double* P_final, double* P_dep, int32_t* n_points,
                     int32_t* status, int64_t traj_first, int64_t traj_count, int32_t traj_max_pts, double* traj_s,
                     double* traj_xyz, double* traj_P, double* traj_dP_ds, double* traj_dP_dV_ray, torj_counters* counters) {
    return TORJ_HOST_JOB.multi_trace(m, "torj_multi_trace", false, 1, &mp, nullptr);
}

int torj_multi_trace_plasmas(torj_multi* m, int32_t n_plasmas, const torj_mplasma* const* plasmas, const int32_t* beam_plasma,
                             const torj_options* opt, int64_t n_rays, const double* pos, const double* dir, const double* weight,
                             const double* freq_hz, const int32_t* mode, int32_t per_ray_fm, double s_max, int32_t n_psi,
                             const double* psi_edges, int32_t n_beams, const int32_t* beam_id, double* dP_dV,
                             double* deposited_power, double* P_final, double* P_dep, int32_t* n_points, int32_t* status,
                             int64_t traj_first, int64_t traj_count, int32_t traj_max_pts, double* traj_s, double* traj_xyz,
                             double* traj_P, double* traj_dP_ds, double* traj_dP_dV_ray, torj_counters* counters) {
    return TORJ_HOST_JOB.multi_trace(m, "torj_multi_trace_plasmas", true, n_plasmas, plasmas, beam_plasma);
}

int torj_fp64_peak(torj_ctx* c, int32_t iters, double* tflops, double* ms) {
    if (set_device(c)) return 1;
    dev_array<double> o_d;
    CK(o_d.resize(1, c->stream));
    double* d = o_d;
    struct Ev {
        cudaEvent_t e = nullptr;
        ~Ev() { if (e) cudaEventDestroy(e); }
    } ev0, ev1;
    CK(cudaEventCreate(&ev0.e));
    CK(cudaEventCreate(&ev1.e));
    cudaEvent_t e0 = ev0.e, e1 = ev1.e;
    int blocks = c->num_sms * 8, threads = 256;
    k_dfma<<<blocks, threads, 0, c->stream>>>(iters / 8 + 1, d);  // warm-up
    c->launches++;
    CK(cudaEventRecord(e0, c->stream));
    k_dfma<<<blocks, threads, 0, c->stream>>>(iters, d);
    c->launches++;
    CK(cudaEventRecord(e1, c->stream));
    CK(cudaEventSynchronize(e1));
    float t = 0;
    CK(cudaEventElapsedTime(&t, e0, e1));
    double flops = 2.0 * 64.0 * (double)iters * (double)blocks * (double)threads;
    if (ms) *ms = t;
    if (tflops) *tflops = flops / (t * 1e-3) / 1e12;
    return 0;
}

// cycles per dependent DFMA (single warp, single chain)
int torj_fp64_latency(torj_ctx* c, int32_t iters, double* cycles_per_dfma) {
    if (set_device(c)) return 1;
    dev_array<double> o_d; dev_array<long long> o_dc;
    CK(o_d.resize(1, c->stream));
    CK(o_dc.resize(1, c->stream));
    double* d = o_d; long long* dc = o_dc;
    k_dfma_latency<<<1, 32, 0, c->stream>>>(iters, 1.0, d, dc);
    c->launches++;
    long long cyc = 0;
    CK(cudaMemcpyAsync(&cyc, dc, sizeof cyc, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    *cycles_per_dfma = (double)cyc / (16.0 * (double)iters);
    return 0;
}

// rcp_fast / rsqrt_fast / sqrt_fast / exp_fast of the device code on host arrays: out[4][n]
int torj_math_probe(torj_ctx* c, int64_t n, const double* x, double* out) {
    if (!c || n < 1 || !x || !out) FAIL("torj_math_probe: bad argument");
    if (set_device(c)) return 1;
    dev_array<double> o_x, o_out;
    CK(o_x.resize((size_t)n, c->stream));
    CK(o_out.resize(4 * (size_t)n, c->stream));
    double *dx = o_x, *dout = o_out;
    CK(cudaMemcpyAsync(dx, x, n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    k_math_probe<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(n, dx, dout);
    c->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, dout, 4 * n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

}  // extern "C"
