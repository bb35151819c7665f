// Kernels of libtorj_cuda.so (sm_100a).
//   k_ray_init : first_point + vacuum_plasma_refraction, one thread per ray   (reference src/solve.jl:18-74,137-144)
//   k_trace    : persistent one-thread-per-ray integrator with warp-ballot retire-and-refill of finished rays,
//                streaming psi-shell deposition into the profile row           (reference src/solve.jl:154-177, src/plasma.jl:91-151)
//   k_finalize : bins / dV -> dP_dV                                            (reference src/plasma.jl:141, src/solve.jl:233-240)
//   k_probe, k_rhs : point probes for parity tests; k_dfma : FP64 peak microbenchmark
#pragma once
#include "torj_device.cuh"
#include "torj_warm.cuh"
#include "torj_handoff.cuh"
#include "torj_exactsum.cuh"

#include <type_traits>

namespace torj {

// Runge-Kutta tableaux (OrdinaryDiffEq Tsit5 / OwrenZen3; SURVEY.md A.2), uploaded once per context
struct Tableau {
    double a[7][7];
    double bt[7];
};
__constant__ Tableau c_tab[2];

struct SolverOpts {
    int n_segments;
    int max_steps;
    double s_max, dtmax, abstol, reltol, psi_stop, p_stop, te_min, alpha_floor;
    int max_harmonic;
};

struct BundleDev {
    long long n_rays;
    const double* pos;     // [3][n] launch positions
    const double* dir;     // [3][n] vacuum directions
    const double* weight;  // [n]
    const double* freq;    // [n] or [1]
    const int* mode;       // [n] or [1]
    int per_ray_fm;
    double* u0;            // [7][n] state at plasma entry
    double* s0;            // [n] vacuum path length
    double* psi_launch;    // [n]
    int* status;           // [n] written by k_ray_init (rays with status != 0 are never traced), then by k_trace at retirement
    double* P_final;       // [n]
    double* P_dep;         // [n] profile-integrated deposited power of the ray
    int* n_points;         // [n]
};

struct TrajDev {
    long long first, count;
    int max_pts;
    double *s, *xyz, *P, *dP, *prof;  // [count][max], [count][3][max], [count][max], [count][max], [count][n_psi]
};

// Plasma set (torj_bundle_trace_plasmas): beam b is traced through plasma beam_plasma[b]. Every plasma of a set is on the
// grid of the DevTables the kernels receive, so a ray's own plasma contributes only its table base and psi_prof_max.
struct PlasmaSetDev {
    const double2* const* A;    // [n_plasmas] table base of each plasma; NULL = one plasma, the DevTables passed
    const DevTables* const* T;  // [n_plasmas] each plasma's DevTables in device memory (ray init, life prediction)
    const int* beam_plasma;     // [n_beams]
    const int* beam_id;         // [n_rays]
};

// the tables of ray i: T0 itself, or with a plasma set those of the ray's plasma (off the hot path: ray init, life prediction)
__device__ __forceinline__ DevTables ray_tables(const DevTables& T0, const PlasmaSetDev& P, long long i) {
    return P.T ? *P.T[P.beam_plasma[P.beam_id[i]]] : T0;
}

// ------------------------------------------------------------------------------------------------
// ray initialisation
// ------------------------------------------------------------------------------------------------
__device__ inline bool box_intersection(const DevTables& T, const double p0[3], const double N0[3], double* t_out) {
    double best = INFINITY;
    const double tiny = 1e-12;
    double a = N0[0] * N0[0] + N0[1] * N0[1];
    double b = 2.0 * (p0[0] * N0[0] + p0[1] * N0[1]);
    for (int k = 0; k < 2; ++k) {
        double Rc = k == 0 ? T.r0 : T.rlast;
        double c = p0[0] * p0[0] + p0[1] * p0[1] - Rc * Rc;
        if (a <= 0.0) continue;
        double disc = b * b - 4.0 * a * c;
        if (disc < 0.0) continue;
        double sq = sqrt(disc);
        for (int sgn = -1; sgn <= 1; sgn += 2) {
            double t = (-b + sgn * sq) / (2.0 * a);
            if (t <= tiny) continue;
            double z = p0[2] + t * N0[2];
            if (z >= T.z0 && z <= T.zlast && t < best) best = t;
        }
    }
    if (N0[2] != 0.0) {
        for (int k = 0; k < 2; ++k) {
            double Zc = k == 0 ? T.z0 : T.zlast;
            double t = (Zc - p0[2]) / N0[2];
            if (t <= tiny) continue;
            double R = hypot(p0[0] + t * N0[0], p0[1] + t * N0[1]);
            if (R >= T.r0 && R <= T.rlast && t < best) best = t;
        }
    }
    if (!isfinite(best)) return false;
    *t_out = best;
    return true;
}

// 3x3 solve with complete pivoting; pivots below 1e-14*scale are skipped (their unknown stays 0): the
// minimum-norm answer for the zero row+column of the tor=0 central ray
__device__ inline void solve3_robust(double A[3][3], double rhs[3], double x[3]) {
    int rp[3] = {0, 1, 2}, cp[3] = {0, 1, 2};
    int rank = 0;
    double scale = 0.0;
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) scale = fmax(scale, fabs(A[i][j]));
    for (int k = 0; k < 3; ++k) {
        int pi = k, pj = k; double best = 0.0;
        for (int i = k; i < 3; ++i) for (int j = k; j < 3; ++j) {
            double v = fabs(A[rp[i]][cp[j]]);
            if (v > best) { best = v; pi = i; pj = j; }
        }
        if (best <= 1e-14 * scale) break;
        int t = rp[k]; rp[k] = rp[pi]; rp[pi] = t;
        t = cp[k]; cp[k] = cp[pj]; cp[pj] = t;
        for (int i = k + 1; i < 3; ++i) {
            double f = A[rp[i]][cp[k]] / A[rp[k]][cp[k]];
            for (int j = k; j < 3; ++j) A[rp[i]][cp[j]] -= f * A[rp[k]][cp[j]];
            rhs[rp[i]] -= f * rhs[rp[k]];
        }
        rank = k + 1;
    }
    x[0] = x[1] = x[2] = 0.0;
    for (int k = rank - 1; k >= 0; --k) {
        double s = rhs[rp[k]];
        for (int j = k + 1; j < rank; ++j) s -= A[rp[k]][cp[j]] * x[cp[j]];
        x[cp[k]] = s / A[rp[k]][cp[k]];
    }
}

// reference src/solve.jl:40-49; J (if non-null) is the analytic Jacobian of F_k = W_k^2 - N_k^2,
// W_k = n0_k + (ndN - sqrt(Ns^2 - 1 + ndN^2)) n_k
__device__ inline void refraction_equations(const double N[3], double X, double Y, const double n0[3], const double n[3],
                                            const double b[3], double moded, double F[3], double (*J)[3]) {
    double ndN = -(n[0] * n0[0] + n[1] * n0[1] + n[2] * n0[2]);
    double Np = N[0] * b[0] + N[1] * b[1] + N[2] * b[2];
    Disp d = refractive_index_sq<true>(X, Y, 1.0 / Y, Np, moded);
    double Ns = sqrt(d.Ns2);
    double coef = 1.0 / Ns * ndN - sqrt(1.0 - 1.0 / (Ns * Ns) * (1.0 - ndN * ndN));
    for (int k = 0; k < 3; ++k) {
        double Fk = n0[k] / Ns + coef * n[k];
        F[k] = Fk * Fk * (Ns * Ns) - N[k] * N[k];
    }
    if (J) {
        double root = sqrt(d.Ns2 - 1.0 + ndN * ndN);
        double c2 = ndN - root;
        for (int k = 0; k < 3; ++k) {
            double W = n0[k] + c2 * n[k];
            double dW = -n[k] / (2.0 * root);
            for (int j = 0; j < 3; ++j) J[k][j] = 2.0 * W * dW * d.dNp * b[j] - (k == j ? 2.0 * N[k] : 0.0);
        }
    }
}

__global__ void k_ray_init(DevTables T0, BundleDev B, SolverOpts O, PlasmaSetDev P) {
    exp_tab_init();
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B.n_rays) return;
    const DevTables T = ray_tables(T0, P, i);
    const long long n = B.n_rays;
    double x0[3] = {B.pos[i], B.pos[n + i], B.pos[2 * n + i]};
    double N0[3] = {B.dir[i], B.dir[n + i], B.dir[2 * n + i]};
    double f = B.per_ray_fm ? B.freq[i] : B.freq[0];
    int mode = B.per_ray_fm ? B.mode[i] : B.mode[0];
    RayConst rc = make_ray_const(f, mode, O.te_min, O.max_harmonic, O.alpha_floor);
    int status = 0;
    B.P_final[i] = 0.0; B.P_dep[i] = 0.0; B.n_points[i] = 0;
    B.psi_launch[i] = psi_at(T, x0);

    // ---- first_point (reference src/solve.jl:18-38)
    double p[3] = {x0[0], x0[1], x0[2]};
    {
        double R = sqrt(x0[0] * x0[0] + x0[1] * x0[1]);
        if (!inside_grid(T, R, x0[2])) {
            double t;
            if (!box_intersection(T, x0, N0, &t)) { B.status[i] = 2; B.n_points[i] = -1; return; }
            for (int k = 0; k < 3; ++k) p[k] = x0[k] + N0[k] * t;
        }
    }
    {
        auto g = [&](double t) {
            double xx[3] = {p[0] + t * N0[0], p[1] + t * N0[1], p[2] + t * N0[2]};
            return psi_at(T, xx) - T.psi_prof_max;
        };
        double a = 0.0, b = 0.5;
        double ga = g(a), gb = g(b), root;
        if (ga == 0.0) root = a;
        else if (gb == 0.0) root = b;
        else {
            if ((ga < 0.0) == (gb < 0.0)) { B.status[i] = 2; B.n_points[i] = -2; return; }
            for (int it = 0; it < 200; ++it) {
                double m = 0.5 * (a + b);
                if (m <= a || m >= b) break;
                double gm = g(m);
                if (gm == 0.0) { a = b = m; ga = gb = 0.0; break; }
                if ((gm < 0.0) == (ga < 0.0)) { a = m; ga = gm; } else { b = m; gb = gm; }
            }
            root = (ga <= 0.0) ? a : b;  // the end with psi <= psi_prof_max (assert src/solve.jl:138)
        }
        for (int k = 0; k < 3; ++k) p[k] += root * N0[k];
        double psi_ref = psi_at(T, p);
        if (!(fabs(psi_ref - T.psi_prof_max) < 1e-6)) { B.status[i] = 2; B.n_points[i] = -3; return; }
        if (psi_ref > T.psi_prof_max)
            for (int k = 0; k < 3; ++k) p[k] += 2.0 * (psi_ref - T.psi_prof_max) * N0[k];
        if (!(psi_at(T, p) <= T.psi_prof_max)) { B.status[i] = 2; B.n_points[i] = -4; return; }
    }
    // ---- vacuum_plasma_refraction (reference src/solve.jl:51-74)
    double Np[3];
    {
        double u[7] = {p[0], p[1], p[2], N0[0], N0[1], N0[2], 1.0}, du[7];
        Counters c0 = {0, 0, 0, 0, 0, 0, 0};
        PointVals pv;
        rhs<false>(T, rc, u, du, c0, &pv);
        Disp d0 = refractive_index_sq<false>(pv.X, pv.Y, 1.0 / pv.Y, 0.0, rc.moded);
        if (!(d0.Ns2 > 0.0)) { B.status[i] = 1; B.n_points[i] = -9; return; }
        double N_est = sqrt(d0.Ns2);
        double R = sqrt(p[0] * p[0] + p[1] * p[1]);
        double psi, pR, pZ;
        eval_psi(T, R, p[2], &psi, &pR, &pZ);
        double nv[3] = {pR * p[0] / R, pR * p[1] / R, pZ};
        double nn = sqrt(nv[0] * nv[0] + nv[1] * nv[1] + nv[2] * nv[2]);
        for (int k = 0; k < 3; ++k) nv[k] /= nn;
        double n0n = sqrt(N0[0] * N0[0] + N0[1] * N0[1] + N0[2] * N0[2]);
        double n0[3] = {N0[0] / n0n, N0[1] / n0n, N0[2] / n0n};
        double N[3] = {N0[0] * N_est, N0[1] * N_est, N0[2] * N_est};
        bool ok = false;
        for (int it = 0; it < 50 && status == 0; ++it) {
            double F[3], J[3][3];
            refraction_equations(N, pv.X, pv.Y, n0, nv, pv.b, rc.moded, F, J);
            double fn = fmax(fabs(F[0]), fmax(fabs(F[1]), fabs(F[2])));
            if (!(fn == fn)) { status = 2; B.n_points[i] = -5; break; }
            if (fn < 1e-12) {
                // ftol reached (reference src/solve.jl:72). The reference then asserts |Λ| < 1e-12 (src/solve.jl:141), and
                // |Λ| = |sum_k F_k| can be up to 3 ftol: keep iterating until that assertion holds too instead of
                // failing the ray on a residual that one more Newton step removes.
                double Lam = N[0] * N[0] + N[1] * N[1] + N[2] * N[2]
                             - refractive_index_sq<false>(pv.X, pv.Y, 1.0 / pv.Y, N[0] * pv.b[0] + N[1] * pv.b[1] + N[2] * pv.b[2], rc.moded).Ns2;
                if (fabs(Lam) < 5e-13 || it >= 40) { ok = true; break; }
            }
            double r[3] = {-F[0], -F[1], -F[2]}, dx[3];
            solve3_robust(J, r, dx);
            double lam = 1.0, f2 = F[0] * F[0] + F[1] * F[1] + F[2] * F[2];
            bool stepped = false;
            for (int ls = 0; ls < 30; ++ls) {
                double Nt[3] = {N[0] + lam * dx[0], N[1] + lam * dx[1], N[2] + lam * dx[2]}, Ft[3];
                refraction_equations(Nt, pv.X, pv.Y, n0, nv, pv.b, rc.moded, Ft, nullptr);
                double f2t = Ft[0] * Ft[0] + Ft[1] * Ft[1] + Ft[2] * Ft[2];
                if (f2t == f2t && f2t < f2) { for (int k = 0; k < 3; ++k) N[k] = Nt[k]; stepped = true; break; }
                lam *= 0.5;
            }
            if (!stepped) { status = 2; B.n_points[i] = -6; break; }
        }
        if (!ok && status == 0) { status = 2; B.n_points[i] = -7; }
        if (status != 0) { B.status[i] = status; return; }
        for (int k = 0; k < 3; ++k) Np[k] = N[k];
        // assert |Λ| < 1e-12 (reference src/solve.jl:141)
        double u2[7] = {p[0], p[1], p[2], Np[0], Np[1], Np[2], 1.0};
        rhs<false>(T, rc, u2, du, c0, &pv);
        // Λ as the reference forms it: norm(N)^2 - Ns^2
        if (!(fabs(pv.Lambda) < 1e-12)) { B.status[i] = 2; B.n_points[i] = -8; return; }
    }
    B.u0[i] = p[0]; B.u0[n + i] = p[1]; B.u0[2 * n + i] = p[2];
    B.u0[3 * n + i] = Np[0]; B.u0[4 * n + i] = Np[1]; B.u0[5 * n + i] = Np[2];
    B.u0[6 * n + i] = 1.0;
    double dx0 = p[0] - x0[0], dx1 = p[1] - x0[1], dx2 = p[2] - x0[2];
    B.s0[i] = sqrt(dx0 * dx0 + dx1 * dx1 + dx2 * dx2);
    B.status[i] = 0;
}

// ------------------------------------------------------------------------------------------------
// trace kernel
// ------------------------------------------------------------------------------------------------
struct TraceArgs {
    DevTables T;
    BundleDev B;
    SolverOpts O;
    TrajDev J;
    int n_psi;
    int n_beams;                      // one profile row per beam, booked with global-memory RED.ADD.F64
    const int* beam_id;               // [n] (n_beams > 1 only)
    const double* psi_edges;          // [n_psi]
    double* bins;                     // [n_beams][n_psi+2]: weighted shell power, then sum w_i P_i and sum w_i
    unsigned long long* next_ray;     // work queue head
    unsigned long long* counters;     // n_acc, n_rej, n_rhs, n_alpha, n_harm, n_rays_ok, n_prune, n_askip
    // segment hand-off (interleave = 1): work item i is segment i / n of ray i % n; a ray changes lanes between
    // segments, so all rays advance together and the bundle ends after n/lanes ray-times instead of ceil(n/lanes)
    int interleave;
    double* hand;                     // [n][TORJ_HAND_D] ray state between two segments
    int* seg_done;                    // [n] the ray's hand-off word: segments completed, dropped items, whether a lane holds
                                      // the ray, or TORJ_SEG_RETIRED (layout and transitions in torj_handoff.cuh)
    int* rays_left;                   // rays not yet retired
    const double2* warm_tab;          // [501] (t_i, exp(-t_i^2) dt): set_extv! tables of the warm-plasma model
    double* u_final;                  // [7][n] state of every ray at retirement, or NULL
    // life-ordered rounds (k_predict_life): ray r's segment k is item (round k + lmax - life[r], r), so that long-lived rays
    // start first and all rays END together — no tail of a few long rays running alone. NULL = every ray starts in round 0
    const int* life;                  // [n] predicted cost of every ray in rounds (segments, those inside the absorbing layer weighted)
    const int* lmax;                  // max of life[]
    PlasmaSetDev P;                   // k_trace<..., SET = true> only (last member: the other instantiations keep their layout)
    // exact-sum mode (torj_exactsum.cuh), k_trace<..., XS = true> only: every booking goes, exactly, into
    // xs[bin * TORJ_XS_WORDS ...] (bins as in `bins`); the buffer's status words are xs[-2], xs[-1]
    long long* xs;
};
#define TORJ_HAND_D 20

__device__ __forceinline__ double eps_of(double x) {  // Julia eps(x)
    x = fabs(x);
    return __longlong_as_double(__double_as_longlong(x) + 1) - x;
}

__device__ __forceinline__ double rms7(const double v[7]) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 7; ++i) s = fma(v[i], v[i], s);
    return sqrt(s / 7.0);
}

// Final position outside the grid? Out of line on purpose: inlined, the compiler hoisted the side-effect-free sqrt(x^2 + y^2)
// out of the retirement branch and ran it on EVERY trip (20 instructions, 2.2 % of the kernel's stall samples in ncu).
__device__ __noinline__ bool left_grid(double r0, double rlast, double z0, double zlast, double x, double y, double z) {
    const double R = sqrt(x * x + y * y);
    return !(R >= r0 && R <= rlast && z >= z0 && z <= zlast);
}

// pow() expands to ~150 instructions with slow paths; the controller needs it only on rejected / shrinking steps,
// so one out-of-line copy keeps the hot loop small
__device__ __noinline__ double pow_nl(double x, double y) { return pow(x, y); }

template <int SCH>
struct Scheme;
template <> struct Scheme<0> { static constexpr int S = 7; static constexpr int ORDER = 5; };
template <> struct Scheme<1> { static constexpr int S = 4; static constexpr int ORDER = 3; };

#define TORJ_TPB 128
// Runge-Kutta stage derivatives k[S][7] live in shared memory, not in (L1-backed) local memory, stored as 4 double2 per
// stage and thread (8th slot unused), so that a stage is read with 4 LDS.128 instead of 7 LDS.64
#define TORJ_K_WORDS (56 * TORJ_TPB)  // doubles of stage storage per CTA
#define TORJ_PARK_SLOTS 9  // doubles per thread of parked per-segment / per-ray scalars (7 doubles + 4 ints)
#define TORJ_LIFE_HARM_COST 0.25  // k_predict_life: rounds one evaluated harmonic integral per pilot point adds to a ray's predicted
                                  // cost (segments inside the absorbing layer take longer). 1/16 and 1/8 shards of the 1 M-ray sweep:
                                  // 0 -> 174.8 / 299.2 ms, 0.25 -> 166.7 / 288.9, 0.5 -> 168.1 / 291.0, 0.75 -> 176.3 / 295.3; beam unchanged
#define TORJ_MINB 2  // resident CTAs per SM the register allocation is bounded for (2 -> 255 regs, 3 -> 168, 4 -> 128)
// per-ray status codes of include/torj_cuda.h: everything but OK(0), LEFT_GRID(3) and TRAJ_TRUNCATED(6) ends the ray
#define TORJ_FATAL(s) ((s) != 0 && (s) != 6 && (s) != 3)

// The lane's count of exact bookings: k_trace's parked int slot PKI(3) (flushed into the status word before it can wrap,
// the rest at the end of k_trace)
__device__ __forceinline__ unsigned* xs_count_slot() {
    extern __shared__ __align__(16) double smem[];
    return reinterpret_cast<unsigned*>(smem + TORJ_K_WORDS + 7 * TORJ_TPB) + 3 * TORJ_TPB + threadIdx.x;
}

// One exact booking (exact-sum mode): v's digits into the words of bin `bin`, fire-and-forget integer REDs. Out of line and
// with few arguments, by value, so the hot loop carries only the call. The status words precede the words.
__device__ __noinline__ void xs_book(long long* xs, size_t bin, double v) {
    unsigned long long* stat = reinterpret_cast<unsigned long long*>(xs - TORJ_XS_STAT);
    unsigned* nb = xs_count_slot();
    const TorjXsSplit s = torj_xs_split(v);
    if (!s.ok) { atomicAdd(&stat[1], 1ull); return; }
    unsigned long long* w = reinterpret_cast<unsigned long long*>(xs + bin * TORJ_XS_WORDS + s.k);
#pragma unroll
    for (int j = 0; j < 3; ++j)
        if (s.d[j]) atomicAdd(&w[j], (unsigned long long)s.d[j]);  // two's complement: a signed add
    const unsigned c = *nb + 1;
    if (c == 0x80000000u) { atomicAdd(&stat[0], (unsigned long long)c); *nb = 0; }
    else *nb = c;
}

// A retiring ray's two per-beam bookings, w P_dep and w, into the bins row_bin + n_psi, + n_psi + 1: one call site less
// in k_trace
__device__ __noinline__ void xs_book_ray(long long* xs, size_t row_bin, double w_pdep, double w) {
    xs_book(xs, row_bin, w_pdep);
    xs_book(xs, row_bin + 1, w);
}

// Integrator phases. Every trip of the kernel's main loop evaluates the RHS exactly once per lane that holds a
// ray, whatever that lane's phase, so the expensive code is always warp-converged; the cheap phase-specific
// bookkeeping after it is the only divergent part. A lane that retires its ray draws a new one on the next trip.
// PH_WAIT / PH_RESUME (segment hand-off only): the lane holds a work item whose previous segment is still running on
// another lane / has just loaded a ray's state. Phases >= PH_SEED evaluate the RHS.
enum { PH_IDLE = 0, PH_WAIT = 1, PH_RESUME = 2, PH_SEED = 3, PH_INITDT = 4, PH_STAGE = 5, PH_CALLBACK = 6 };
enum { ACT_NONE = 0, ACT_BEGIN_SEGMENT = 1, ACT_BEGIN_STEP = 2, ACT_END_SEGMENT = 3, ACT_AFTER_ACCEPT = 4 };

// HIGH = true: harmonics above the third enabled (torj_options.max_harmonic > 3); see abs_albajar
// MODEL: 0 = Albajar absorption (reference src/absorption.jl), 1 = warm-plasma damping (src/general_absorption.jl α,
//   torj_warm.cuh): the RHS leaves alpha out and the warp evaluates it cooperatively right after.
// LPR: lanes per ray (torj_options.lanes_per_ray): 1 = a thread per ray; 8 / 32 = a group of 8 lanes / a whole warp per
//   ray. All lanes of a group carry the same ray state and run the same bookkeeping (no divergence inside the group,
//   nothing to broadcast); the parallel parts — the nodes of the harmonic integrals / of the warm quadrature — are split
//   over the group and butterfly-reduced, so every lane of it sees bit-identical sums. The group's first lane alone
//   performs the side effects (bins, per-ray outputs, queue bookkeeping). For bundles below the resident lanes
//   (37 888), where the time is one ray's latency, for the tail of a large bundle (`resume`), and for the warm model,
//   whose alpha costs ~100x the rest of the RHS.
// SET = true: a plasma set (a.P). The grid comes from a.T as always; the table base is per lane, bound with the ray
//   (a ray's plasma is that of its beam), so rays of several equilibria share one launch.
template <int SCH, bool HIGH = false, int MODEL = 0, int LPR = 1, bool SET = false, bool XS = false>
__global__ void __launch_bounds__(TORJ_TPB, TORJ_MINB) k_trace(TraceArgs a) {
    exp_tab_init();
    constexpr bool COOP = LPR == 32;
    constexpr int S = Scheme<SCH>::S;
    constexpr int ORDER = Scheme<SCH>::ORDER;
    extern __shared__ __align__(16) double smem[];
    const double* __restrict__ s_edges = a.psi_edges;      // psi levels: read-only, through L1 (__ldg)
    double* ks = smem + 2 * threadIdx.x;                   // KK(j, 2p + q) at ks[(j*4+p)*2*TORJ_TPB + q]: 16-byte pairs
#define KK(j, i) ks[((j) * 4 + ((i) >> 1)) * 2 * TORJ_TPB + ((i) & 1)]
    __shared__ unsigned long long s_cnt[8];
    __shared__ double s_tot[2];
    __shared__ double s_a[7][7], s_bt[7];
    const int n_psi = a.n_psi;
    if (threadIdx.x < 8) s_cnt[threadIdx.x] = 0ull;
    if (threadIdx.x < 2) s_tot[threadIdx.x] = 0.0;
    if (threadIdx.x < 49) s_a[threadIdx.x / 7][threadIdx.x % 7] = c_tab[SCH].a[threadIdx.x / 7][threadIdx.x % 7];
    if (threadIdx.x < 7) s_bt[threadIdx.x] = c_tab[SCH].bt[threadIdx.x];
    __syncthreads();

    std::conditional_t<SET, DevTables, const DevTables> T = a.T;  // SET: T.A is rebound per ray
    const SolverOpts& O = a.O;
    const long long n = a.B.n_rays;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned FULL = 0xffffffffu;
    const bool writer = (lane & (unsigned)(LPR - 1)) == 0;  // the lane that performs a ray's side effects
    const unsigned gmask = group_mask(LPR);                 // the lanes that hold my ray
    const unsigned gleader = lane & ~(unsigned)(LPR - 1);
    const unsigned leaders = LPR == 1 ? FULL : LPR == 2 ? 0x55555555u : LPR == 4 ? 0x11111111u : LPR == 8 ? 0x01010101u : 1u;
    static_assert(LPR == 1 || LPR == 2 || LPR == 4 || LPR == 8 || LPR == 32, "lanes per ray");
    const double beta1 = 7.0 / (10.0 * ORDER), beta2 = 2.0 / (5.0 * ORDER);
    const double gamma_c = 0.9, qmin = 0.2, qmax = 10.0, qoldinit = 1e-4;
    // OrdinaryDiffEq's step_accept_controller! holds the step (q := 1) when qsteady_min = 1 <= q <= qsteady_max = 1.2.
    // q = EEst^beta1 / qold^beta2 / gamma <= 1.2  <=>  EEst^7 <= (1.2 gamma)^(10 k) qold^4   (beta1 = 7/(10k), beta2 = 4/(10k))
    const double qsteady_min = 1.0, qsteady_max = 1.2;
    const double gamma_pow = pow(qsteady_max * gamma_c, 10.0 * ORDER);
    const double dtmax_pow = pow(O.dtmax, -(double)ORDER);
    const double s_step = O.s_max / (double)O.n_segments;

    // per-lane ray state
    // Scalars touched once per segment or per ray live in shared memory ([slot][thread], conflict-free): the kernel
    // sits at the 255-register limit and the compiler, not knowing trip frequencies, otherwise spills values that
    // every RHS evaluation touches (ray constants, counters) to local memory (122 -> 72 bytes of spills, -1 % time;
    // parking the once-per-step scalars as well removes the spills altogether but gains nothing more).
    double* pk = smem + TORJ_K_WORDS + threadIdx.x;
#define PK(k) pk[(k) * TORJ_TPB]
    long long& ray = *reinterpret_cast<long long*>(&PK(0));
    long long& tj = *reinterpret_cast<long long*>(&PK(1));  // index into the trajectory window or -1
    double& s0 = PK(2);
    double& dt0 = PK(3);
    double& d1 = PK(4);
    double& tot_dep = PK(5);
    double& tot_w = PK(6);
    int* pki = reinterpret_cast<int*>(pk + 7 * TORJ_TPB - threadIdx.x) + threadIdx.x;
#define PKI(k) pki[(k) * TORJ_TPB]
    int& seg = PKI(0);
    int& last_stat = PKI(1);
    unsigned int& rays_ok = *reinterpret_cast<unsigned int*>(&PKI(2));
    ray = -1; tj = -1; s0 = 0.0; dt0 = 0.0; d1 = 0.0; tot_dep = 0.0; tot_w = 0.0; seg = 0; last_stat = 0; rays_ok = 0;
    if constexpr (XS) PKI(3) = 0;  // exact-sum bookings of this lane (xs_count_slot)
    // warm model, one ray per lane: shared-memory slots where a lane's quadrature sums wait for the serial solve
    double* wstash = smem + TORJ_K_WORDS + TORJ_PARK_SLOTS * TORJ_TPB + threadIdx.x;
    int phase = PH_IDLE, st = 0;
    bool exhausted = false;
    double u[7], tmp[7];
    double wgt = 0.0, pdep = 0.0;
    double t = 0.0, tstop = 0.0, dt = 0.0, qold = qoldinit, dtnew = 0.0;
    double psi_cur = 0.0, dpsi_cur = 0.0, psi_new = 0.0, dpsi_new = 0.0, P_a = 1.0, dP_a = 0.0, hstep = 0.0;
    int npts = 0, rstat = 0, nstep = 0;
    bool a_skip = false, a_skip_next = false;
    int wseg = 0;  // segment index of the work item held (segment hand-off)
    bool own = false;  // PH_WAIT: the ray's state is already in this lane's registers (continuation), nothing to load
    int cadence = 0;  // trip number modulo the trips per step (warp-uniform)
    RayConst rc = make_ray_const(1e11, 1, O.te_min, O.max_harmonic, O.alpha_floor);
    DepoState dst = {0, 0, 1.0};
    Counters cnt = {0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int i = 0; i < 7; ++i) { u[i] = 0.0; tmp[i] = 0.0; }
#pragma unroll
    for (int j = 0; j < S; ++j)
#pragma unroll
        for (int i = 0; i < 7; ++i) KK(j, i) = 0.0;

    double* beam_bins = a.bins;  // this ray's beam row (scans: rays of many launchers / frequencies in one bundle)
    auto sink = [&](int shell, double dP) {
        pdep += dP;
        if (!writer) return;
        if constexpr (XS) xs_book(a.xs, (size_t)(beam_bins - a.bins) + shell, wgt * dP);
        else atomicAdd(&beam_bins[shell], wgt * dP);
        if (tj >= 0) atomicAdd(&a.J.prof[tj * n_psi + shell], dP);  // (a ray may change SMs between segments)
    };
    auto put_point = [&](double s, const double* xx, double P, double dP) {
        if (tj >= 0) {
            if (npts < a.J.max_pts) {
                if (writer) {
                size_t o = (size_t)tj * a.J.max_pts + npts;
                a.J.s[o] = s; a.J.P[o] = P; a.J.dP[o] = dP;
                size_t ox = (size_t)tj * 3 * a.J.max_pts + npts;
                a.J.xyz[ox] = xx[0]; a.J.xyz[ox + a.J.max_pts] = xx[1]; a.J.xyz[ox + 2 * (size_t)a.J.max_pts] = xx[2];
                }
            } else if (rstat == 0) {
                rstat = 6;  // TORJ_RAY_TRAJ_TRUNCATED
            }
        }
        npts++;
    };

    // per-ray constants of the lane (both at the first pick-up of a ray and when a hand-off state is loaded)
    auto bind_ray = [&](long long idx) {
        ray = idx;
        s0 = a.B.s0[idx];
        wgt = a.B.weight[idx];
        double f = a.B.per_ray_fm ? a.B.freq[idx] : a.B.freq[0];
        int mode = a.B.per_ray_fm ? a.B.mode[idx] : a.B.mode[0];
        rc = make_ray_const(f, mode, O.te_min, O.max_harmonic, O.alpha_floor);
        if (a.n_beams > 1) beam_bins = a.bins + (size_t)a.beam_id[idx] * (n_psi + 2);
        if constexpr (SET) T.A = a.P.A[a.P.beam_plasma[a.beam_id[idx]]];
        if (TORJ_FATAL(last_stat)) {  // a dead ray may have left NaN/Inf in the stage slots (0 * NaN != 0)
#pragma unroll
            for (int j = 0; j < S; ++j)
#pragma unroll
                for (int i = 0; i < 7; ++i) KK(j, i) = 0.0;
            last_stat = 0;
        }
        tj = (idx >= a.J.first && idx < a.J.first + a.J.count) ? idx - a.J.first : -1;
    };
    auto start_ray = [&](long long idx) {
        bind_ray(idx);
#pragma unroll
        for (int i = 0; i < 7; ++i) { u[i] = a.B.u0[(size_t)i * n + idx]; tmp[i] = u[i]; }
        seg = 0; npts = 0; rstat = 0; pdep = 0.0;
        // samples 1 and 2: launch point and plasma entry (reference src/solve.jl:149-153)
        double xl[3] = {a.B.pos[idx], a.B.pos[n + idx], a.B.pos[2 * n + idx]};
        put_point(0.0, xl, 1.0, 0.0);
        put_point(s0, u, 1.0, 0.0);
        phase = PH_SEED;
        a_skip = false;
    };
    // segment hand-off: the state a ray carries from one segment to the next (L2-coherent accesses: another SM wrote it)
    auto save_ray = [&]() {
        if (!writer) return;
        double2* h = reinterpret_cast<double2*>(a.hand + (size_t)ray * TORJ_HAND_D);
        __stcg(h + 0, make_double2(u[0], u[1])); __stcg(h + 1, make_double2(u[2], u[3]));
        __stcg(h + 2, make_double2(u[4], u[5])); __stcg(h + 3, make_double2(u[6], KK(0, 0)));
        __stcg(h + 4, make_double2(KK(0, 1), KK(0, 2))); __stcg(h + 5, make_double2(KK(0, 3), KK(0, 4)));
        __stcg(h + 6, make_double2(KK(0, 5), KK(0, 6))); __stcg(h + 7, make_double2(psi_cur, dpsi_cur));
        __stcg(h + 8, make_double2(dst.P_last, pdep));
        __stcg(h + 9, make_double2(__hiloint2double(dst.shell, dst.valid), __hiloint2double(npts, rstat | (a_skip ? 256 : 0))));
        __threadfence();
    };
    auto load_ray = [&](long long idx) {
        bind_ray(idx);
        const double2* h = reinterpret_cast<const double2*>(a.hand + (size_t)idx * TORJ_HAND_D);
        double2 q;
        q = __ldcg(h + 0); u[0] = q.x; u[1] = q.y;
        q = __ldcg(h + 1); u[2] = q.x; u[3] = q.y;
        q = __ldcg(h + 2); u[4] = q.x; u[5] = q.y;
        q = __ldcg(h + 3); u[6] = q.x; KK(0, 0) = q.y;
        q = __ldcg(h + 4); KK(0, 1) = q.x; KK(0, 2) = q.y;
        q = __ldcg(h + 5); KK(0, 3) = q.x; KK(0, 4) = q.y;
        q = __ldcg(h + 6); KK(0, 5) = q.x; KK(0, 6) = q.y;
        q = __ldcg(h + 7); psi_cur = q.x; dpsi_cur = q.y;
        q = __ldcg(h + 8); dst.P_last = q.x; pdep = q.y;
        q = __ldcg(h + 9);
        dst.shell = __double2hiint(q.x); dst.valid = __double2loint(q.x);
        npts = __double2hiint(q.y);
        const int fl = __double2loint(q.y);
        rstat = fl & 255; a_skip = (fl & 256) != 0;
        seg = wseg;
        phase = PH_RESUME;
    };
    // the held item (ray idx, segment wseg) is ready: take the ray over
    auto start_item = [&](long long idx) {
        __threadfence();
        if (wseg > 0) {
            load_ray(idx);
        } else if (a.B.status[idx] == 0) {
            start_ray(idx);
        } else {  // failed initialisation (k_ray_init): retire at once
            if (writer) {
                atomicExch(&a.seg_done[idx], TORJ_SEG_RETIRED);
                atomicSub(a.rays_left, 1);
            }
            phase = PH_IDLE; ray = -1;
        }
    };
    // A freshly drawn item (ray idx, segment wseg). Nobody ever waits for an unfinished predecessor: if the ray's previous
    // segment is still running, the item is DROPPED and marked as such in the ray's word, and the lane that runs that segment
    // finds the mark when it hands in and continues with the ray itself (ACT_END_SEGMENT). A ready claim sets the word's
    // RUNNING bit, and a claim that finds it set is void: the holder already continues with that segment. Claims and
    // hand-ins change the word only through the transitions of torj_handoff.cuh, each in one compare-and-swap, so exactly
    // one lane runs every segment. (Idle lanes that ran ahead in the queue used to hold such items and block; with
    // life-ordered rounds that would idle most lanes while the long rays start.)
    auto claim = [&](long long idx, bool aligned) {
        ray = idx;
        int verdict = 0;  // 0 void, 1 ready
        if (writer) {
            int w = wseg;  // first guess: ready, nothing dropped (the usual case, then one CAS); a wrong guess reads the word
            for (;;) {
                const TorjSegMove m = torj_seg_claim(w, wseg);
                if (m.w == w) break;  // void with nothing to mark: retired, already run, held, or already dropped
                const int old = atomicCAS(&a.seg_done[idx], w, m.w);
                if (old == w) { verdict = m.go; break; }
                w = old;
            }
        }
        if (LPR > 1) verdict = __shfl_sync(gmask, verdict, gleader);
        if (verdict == 0) {
            phase = PH_IDLE; ray = -1;
        } else if (aligned) {
            start_item(idx);
        } else {
            own = false;
            phase = PH_WAIT;  // ready, and mine: starts on the warp's next aligned trip
        }
    };

    // item space: item i = (round i / n, ray i % n); the ray's segment is the round, shifted by its predicted life
    const int lmax = a.life ? __ldg(a.lmax) : 0;
    const int n_rounds = O.n_segments + (a.life ? lmax - 1 : 0);  // a ray of predicted life 1 starts in round lmax - 1
    const long long n_items = n * (long long)n_rounds;
    for (;;) {
        // ---- warp-ballot retire-and-refill: idle lanes draw the next work items from the global queue.
        // With segment hand-off a segment starts only on every (S-1)-th trip of the warp: a step is S-1 trips, so the
        // FSAL stages — the only ones that evaluate alpha in full — of all lanes of a warp fall on the same trips for
        // good, instead of some lane paying for alpha on every trip (-2.8 % on both bench workloads).
        // (Restarting the cadence whenever no lane of the warp is inside a segment would save the in-step lanes their
        // <= 4 idle trips per segment, but measured +1.5 %: the fixed cadence is also what regroups stragglers.)
        const bool aligned = (cadence == 0);
        cadence = (cadence + 1 == S - 1) ? 0 : cadence + 1;
        // (wrapping the refill logic below into one vote over "some lane is not busy" measured neutral to slower: 99.2 against 99.0)
        if (a.interleave && phase == PH_WAIT && aligned) {
            if (own) phase = PH_RESUME;  // continuation: the state is here
            else start_item(ray);
        }
        unsigned need = __ballot_sync(FULL, phase == PH_IDLE && !exhausted);
        if (need) {
            int leader = __ffs(need) - 1;
            unsigned long long base = 0;
            int left = 1;
            if ((int)lane == leader) {
                base = atomicAdd(a.next_ray, (unsigned long long)__popc(need & leaders));
                if (a.interleave) left = atomicAdd(a.rays_left, 0);
            }
            base = __shfl_sync(FULL, base, leader);
            left = __shfl_sync(FULL, left, leader);
            if (phase == PH_IDLE && !exhausted) {
                long long idx = (long long)base + __popc(need & leaders & ((1u << gleader) - 1u));
                if (!a.interleave) {
                    if (idx >= n) {
                        exhausted = true;
                    } else if (a.B.status[idx] == 0) {  // failed initialisations were reported by k_ray_init
                        start_ray(idx);
                    }
                } else {
                    // item idx = segment idx / n of ray idx % n; items of retired rays are void
                    if (left == 0 || idx >= n_items) {
                        exhausted = true;
                    } else {
                        const int round = (int)(idx / n);
                        const long long r = idx - (long long)round * n;
                        wseg = a.life ? round - (lmax - __ldg(a.life + r)) : round;
                        if (wseg >= 0 && wseg < O.n_segments) claim(r, aligned);  // else: the ray has not started yet / is over
                    }
                }
            }
        }
        if (__all_sync(FULL, phase == PH_IDLE && exhausted)) break;

        // ---- the one RHS evaluation of this trip (reference src/solve.jl:85-95), warp-converged
        double out[9];
        const bool inner = (phase == PH_STAGE && st < S - 1);  // an inner Runge-Kutta stage: five trips of six
        // alpha is evaluated in full at the FSAL stage (= first stage of the next step) and in the seed / callback /
        // initial-dt phases; the inner stages take alpha = 0 when that evaluation found every harmonic negligible
        // with a 1e10 margin (abs_albajar)
        if (MODEL == 0) {
            if (phase >= PH_SEED) {
                rhs<true, true, HIGH, LPR>(T, rc, tmp, out, cnt, nullptr, inner && a_skip, &a_skip_next, nullptr,
                                            !inner && phase != PH_INITDT);  // psi_N is used at the FSAL / seed / callback stages only
                if (!inner) a_skip = a_skip_next;
            }
        } else {
            // warm-plasma model: the RHS without alpha, then the warp-cooperative alpha of every lane that needs one
            AlphaIn ain;
            ain.X = 0.1; ain.Y = 0.5; ain.N2 = 1.0; ain.Np = 0.0; ain.lnTe = -1e300; ain.inorm = 1.0;
            const bool evaluated = phase >= PH_SEED;
            if (evaluated) rhs<false, true, false, false>(T, rc, tmp, out, cnt, nullptr, false, nullptr, &ain, !inner && phase != PH_INITDT);
            const bool want = evaluated && !(inner && a_skip);
            if (evaluated && !want) cnt.n_askip++;
            const double alpha = warm_alpha_warp<COOP>(a.warm_tab, rc, ain, want, wstash, TORJ_TPB, cnt, a_skip_next);
            if (evaluated) {
                out[6] = -tmp[6] * alpha;
                if (!inner) a_skip = a_skip_next;
            }
        }

        // ---- phase bookkeeping
        int act = ACT_NONE;
        // (the common case first and on its own predicate: a ladder over the phases costs three compare-and-branch per trip)
        if (inner) {
            {
#pragma unroll
                for (int i = 0; i < 7; ++i) KK(st, i) = out[i];
                st++;
                // u + dt * sum_j a[st][j] k_j over the st stages computed so far. The cadence keeps the lanes of a warp
                // at the same stage, so the trip count is warp-uniform. A real loop, not unrolled: together with the
                // rolled error sum below, 170 hot instructions less against a 32 KB instruction cache (132.0 -> 126.7 ms);
                // bounded by st rather than summing all S-1 zero-padded rows: 121.9 -> 119.8 ms
                double acc[7];
                {
                    const double a0 = s_a[st][0];  // st >= 2 here: the first term initialises the sums
#pragma unroll
                    for (int i = 0; i < 7; ++i) acc[i] = a0 * KK(0, i);
                }
#pragma unroll 1
                for (int j = 1; j < st; ++j) {
                    const double aj = s_a[st][j];
#pragma unroll
                    for (int i = 0; i < 7; ++i) acc[i] = fma(aj, KK(j, i), acc[i]);
                }
#pragma unroll
                for (int i = 0; i < 7; ++i) tmp[i] = fma(dt, acc[i], u[i]);
            }
        } else if (phase == PH_STAGE) {
            {
#pragma unroll
                for (int i = 0; i < 7; ++i) KK(st, i) = out[i];
                // tmp is the proposed new state (FSAL); embedded error estimate (err = sum_j btilde_j k_j, accumulated
                // stage by stage) and PI controller
                psi_new = out[7];
                dpsi_new = out[8];
                double at[7];
                bool bad = false;
                double utv[7] = {0, 0, 0, 0, 0, 0, 0};
#pragma unroll 1
                for (int j = 0; j < S; ++j) {
                    const double bj = s_bt[j];
#pragma unroll
                    for (int i = 0; i < 7; ++i) utv[i] = fma(bj, KK(j, i), utv[i]);
                }
#pragma unroll
                for (int i = 0; i < 7; ++i) {
                    const double ut = utv[i] * dt;
                    const double au = fabs(u[i]), an = fabs(tmp[i]);
                    at[i] = ut * rcp_fast(O.abstol + (au > an ? au : an) * O.reltol);
                    if (!(tmp[i] == tmp[i])) bad = true;
                }
                if (bad) {
                    rstat = 5;  // TORJ_RAY_NAN
                    act = ACT_END_SEGMENT;
                } else {
                    double EEst = rms7(at);
                    if (EEst <= 1.0) {
                        cnt.n_acc++;
                        double ttmp = t + dt;
                        if (fabs(ttmp - tstop) < 100.0 * eps_of(fmax(t, tstop))) ttmp = tstop;
                        // dt/q >= dt whenever q <= 1 and q := 1 in the dead band 1 <= q <= 1.2; at dt == dtmax the
                        // proposal is clipped back to dtmax, so the two pow() are needed only when the step must
                        // shrink or has to grow back. After the last step of a segment the proposal is never used
                        // (the next segment is a fresh problem).
                        const double e2 = EEst * EEst, q2 = qold * qold;
                        if (ttmp == tstop || (dt == O.dtmax && e2 * e2 * e2 * EEst <= gamma_pow * (q2 * q2))) {
                            dtnew = dt;
                        } else {
                            double qq = 1.0 / qmax;
                            if (EEst != 0.0) {
                                qq = pow_nl(EEst, beta1) / pow_nl(qold, beta2);
                                qq = fmax(1.0 / qmax, fmin(1.0 / qmin, qq / gamma_c));
                            }
                            if (qq >= qsteady_min && qq <= qsteady_max) qq = 1.0;  // steady-state dead band
                            dtnew = dt / qq;
                        }
                        qold = fmax(EEst, qoldinit);
                        hstep = ttmp - t;
                        P_a = u[6]; dP_a = KK(0, 6);
                        t = ttmp;
#pragma unroll
                        for (int i = 0; i < 7; ++i) { u[i] = tmp[i]; KK(0, i) = KK(S - 1, i); }
                        if (u[6] < 0.0) {  // positivity callback (reference src/solve.jl:78-83,159-160): re-evaluate f(u)
                            u[6] = 0.0;
                            tmp[6] = 0.0;
                            phase = PH_CALLBACK;
                        } else {
                            act = ACT_AFTER_ACCEPT;
                        }
                    } else {
                        cnt.n_rej++;
                        double q11 = pow_nl(EEst, beta1);
                        dt = dt / fmin(1.0 / qmin, q11 / gamma_c);
                        act = ACT_BEGIN_STEP;
                    }
                }
            }
        } else if (phase == PH_SEED) {
            // derivative at entry (FSAL seed), psi there, and the vacuum leg launch -> entry (P = 1, straight line)
#pragma unroll
            for (int i = 0; i < 7; ++i) KK(0, i) = out[i];
            psi_cur = out[7];
            dpsi_cur = out[8];
            double psl = a.B.psi_launch[ray];
            dst.shell = locate_shell(s_edges, n_psi, psl);
            dst.valid = 0; dst.P_last = 1.0;
            double dlin = (psi_cur - psl) / s0;
            depo_step(dst, s_edges, n_psi, s0, psl, psi_cur, dlin, dlin, 1.0, 1.0, 0.0, 0.0, sink);
            act = ACT_BEGIN_SEGMENT;
        } else if (phase == PH_INITDT) {
            // second half of OrdinaryDiffEq's ode_determine_initdt (Hairer): out = f(u + dt0 f0)
            double v[7];
#pragma unroll
            for (int i = 0; i < 7; ++i) v[i] = (out[i] - KK(0, i)) / (O.abstol + fabs(u[i]) * O.reltol);
            double d2 = rms7(v) / dt0;
            double md = fmax(d1, d2);
            // 10^(-(2 + log10 md)/order) = (100 md)^(-1/order)
            // dt1 = 10^(-(2 + log10 md)/order) = (100 md)^(-1/order) >= dtmax  <=>  100 md <= dtmax^-order: the usual
            // case (dt = dtmax) needs no pow()
            if (md > 1e-15 && 100.0 * md <= dtmax_pow && 100.0 * dt0 >= O.dtmax) {
                dt = O.dtmax;
            } else {
                double dt1 = (md <= 1e-15) ? fmax(1e-6, dt0 * 1e-3) : pow_nl(100.0 * md, -1.0 / (double)ORDER);
                dt = fmin(fmin(100.0 * dt0, dt1), O.dtmax);
            }
            act = ACT_BEGIN_STEP;
        } else if (phase == PH_CALLBACK) {
#pragma unroll
            for (int i = 0; i < 7; ++i) KK(0, i) = out[i];
            psi_new = out[7];
            dpsi_new = out[8];
            act = ACT_AFTER_ACCEPT;
        } else if (phase == PH_RESUME) {
            act = ACT_BEGIN_SEGMENT;
        }

        // ---- transitions that need no RHS evaluation. The blocks stand in the order of the chain accept -> next step ->
        // segment end -> next segment, so one pass handles every case but one (a fresh segment that skips its initial-dt probe
        // goes back to the step block); as an else-if ladder inside the loop every link of the chain cost a loop trip
        // (five trips of six no lane of a warp in step has a transition: one vote skips the whole ladder)
        if (__any_sync(FULL, act != ACT_NONE))
        while (act != ACT_NONE) {
            if (act == ACT_AFTER_ACCEPT) {
                put_point(t, u, u[6], -KK(0, 6));  // dP/ds sample = P*alpha (reference src/solve.jl:171)
                // streaming deposition over this step (psi and its arc-length derivative came with the FSAL stage)
                depo_step(dst, s_edges, n_psi, hstep, psi_cur, psi_new, dpsi_cur, dpsi_new, P_a, u[6], dP_a, KK(0, 6), sink);
                psi_cur = psi_new; dpsi_cur = dpsi_new;
                dt = fmin(O.dtmax, dtnew);
                act = ACT_BEGIN_STEP;
            }
            if (act == ACT_BEGIN_STEP) {
                if (!(t < tstop)) {
                    act = ACT_END_SEGMENT;
                } else if (++nstep > O.max_steps) {
                    rstat = 4;  // TORJ_RAY_MAX_STEPS
                    act = ACT_END_SEGMENT;
                } else {
                    dt = fmin(dt, tstop - t);
                    st = 1;
                    const double a10 = dt * s_a[1][0];
#pragma unroll
                    for (int i = 0; i < 7; ++i) {
                        const double k0 = KK(0, i);
                        tmp[i] = fma(a10, k0, u[i]);
                    }
                    phase = PH_STAGE;
                    act = ACT_NONE;
                }
            }
            if (act == ACT_END_SEGMENT) {
                // termination tests at the segment end (reference src/solve.jl:174-176) and retirement
                bool done = TORJ_FATAL(rstat) || seg >= O.n_segments || psi_cur > O.psi_stop || u[6] < O.p_stop;
                if (done) {
                    if (rstat == 0 && left_grid(T.r0, T.rlast, T.z0, T.zlast, u[0], u[1], u[2])) rstat = 3;  // TORJ_RAY_LEFT_GRID
                    last_stat = rstat;
                    if (writer) {
                        a.B.status[ray] = rstat;
                        a.B.n_points[ray] = npts;
                        if (a.u_final) {
#pragma unroll
                            for (int i = 0; i < 7; ++i) a.u_final[(size_t)i * n + ray] = u[i];
                        }
                        if (!TORJ_FATAL(rstat)) {
                            a.B.P_final[ray] = u[6];
                            a.B.P_dep[ray] = pdep;
                            if constexpr (XS) {  // per ray, also with one beam: the block sum below would round
                                xs_book_ray(a.xs, (size_t)(beam_bins - a.bins) + n_psi, wgt * pdep, wgt);
                            } else if (a.n_beams > 1) {
                                atomicAdd(&beam_bins[n_psi], wgt * pdep);
                                atomicAdd(&beam_bins[n_psi + 1], wgt);
                            } else {
                                tot_dep += wgt * pdep;
                                tot_w += wgt;
                            }
                            rays_ok++;
                        }
                        if (a.interleave) {
                            atomicExch(&a.seg_done[ray], TORJ_SEG_RETIRED);
                            atomicSub(a.rays_left, 1);
                        }
                    }
                    ray = -1;
                    phase = PH_IDLE;
                    act = ACT_NONE;
                } else if (a.interleave) {
                    // hand the segment in. The next one is a separate work item, usually taken by another lane — unless that
                    // item was drawn while this segment was still running and dropped (claim): then this lane keeps the ray
                    // (the word is read before save_ray's stores and fence, which hide the load; a stale value costs one
                    // more round, the CAS checks it)
                    int w = writer ? __ldcg(&a.seg_done[ray]) : 0;
                    save_ray();
                    int go = 0;
                    if (writer) {
                        for (;;) {
                            const TorjSegMove m = torj_seg_hand_in(w, seg);
                            const int old = atomicCAS(&a.seg_done[ray], w, m.w);
                            if (old == w) { go = m.go; break; }
                            w = old;
                        }
                    }
                    if (LPR > 1) go = __shfl_sync(gmask, go, gleader);
                    if (go) {
                        wseg = seg;
                        own = true;
                        phase = PH_WAIT;  // next segment on the warp's next aligned trip
                    } else {
                        ray = -1;
                        phase = PH_IDLE;
                    }
                    act = ACT_NONE;
                } else {
                    act = ACT_BEGIN_SEGMENT;
                }
            }
            if (act == ACT_BEGIN_SEGMENT) {  // one fresh ODEProblem of the reference (src/solve.jl:155-161)
                seg++;
                t = (double)(seg - 1) * s_step + s0;
                tstop = (double)seg * s_step + s0;
                qold = qoldinit;
                nstep = 0;
                // first half of ode_determine_initdt; k[0] = f(u) is the FSAL derivative
                double v0[7], v1[7];
#pragma unroll
                for (int i = 0; i < 7; ++i) {
                    double sk = O.abstol + fabs(u[i]) * O.reltol;
                    v0[i] = u[i] / sk; v1[i] = KK(0, i) / sk;
                }
                double d0 = rms7(v0);
                d1 = rms7(v1);
                dt0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : (d0 / d1) / 100.0;
                dt0 = fmin(dt0, O.dtmax);
                if (dt0 < 10.0 * 2.220446049250313e-16) {
                    dt = 1e-6;
                    act = ACT_BEGIN_STEP;
                } else {
#pragma unroll
                    for (int i = 0; i < 7; ++i) tmp[i] = fma(dt0, KK(0, i), u[i]);
                    phase = PH_INITDT;
                    act = ACT_NONE;
                }
            }
        }
    }

    // ---- block reduction: warp shuffles, shared-memory atomics, then global atomics
    unsigned long long c6[8] = {cnt.n_acc, cnt.n_rej, cnt.n_rhs, cnt.n_alpha, cnt.n_harm, rays_ok, cnt.n_prune, cnt.n_askip};
    if (!writer) {  // LPR > 1: the other lanes of a group carry copies of its first lane's counts
#pragma unroll
        for (int q = 0; q < 8; ++q) c6[q] = 0ull;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        tot_dep += __shfl_down_sync(FULL, tot_dep, off);
        tot_w += __shfl_down_sync(FULL, tot_w, off);
#pragma unroll
        for (int q = 0; q < 8; ++q) c6[q] += __shfl_down_sync(FULL, c6[q], off);
    }
    if (lane == 0) {
        atomicAdd(&s_tot[0], tot_dep);
        atomicAdd(&s_tot[1], tot_w);
#pragma unroll
        for (int q = 0; q < 8; ++q) atomicAdd(&s_cnt[q], c6[q]);
    }
    __syncthreads();
    if (threadIdx.x < 2 && !XS) atomicAdd(&a.bins[n_psi + threadIdx.x], s_tot[threadIdx.x]);  // exact mode booked per ray
    if (threadIdx.x < 8) atomicAdd(&a.counters[threadIdx.x], s_cnt[threadIdx.x]);
    if constexpr (XS) {  // the bookings not yet flushed by xs_book
        unsigned long long nb = (unsigned)PKI(3);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) nb += __shfl_down_sync(FULL, nb, off);
        if (lane == 0 && nb) atomicAdd(reinterpret_cast<unsigned long long*>(a.xs - TORJ_XS_STAT), nb);
    }
#undef KK
#undef PK
#undef PKI
}

// Predicted life of every ray in segments, for the order of the hand-off rounds only (never for a result): a straight march
// from the plasma entry along the refracted direction, one point per segment end, with the real fields and the real
// absorption coefficient there; P <- P exp(-alpha s_step) until the ray would stop (psi_N > psi_stop or P < p_stop,
// reference src/solve.jl:174-176). Rays bend by millimetres over a segment: good to about one segment. ~100 RHS per ray
// against ~21 000 in the trace.
// The prediction is then made uniform over every aligned block of 32 consecutive rays (their maximum): a warp of the trace
// kernel draws 32 consecutive items, and they must be all real or all void — lanes that each skip ahead to their own next
// real item would end up with rays from all over the bundle, and neighbouring rays on neighbouring lanes is what keeps
// the stencil loads and the absorbing layer coherent (a random ray order costs 40 %, DESIGN.md §8).
__global__ void k_predict_life(DevTables T0, BundleDev B, SolverOpts O, PlasmaSetDev P, double harm_cost,
                               int* __restrict__ life, int* __restrict__ lmax) {
    exp_tab_init();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // blockDim.x is a multiple of 32: warp = ray block
    const long long n = B.n_rays;
    double cost = 1.0;
    if (i < n && B.status[i] == 0) {
        const DevTables T = ray_tables(T0, P, i);
        const double f = B.per_ray_fm ? B.freq[i] : B.freq[0];
        const int mode = B.per_ray_fm ? B.mode[i] : B.mode[0];
        const RayConst rc = make_ray_const(f, mode, O.te_min, O.max_harmonic, O.alpha_floor);
        double u[7], du[9];
        for (int q = 0; q < 7; ++q) u[q] = B.u0[(size_t)q * n + i];
        const double in = rsqrt(u[3] * u[3] + u[4] * u[4] + u[5] * u[5]);
        const double s_step = O.s_max / (double)O.n_segments;
        const double dx = u[3] * in * s_step, dy = u[4] * in * s_step, dz = u[5] * in * s_step;
        double P = 1.0;
        Counters c = {0, 0, 0, 0, 0, 0, 0};
        cost = 0.0;
        for (int k = 1; k <= O.n_segments; ++k) {
            u[0] += dx; u[1] += dy; u[2] += dz;
            const unsigned long long h0 = c.n_harm;
            rhs<true, true, true>(T, rc, u, du, c);
            cost += 1.0 + harm_cost * (double)(c.n_harm - h0);  // a segment inside the absorbing layer costs more trips' worth
            const double alpha = -du[6];  // u[6] = 1
            if (alpha > 0.0) P *= exp(-alpha * s_step);
            if (du[7] > O.psi_stop || P < O.p_stop || !(alpha == alpha)) break;
        }
    }
    int L = (int)ceil(cost);
    L = __reduce_max_sync(0xffffffffu, L);
    if (i < n) life[i] = L;
    if ((threadIdx.x & 31) == 0) atomicMax(lmax, L);
}

// dP_dV[j] = bins[j] / (V(psi_{j+1}) - V(psi_j)); last entry 0 (reference src/plasma.jl:103,141). dV: one row for all beams,
// or one row per beam (dV_per_beam: a plasma set, each beam normalised by its own plasma's volume)
__global__ void k_finalize(const double* bins, const double* dV, int n_psi, int n_beams, int dV_per_beam, double* profile) {
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= (long long)n_beams * (n_psi + 2)) return;
    int j = (int)(g % (n_psi + 2));
    if (dV_per_beam) dV += (g / (n_psi + 2)) * n_psi;
    if (j < n_psi - 1) profile[g] = bins[g] / dV[j];
    else if (j == n_psi - 1) profile[g] = 0.0;
    else profile[g] = bins[g];
}

// k_finalize of the exact-sum mode: bin g is the correctly rounded value of its words xs[g * 8 ..] (status words at xs[-2],
// xs[-1]); same layout rules. An invalid buffer (a refused booking, or more bookings than the words' headroom allows)
// yields NaN everywhere; the results call reports it.
__global__ void k_finalize_exact(const long long* xs, const double* dV, int n_psi, int n_beams, int dV_per_beam, double* profile) {
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nb = (long long)n_beams * (n_psi + 2);
    if (g >= nb) return;
    int j = (int)(g % (n_psi + 2));
    if (dV_per_beam) dV += (g / (n_psi + 2)) * n_psi;
    const long long* st = xs - TORJ_XS_STAT;
    const double v = torj_xs_valid(st[0], st[1]) ? torj_xs_to_double(xs + g * TORJ_XS_WORDS) : __longlong_as_double(0x7ff8000000000000ll);
    if (j < n_psi - 1) profile[g] = v / dV[j];
    else if (j == n_psi - 1) profile[g] = 0.0;
    else profile[g] = v;
}

// ------------------------------------------------------------------------------------------------
// probes
// ------------------------------------------------------------------------------------------------
// out[11][n]: psi, ne, Te, Bx, By, Bz, X, Y, N_par, Lambda, alpha
// model: 0 Albajar, 1 warm-plasma (needs 19 * blockDim doubles of dynamic shared memory; whole warps take part)
__global__ void k_probe(DevTables T, long long n, const double* x, const double* N, double f, int mode, double te_min,
                        int max_harmonic, double alpha_floor, int model, const double2* warm_tab, double* out) {
    exp_tab_init();
    extern __shared__ __align__(16) double smem[];
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = i < n;
    if (!active) i = n - 1;
    RayConst rc = make_ray_const(f, mode, te_min, max_harmonic, alpha_floor);
    double u[7] = {x[i], x[n + i], x[2 * n + i], N[i], N[n + i], N[2 * n + i], 1.0}, du[7];
    Counters c = {0, 0, 0, 0, 0, 0, 0};
    PointVals pv;
    if (model == 1) {
        AlphaIn ain;
        bool safe;
        rhs<false, false, false>(T, rc, u, du, c, &pv, false, nullptr, &ain);
        du[6] = -u[6] * warm_alpha_warp<false>(warm_tab, rc, ain, active, smem + threadIdx.x, blockDim.x, c, safe);
    } else {
        rhs<true, false, true>(T, rc, u, du, c, &pv);
    }
    if (!active) return;
    double Babs = pv.Y / rc.cY;
    out[i] = psi_at(T, u);
    out[n + i] = pv.X / rc.cX;
    out[2 * n + i] = pv.Te;
    out[3 * n + i] = pv.b[0] * Babs; out[4 * n + i] = pv.b[1] * Babs; out[5 * n + i] = pv.b[2] * Babs;
    out[6 * n + i] = pv.X; out[7 * n + i] = pv.Y; out[8 * n + i] = pv.N_par; out[9 * n + i] = pv.Lambda;
    out[10 * n + i] = -du[6];
}

__global__ void k_rhs(DevTables T, long long n, const double* u, double f, int mode, double te_min, int max_harmonic,
                      double alpha_floor, int model, const double2* warm_tab, double* du) {
    exp_tab_init();
    extern __shared__ __align__(16) double smem[];
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = i < n;
    if (!active) i = n - 1;
    RayConst rc = make_ray_const(f, mode, te_min, max_harmonic, alpha_floor);
    double uu[7], dd[7];
    for (int q = 0; q < 7; ++q) uu[q] = u[(size_t)q * n + i];
    Counters c = {0, 0, 0, 0, 0, 0, 0};
    if (model == 1) {
        AlphaIn ain;
        bool safe;
        rhs<false, false, false>(T, rc, uu, dd, c, nullptr, false, nullptr, &ain);
        dd[6] = -uu[6] * warm_alpha_warp<false>(warm_tab, rc, ain, active, smem + threadIdx.x, blockDim.x, c, safe);
    } else {
        rhs<true, false, true>(T, rc, uu, dd, c);
    }
    if (!active) return;
    for (int q = 0; q < 7; ++q) du[(size_t)q * n + i] = dd[q];
}

// α(omega, X, Y, N_r, theta, te, v_g_perp, imod) of reference src/general_absorption.jl:1328-1337 at n points (parity
// probe). in[7][n]: omega, X, Y, N_r, theta, te, v_g_perp; out[5][n]: N_warm, alpha, lrm, ierr, iterations.
// One point per lane; the warp does the quadratures one after the other, the owner finishes its own.
__global__ void k_warm_alpha(long long n, const double* in, int imod, const double2* warm_tab, double* out) {
    exp_tab_init();
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = i < n;
    if (!active) i = n - 1;
    const unsigned lane = threadIdx.x & 31u;
    const double omega = in[i], X = in[n + i], Y = in[2 * n + i], N_r = in[3 * n + i], theta = in[4 * n + i], te = in[5 * n + i],
                 vg = in[6 * n + i];
    RayConst rc = make_ray_const(omega / (2.0 * M_PI), imod, 0.0, 3, 0.0);
    rc.w_over_c = omega / TORJ_C;
    AlphaIn ain;
    ain.X = X; ain.Y = Y; ain.N2 = N_r * N_r; ain.Np = N_r * cos(theta); ain.lnTe = log(te); ain.inorm = vg;
    rc.ln_te_min = -1e300;
    WarmPrep wp;
    wp.yg = 0.5; wp.anpl = 0.0; wp.amu = 100.0; wp.anprc = 1.0; wp.sinth = 1.0; wp.lrm = 1;
    double alpha = 0.0, N_warm = 0.0;
    int ierr = 0, iters = 0;
    bool gated, safe;
    bool needq = active && warm_prepare(rc, ain, wp, alpha, gated, safe);
    if (active && !needq && wp.lrm < 1) ierr = 98;
    const int llm = wp.lrm < 3 ? wp.lrm : 3;
    unsigned m = __ballot_sync(0xffffffffu, needq);
    while (m) {
        const int src = __ffs(m) - 1;
        m &= m - 1;
        const double yg = __shfl_sync(0xffffffffu, wp.yg, src), anpl = __shfl_sync(0xffffffffu, wp.anpl, src);
        const double amu = __shfl_sync(0xffffffffu, wp.amu, src);
        const int l3 = __shfl_sync(0xffffffffu, llm, src);
        double H[TORJ_WARM_H];
        warm_hermitian_warp(warm_tab, yg, anpl, amu, l3, H);
        if ((int)lane == src) alpha = warm_alpha_finish(rc, ain, wp, H, &N_warm, &ierr, &iters);
    }
    if (!active) return;
    out[i] = N_warm; out[n + i] = alpha; out[2 * n + i] = (double)wp.lrm; out[3 * n + i] = (double)ierr;
    out[4 * n + i] = (double)iters;
}

// FP64 peak: 8 independent DFMA chains per thread, register resident
__global__ void k_dfma(int iters, double* out) {
    double a0 = 1.0 + threadIdx.x * 1e-9, a1 = a0 + 1e-3, a2 = a0 + 2e-3, a3 = a0 + 3e-3;
    double a4 = a0 + 4e-3, a5 = a0 + 5e-3, a6 = a0 + 6e-3, a7 = a0 + 7e-3;
    const double m = 0.999999, c = 1e-7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
            a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
        }
    }
    double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 12345.6789) out[0] = s;
}

// ------------------------------------------------------------------------------------------------
// Plasma construction on the device (reference src/plasma.jl:16-58): prefilter and table packing
// ------------------------------------------------------------------------------------------------
// One thread per line: natural-end cubic B-spline prefilter (rows 1/6, 2/3, 1/6; c[1] = y[0], c[n] = y[n-1]).
// cp[k] are the data-independent Thomas pivots for this n. in/out are addressed with (line, element) strides so the
// same kernel does the R pass (lines = Z rows) and the Z pass (lines = R columns of the intermediate array).
__global__ void k_prefilter_lines(const double* __restrict__ in, double* __restrict__ out, int n, int n_lines,
                                  long long in_ls, long long in_es, long long out_ls, long long out_es,
                                  const double* __restrict__ cp) {
    int line = blockIdx.x * blockDim.x + threadIdx.x;
    if (line >= n_lines) return;
    const double* y = in + (long long)line * in_ls;
    double* c = out + (long long)line * out_ls;
    const double a = 1.0 / 6.0, b = 2.0 / 3.0;
    const double s_first = y[0], s_last = y[(long long)(n - 1) * in_es];
    const int m = n - 2;
    // forward sweep; dp[k] is parked in c[k+2] (the slot of sol[k+1])
    if (m >= 1) {
        double prev = (y[in_es] - a * s_first - (m == 1 ? a * s_last : 0.0)) / b;
        c[2 * out_es] = prev;
        for (int k = 1; k < m; ++k) {
            double r = y[(long long)(k + 1) * in_es];
            if (k == m - 1) r -= a * s_last;
            prev = (r - a * prev) / (b - a * cp[k - 1]);
            c[(long long)(k + 2) * out_es] = prev;
        }
        // back substitution: sol[m] = dp[m-1]; sol[k+1] = dp[k] - cp[k] sol[k+2]
        double nxt = c[(long long)(m + 1) * out_es];
        for (int k = m - 2; k >= 0; --k) {
            nxt = c[(long long)(k + 2) * out_es] - cp[k] * nxt;
            c[(long long)(k + 2) * out_es] = nxt;
        }
    }
    c[out_es] = s_first;
    c[(long long)n * out_es] = s_last;
    const double s1 = (n > 2) ? c[2 * out_es] : s_last;
    const double sm2 = (n > 2) ? c[(long long)(n - 1) * out_es] : s_first;
    c[0] = 2.0 * s_first - s1;
    c[(long long)(n + 1) * out_es] = 2.0 * s_last - sm2;
}

// ln(profile) on the grid: 1-D cubic B-spline (uniform psi range, Line extrapolation) evaluated at every psi_N node
// (reference src/plasma.jl:19-20)
__global__ void k_profile_to_grid(const double* __restrict__ psi_nodes, long long n_nodes, const double* __restrict__ c1,
                                  int n, double x0, double h, double* __restrict__ out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    double x = psi_nodes[i];
    double xl = x0 + h * (n - 1);
    double xc = fmin(fmax(x, x0), xl);
    double u = (xc - x0) / h + 1.0;
    int k = min(max((int)floor(u), 1), n - 1);
    double d = u - (double)k, e = 1.0 - d;
    double w0 = e * e * e / 6.0, w1 = 2.0 / 3.0 - d * d + d * d * d / 2.0, w2 = 2.0 / 3.0 - e * e + e * e * e / 2.0, w3 = d * d * d / 6.0;
    double g0 = -e * e / 2.0 / h, g1 = (-2.0 * d + 1.5 * d * d) / h, g2 = (2.0 * e - 1.5 * e * e) / h, g3 = d * d / 2.0 / h;
    const double* cc = c1 + (k - 1);
    double v = w0 * cc[0] + w1 * cc[1] + w2 * cc[2] + w3 * cc[3];
    double dv = g0 * cc[0] + g1 * cc[1] + g2 * cc[2] + g3 * cc[3];
    out[i] = v + (x - xc) * dv;
}

// six coefficient tables -> the interleaved node layout of DevTables
__global__ void k_pack_tables(const double* psi, const double* lnne, const double* lnTe, const double* BR, const double* BZ,
                              const double* Bp, long long nodes, double2* A) {
    long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nodes) return;
    A[3 * k] = make_double2(BR[k], BZ[k]);
    A[3 * k + 1] = make_double2(Bp[k], lnne[k]);
    A[3 * k + 2] = make_double2(lnTe[k], psi[k]);
}

// ------------------------------------------------------------------------------------------------
// launch_peripheral_rays for many launchers at once (reference src/launch.jl:24-132, quirks included): one thread per ray
// ------------------------------------------------------------------------------------------------
struct LaunchArgs {
    int n_launchers, n_rings, n_per;   // rays per launcher (identical for all: N_theta depends on the rings only)
    const double* x0;                  // [3][nl]
    const double* N0;                  // [3][nl]
    const double* w;                   // [nl] beam width
    const double* inv_Rc;              // [nl] inverse curvature radius (inf = paraxial)
    const double* f;                   // [nl]
    const int* mode;                   // [nl]
    const double* r_unit;              // [n_rings] Gauss-Hermite radii / (w/sqrt2)
    const double* rw_unit;             // [n_rings] Gauss-Hermite weights / (w/sqrt2)
    const int* ring_start;             // [n_rings+1] prefix sum of N_theta
    double wsum_unit;                  // sum_i r_i rw_i 2 pi in unit widths (weights of one launcher sum to wsum_unit w^2/2)
    int normalize;
    // outputs: bundle arrays over n = nl * n_per rays
    double *pos, *dir, *weight, *freq;
    int *mode_out, *beam;
};

__global__ void k_launch_rays(LaunchArgs A) {
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long n = (long long)A.n_launchers * A.n_per;
    if (g >= n) return;
    const int L = (int)(g / A.n_per), k = (int)(g % A.n_per);
    int ring = 0;
    while (ring + 1 < A.n_rings && k >= A.ring_start[ring + 1]) ++ring;
    const int j = k - A.ring_start[ring], nth = A.ring_start[ring + 1] - A.ring_start[ring];
    const int nl = A.n_launchers;
    const double x0[3] = {A.x0[L], A.x0[nl + L], A.x0[2 * nl + L]};
    double n0[3] = {A.N0[L], A.N0[nl + L], A.N0[2 * nl + L]};
    const double nn = sqrt(n0[0] * n0[0] + n0[1] * n0[1] + n0[2] * n0[2]);
    for (int c = 0; c < 3; ++c) n0[c] /= nn;
    const double w = A.w[L], irc = A.inv_Rc[L], f = A.f[L];
    const bool curved = isfinite(irc);
    double w0 = w, xw[3] = {0, 0, 0};
    if (curved) {  // src/launch.jl:34-47
        const double Rc = 1.0 / irc, lam = TORJ_C / f;
        const double den = lam * lam * Rc * Rc + M_PI * M_PI * w * w * w * w;
        w0 = (lam * fabs(Rc) * w) / sqrt(den);
        const double zw = M_PI * M_PI * Rc * w * w * w * w / den;
        for (int c = 0; c < 3; ++c) xw[c] = x0[c] - n0[c] * zw;
    }
    double ec[3] = {1.0, 0.0, -n0[0] / n0[2]};                       // src/launch.jl:54-57
    double eu[3] = {-n0[0] * n0[1] / n0[2], n0[2] - n0[0], -n0[1]};  // src/launch.jl:61-64
    const double nc = sqrt(ec[0] * ec[0] + ec[1] * ec[1] + ec[2] * ec[2]), nu = sqrt(eu[0] * eu[0] + eu[1] * eu[1] + eu[2] * eu[2]);
    for (int c = 0; c < 3; ++c) { ec[c] /= nc; eu[c] /= nu; }
    const double sc = w / sqrt(2.0);
    const double r = A.r_unit[ring] * sc, rw = A.rw_unit[ring] * sc;
    const double th = 2.0 * M_PI * (double)j / (double)nth;
    const double chi = r * cos(th), ups = r * sin(th);
    double p[3], d[3];
    for (int c = 0; c < 3; ++c) p[c] = chi * ec[c] + ups * eu[c] + x0[c];
    if (curved) {  // src/launch.jl:102-113
        const double sg = irc > 0.0 ? 1.0 : (irc < 0.0 ? -1.0 : 0.0);
        for (int c = 0; c < 3; ++c) d[c] = w0 / w * (chi * ec[c] + ups * eu[c]) * sg + xw[c];
        if (irc < 0.0) { for (int c = 0; c < 3; ++c) d[c] -= p[c]; }
        else { for (int c = 0; c < 3; ++c) d[c] = -d[c] + p[c]; }
        const double dn = sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
        for (int c = 0; c < 3; ++c) d[c] /= dn;
    } else {
        for (int c = 0; c < 3; ++c) d[c] = n0[c];
    }
    double wt = r * rw * (2.0 * M_PI / (double)nth);                 // src/launch.jl:120
    if (A.normalize) wt /= (A.wsum_unit * sc * sc);                  // src/launch.jl:125-126
    else wt *= 2.0 / (w * w * M_PI);
    for (int c = 0; c < 3; ++c) { A.pos[c * n + g] = p[c]; A.dir[c * n + g] = d[c]; }
    A.weight[g] = wt;
    A.freq[g] = f;
    A.mode_out[g] = A.mode[L];
    A.beam[g] = L;
}

// dependent-issue latency of DFMA: one warp, one chain, cycles from clock64()
__global__ void k_dfma_latency(int iters, double seed, double* out, long long* cycles) {
    double a = seed;
    const double m = 0.999999, c = 1e-7;
    long long t0 = clock64();
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int r = 0; r < 16; ++r) a = fma(a, m, c);
    }
    long long t1 = clock64();
    if (threadIdx.x == 0) { cycles[0] = t1 - t0; out[0] = a; }
}

// the kernel's own elementary functions on n arguments (accuracy tests): out[0..3][n] = rcp, rsqrt, sqrt, exp
__global__ void k_math_probe(long long n, const double* x, double* out) {
    exp_tab_init();
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double v = x[i];
    out[i] = rcp_fast(v);
    out[n + i] = rsqrt_fast(v);
    out[2 * n + i] = sqrt_fast(v);
    out[3 * n + i] = exp_fast(v);
}

}  // namespace torj
