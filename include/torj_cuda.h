/*
 * libtorj_cuda.so — C ABI of the B200-native TorJ ray-tracing hot path.
 *
 * The reference (ProjectTorreyPines/TorJ.jl) has no FFI: its seam is the Julia function level.  Each entry
 * point below names the reference interface it replaces (file:line into the reference repository); the Julia
 * `ccall` shim a maintainer would add is shown in INTEGRATION.md and mirrored, name for name, by the Python
 * host package torj_jl_b200 (Julia is not installed in this environment).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on a library / CUDA failure; torj_last_error() has the text.
 *   - per-ray physics failures never abort a batch: they are reported in status[] (TORJ_RAY_*).
 *   - the caller owns every host buffer; nothing is retained past the call that received it.
 *   - 2-D tables are "R fastest" (a Julia Matrix[nR+2, nZ+2] passed as is); ray positions/directions are
 *     component-major [3][n] (a Julia Matrix[n,3] passed as is, reference src/launch.jl:84-85).
 *   - all arithmetic is FP64.  There is no CPU fallback: without a CUDA device torj_ctx_create fails.
 *   - calls are blocking unless stated otherwise; a torj_ctx (and the objects created on it) must not be used from two
 *     threads at once — use one context per host thread / per GPU.
 */
#ifndef TORJ_CUDA_H
#define TORJ_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TORJ_ABI_VERSION 3

typedef struct torj_ctx torj_ctx;       /* one per (process, device): stream, quadrature nodes, launch counter */
typedef struct torj_plasma torj_plasma; /* device-resident equilibrium tables (reference struct Plasma, src/plasma.jl:2-14) */
typedef struct torj_bundle torj_bundle; /* device-resident ray bundle, its state and results */

/* per-ray status */
enum {
    TORJ_RAY_OK = 0,
    TORJ_RAY_CUTOFF_AT_ENTRY = 1, /* reference src/solve.jl:55-59 returns (false, nothing) */
    TORJ_RAY_INIT_FAILED = 2,     /* bisection bracket (src/solve.jl:29), asserts src/solve.jl:32,138,141, Newton failure */
    TORJ_RAY_LEFT_GRID = 3,       /* informational, like 6: the ray ended outside the (R,Z) grid box, where every field is the
                                     splines' linear extrapolation (Interpolations.jl `Line()`, src/plasma.jl:36-41); it was
                                     traced and deposited to the end exactly as the reference does */
    TORJ_RAY_MAX_STEPS = 4,
    TORJ_RAY_NAN = 5,
    TORJ_RAY_TRAJ_TRUNCATED = 6   /* trajectory window full; tracing and deposition still completed */
};

/* Solver constants hard-coded in the reference, carried here with the reference values as defaults. */
typedef struct torj_options {
    int32_t scheme;                /* 0 = Tsit5: what `solve(prob)` runs, the `OwrenZen3()` at src/solve.jl:156 being
                                      passed as the parameter object; 1 = OwrenZen3 (the scheme the source names) */
    int32_t n_segments;            /* 100   src/solve.jl:145; >= 1. The segment hand-off (schedule 2 / 3) takes at most 16000:
                                      above that, schedule 0 traces whole rays and schedules 2 and 3 are refused */
    double dtmax;                  /* 1e-4  src/solve.jl:157 */
    double abstol;                 /* 1e-6  src/solve.jl:157 */
    double reltol;                 /* 1e-6  src/solve.jl:157 */
    double psi_stop;               /* 1.0   src/solve.jl:174 */
    double p_stop;                 /* 1e-6  src/solve.jl:176 */
    double te_min;                 /* 20 eV src/absorption.jl:194 */
    int32_t max_harmonic;          /* 3     src/absorption.jl:199; 1 = no absorption, 4..16 add the harmonics the reference
                                      leaves out with the same integral (src/absorption.jl:170-189), Bessel functions
                                      from libm jn() */
    int32_t max_steps_per_segment; /* safety cap, 100000 */
    double alpha_floor;            /* 1e-14 m^-1: a harmonic integral (src/absorption.jl:170-189) is skipped when a rigorous
                                      upper bound of its contribution to alpha is below this (|J_n|<=1, sum of weights 2,
                                      max exponent on the resonance curve); optical-depth error <= 2*alpha_floor*path.
                                      0 = evaluate every integral exactly as the reference does */
    int32_t schedule;              /* how rays are mapped to GPU lanes; results do not depend on it.
                                      0 = automatic; 1 = a lane keeps a ray from entry to retirement;
                                      2 = segment hand-off: a ray may change lanes between two of its n_segments
                                      segments, so all rays advance together: no partly filled last wave, and the lanes
                                      of a warp stay in step (automatic picks this when the bundle exceeds the resident
                                      lanes, 37 888 on a B200). With the Albajar model the rounds of the hand-off are
                                      life-ordered: a pilot march (straight line, real fields and alpha, one point per
                                      segment) predicts every ray's life and the long-lived rays start first, so that all
                                      rays end together instead of the longest ones finishing alone;
                                      3 = plain segment hand-off: every ray starts in round 0.
                                      The hand-off needs n_segments <= 16000 (see n_segments) */
    int32_t absorption_model;      /* 0 = Albajar (reference src/absorption.jl:191-235, what the reference's gradΛ! calls);
                                      1 = warm-plasma damping: alpha = α(ω, X, Y, |N|, acos(N∥/|N|), Te, v_g_perp, mode)[2] of
                                      reference src/general_absorption.jl:1328-1337 (iwarm = 3, Larmor order lrm <= 5) in the
                                      place of α_approx. That file is dead code in the reference (never include()d), so the
                                      wiring is BUILD-DEFINED: v_g_perp = 1/|dΛ/dN| (SURVEY.md §8(a) a21), same Te gate
                                      (te_min); the debug assertion at :314-316 is dropped (it calls an un-imported function).
                                      With alpha_floor > 0 the 501-node quadrature is skipped where the anti-Hermitian part is
                                      below the floor by construction (torj_warm.cuh); 0 evaluates it everywhere */
    int32_t lanes_per_ray;         /* 0 = automatic; 1 = one GPU thread per ray; 2 / 4 / 8 / 32 = a group of lanes / a warp per ray
                                      (the nodes of the harmonic integrals / of the warm quadrature are split over the lanes):
                                      for bundles below the resident lanes, where the time is one ray's latency, and for the
                                      warm model (1 or 32 only). Results agree to rounding (summation order) */
    int32_t reserved_;             /* keeps the struct size a multiple of 8; must be 0 */
} torj_options;

typedef struct torj_counters {
    int64_t n_acc;   /* accepted integrator steps (the "ray-steps" of the headline metric) */
    int64_t n_rej;   /* rejected steps */
    int64_t n_rhs;   /* evaluations of gradΛ! (src/solve.jl:85-95) */
    int64_t n_alpha; /* abs_Albajar_fast calls past the Te gate (src/absorption.jl:194); warm model: α calls past the gate */
    int64_t n_harm;  /* harmonic integrals evaluated (src/absorption.jl:217); warm model: resonance indices n integrated over
                        the 501 nodes (2 llm + 1 per α call, src/general_absorption.jl:669-710) */
    int64_t n_rays_ok;
    int64_t n_harm_pruned; /* harmonic integrals skipped by the alpha_floor bound */
    int64_t n_alpha_skipped; /* inner Runge-Kutta stages that took alpha = 0 on the 1e10-margin rule (alpha_floor > 0 only) */
} torj_counters;

typedef struct torj_grid {
    int32_t nR, nZ;        /* data points per axis; coefficient tables are (nR+2) x (nZ+2) */
    double R_first, R_last;
    double Z_first, Z_last;
} torj_grid;

void torj_options_default(torj_options* o);
const char* torj_last_error(void);
int torj_abi_version(void);

/* --- context ---------------------------------------------------------------------------------------------- */
/* cuda_stream: a cudaStream_t to launch on (e.g. the caller's current stream) or NULL for a private stream. */
int torj_ctx_create(int device, void* cuda_stream, torj_ctx** out);
void torj_ctx_destroy(torj_ctx* ctx);
int torj_ctx_sync(torj_ctx* ctx);
/* kernels launched by this library on ctx since creation */
int64_t torj_ctx_launch_count(const torj_ctx* ctx);
/* device duration (CUDA events on the context stream) of the most recent trace-kernel launch; synchronises on it */
int torj_ctx_last_trace_ms(torj_ctx* ctx, double* ms);
/* Exact deposition sums, for every later torj_trace(_plasmas) and torj_bundle_trace(_plasmas) on bundles of ctx.
 * on = 0 (default): each booking into a profile bin is a floating-point atomicAdd, whose order changes from run to run, so
 * dP_dV and deposited_power may differ in their last bits (the per-ray results never do).
 * on = 1: each booking (w dP, w P_deposited_ray, w; rounded once to a double, as with 0) is rounded to 2^-160 and summed
 * without error in a fixed-point integer accumulator; the profile is the correctly rounded value of that exact sum over
 * dV. It is bit-identical under any schedule, ray order, sharding and device count, at a fixed lanes_per_ray (the per-ray
 * arithmetic depends on it). Weights must satisfy |w| <= 2^40 (else the trace is refused); a booking of |w dP| >= 2^64 or
 * NaN, or more than 2^34 bookings in one trace, makes torj_bundle_results fail (the device profile is then NaN).
 * Other values of `on` are refused. The mode is state of the context and persists until the next call: a caller that
 * shares a context with code that may have turned it on (the Python package's per-device context, for example) sets it
 * explicitly before tracing, as every Python entry point does. */
int torj_ctx_set_exact_sum(torj_ctx* ctx, int32_t on);

/* abs_Al_init(N) — reference src/absorption.jl:1-7: Gauss-Legendre nodes/weights on [-1,1] (n <= 64), ascending and
 * symmetric (t[k] = -t[n-1-k], w[k] = w[n-1-k], as gausslegendre(N) returns them; anything else is refused: the kernel
 * evaluates the Bessel functions of a node pair once).
 * Like the reference's module globals (src/constants.jl:7-8) the table is shared: ONE per device. A context created on
 * a device whose table is already set inherits it; setting different nodes synchronises the whole device first and
 * changes them for every context on that device. */
int torj_abs_init(torj_ctx* ctx, int32_t n, const double* nodes, const double* weights);

/* α(omega, X, Y, N_r, theta, te, v_g_perp, imod) — reference src/general_absorption.jl:1328-1337, at n points (arrays
 * of length n): N_warm = Re(N_perp)/sin(theta) and alpha = 2 Im(N_perp^2) omega/c v_g_perp; lrm = min(5, larmornumber),
 * ierr = 99 (negative solution, :1229-1232) / 98 (lrm < 1: the reference throws). set_extv! (:8-13) needs no call. */
int torj_warm_alpha(torj_ctx* ctx, int64_t n, const double* omega, const double* X, const double* Y, const double* N_r,
                    const double* theta, const double* te, const double* v_g_perp, int32_t imod, double* N_warm,
                    double* alpha, int32_t* lrm, int32_t* ierr);

/* --- equilibrium ------------------------------------------------------------------------------------------- */
/* Host helper: cubic B-spline prefilter of cubic_spline_interpolation((r,z), data) — reference src/plasma.jl:36-41
 * (Interpolations.jl BSpline(Cubic(Line(OnGrid())))).  data: nR x nZ, R fastest; coef out: (nR+2) x (nZ+2). */
int torj_bspline_prefilter_2d(int32_t nR, int32_t nZ, const double* data, double* coef);
int torj_bspline_prefilter_1d(int32_t n, const double* data, double* coef);

/* Uploads what the Julia shim extracts from a `Plasma` (src/plasma.jl:2-14): six coefficient tables, the 1-D
 * V(psi_N) spline (n_vol data points -> n_vol+2 coefficients on the uniform range vol_psi0 + k*vol_dpsi) and
 * psi_prof_max. */
int torj_plasma_create(torj_ctx* ctx, const torj_grid* grid, const double* coef_psi, const double* coef_lnne,
                       const double* coef_lnTe, const double* coef_BR, const double* coef_BZ, const double* coef_Bphi,
                       const double* vol_coef, int32_t n_vol, double vol_psi0, double vol_dpsi, double psi_prof_max,
                       torj_plasma** out);
/* The whole `Plasma(R, Z, psiN, psi_prof, ne, Te, BR, BZ, Bphi, psi1d, V1d)` constructor (reference src/plasma.jl:30-58
 * incl. make_2d_prof_spline :16-22) from the raw arrays: 1-D resampling/log/prefilter on the host, the six 2-D
 * prefilters and the table packing on the device. 2-D arrays are nR x nZ, R fastest. Needs nothing of
 * Interpolations.jl's internals on the Julia side. */
int torj_plasma_create_from_data(torj_ctx* ctx, const torj_grid* grid, const double* psi_norm, const double* psi_prof,
                                 const double* ne_prof, const double* Te_prof, int32_t n_prof, const double* BR,
                                 const double* BZ, const double* Bphi, const double* psi_1d, const double* vol_1d,
                                 int32_t n_1d, torj_plasma** out);
void torj_plasma_destroy(torj_plasma* p);

/* Field probes at Cartesian points x[3][n] (tests of reference src/plasma.jl:61-89 / src/dispersion.jl:7-15,
 * cf. reference test/tests/test_trajectory.jl). out[11][n]: psi, ne, Te, Bx, By, Bz, X, Y, N_par, Lambda, alpha */
int torj_probe(torj_ctx* ctx, const torj_plasma* p, const torj_options* opt, int64_t n, const double* x, const double* N,
               double freq_hz, int32_t mode, double* out);
/* du = gradΛ!(u) for u[7][n] (reference src/solve.jl:85-95) */
int torj_rhs(torj_ctx* ctx, const torj_plasma* p, const torj_options* opt, int64_t n, const double* u, double freq_hz,
             int32_t mode, double* du);

/* --- resident bundle API (bench "value": inputs already in HBM) --------------------------------------------- */
/* freq_hz/mode: per ray when per_ray_fm != 0, else length 1. */
int torj_bundle_create(torj_ctx* ctx, int64_t n_rays, const double* pos, const double* dir, const double* weight,
                       const double* freq_hz, const int32_t* mode, int32_t per_ray_fm, torj_bundle** out);
/* launch_peripheral_rays (reference src/launch.jl:24-132) for n_launchers beams at once, on the device: launcher
 * parameters x0/N0 [3][nl], w, inv_Rc, f, mode [nl]; common N_rings / min_azimuthal_points / normalize_weight_sum;
 * gh_nodes/gh_weights = Gauss-Hermite rule of order 2*N_rings+2 (ascending nodes). Ray k of launcher L is ray
 * L*n_per+k; the bundle carries per-ray frequency/mode and one deposition profile per launcher (n_beams = nl). */
int torj_bundle_create_from_launchers(torj_ctx* ctx, int32_t n_launchers, const double* x0, const double* N0, const double* w,
                                      const double* inv_Rc, const double* f, const int32_t* mode, int32_t N_rings,
                                      int32_t min_azimuthal_points, int32_t normalize_weight_sum, const double* gh_nodes,
                                      const double* gh_weights, torj_bundle** out, int64_t* n_rays_out);
/* launch arrays of a bundle back to the host: pos/dir [3][n], weight [n]; any pointer may be NULL */
int torj_bundle_rays(torj_bundle* b, double* pos, double* dir, double* weight);
void torj_bundle_destroy(torj_bundle* b);
/* Trajectories are kept for rays [traj_first, traj_first+traj_count), up to traj_max_pts points each. */
int torj_bundle_set_window(torj_bundle* b, int64_t traj_first, int64_t traj_count, int32_t traj_max_pts);
/* Scans: rays of several beams (launchers, frequencies) in one bundle, one deposition profile per beam — the batched
 * form of a host loop over make_beam (reference src/solve.jl:209-242). beam_id[n] in [0, n_beams); n_beams = 1 or a
 * NULL beam_id restores the single profile. With n_beams > 1 dP_dV is [n_beams][n_psi], deposited_power [n_beams] and
 * the device profile [n_beams][n_psi+2]. */
int torj_bundle_set_beams(torj_bundle* b, int32_t n_beams, const int32_t* beam_id);
/* Enqueues ray init + trace + profile finalize on the context stream; returns without synchronising.
 * Replaces the parallel region and reduction of make_beam (reference src/solve.jl:219-240) and, per ray,
 * make_ray (src/solve.jl:135-181) incl. power_deposition_profile (src/plasma.jl:91-151). */
int torj_bundle_trace(torj_bundle* b, const torj_plasma* p, const torj_options* opt, double s_max, int32_t n_psi,
                      const double* psi_edges);
/* Beams of one bundle traced through several equilibria on one (R,Z) grid: beam b through plasmas[beam_plasma[b]]; its
 * profile row is normalised by that plasma's V(psi). n_beams from torj_bundle_set_beams. The plasmas must have bitwise
 * equal grids (torj_grid of the same values) and live on the bundle's device. Refused (non-zero, torj_last_error):
 * n_plasmas < 1, a NULL plasma, a plasma on another device, two different grids, and with n_plasmas > 1 a NULL or
 * out-of-range beam_plasma or a single beam (a profile row belongs to one plasma). n_plasmas = 1 is torj_bundle_trace
 * (beam_plasma unused). Like torj_bundle_trace it returns without synchronising: the plasmas must outlive the results
 * read. Keep each beam's rays contiguous: a warp whose rays share a plasma shares its table rows. */
int torj_bundle_trace_plasmas(torj_bundle* b, int32_t n_plasmas, const torj_plasma* const* plasmas,
                              const int32_t* beam_plasma /* [n_beams] */, const torj_options* opt, double s_max,
                              int32_t n_psi, const double* psi_edges);
/* Device pointer to n_beams x (n_psi+2) doubles: dP_dV[n_psi], deposited_power, sum of weights per beam — for a caller-side
 * NCCL all-reduce (sum) across GPUs; valid after torj_bundle_trace, ordered on the context stream. With exact sums each
 * device's profile is exact, but a double all-reduce of several devices' profiles is not. */
void* torj_bundle_device_profile(torj_bundle* b);
/* Synchronises and copies results to the host (any pointer may be NULL); fails after an exact-sum trace whose accumulator
 * overflowed or refused a booking (torj_ctx_set_exact_sum). For a ray that failed initialisation
 * (status 1 or 2) P_final and P_deposited_ray are 0 and n_points is minus the failing check's number (-1 no grid entry,
 * -2 no psi bracket, -3/-4 asserts of src/solve.jl:32,138, -5..-7 Newton, -8 assert :141, -9 cut-off :55-59). */
int torj_bundle_results(torj_bundle* b, double* dP_dV, double* deposited_power, double* P_final,
                        double* P_deposited_ray, int32_t* n_points, int32_t* status, torj_counters* counters);
/* Trajectory window to the host: arrays [traj_count][traj_max_pts] (s, P, dP_ds), [traj_count][3][traj_max_pts]
 * (xyz) and the per-ray profile [traj_count][n_psi]; any pointer may be NULL. */
int torj_bundle_trajectories(torj_bundle* b, double* s, double* xyz, double* P, double* dP_ds, double* dP_dV_ray);
/* Derived ray coordinates (the reference integrates Cartesian u = [x, N, P], src/solve.jl:144; these are the cylindrical
 * position and the optical depth of the same state): R = hypot(x, y), phi = atan2(y, x), tau = -ln P.
 * torj_bundle_final_state: state at retirement of every ray, u_final [7][n] and/or R, phi, tau [n]; rays that failed
 * initialisation get NaN. torj_bundle_trajectories_cyl: the same per sample of the trajectory window,
 * [traj_count][traj_max_pts] each. Any pointer may be NULL. */
int torj_bundle_final_state(torj_bundle* b, double* u_final, double* R, double* phi, double* tau);
int torj_bundle_trajectories_cyl(torj_bundle* b, double* R, double* phi, double* tau);

/* --- one-shot host-buffer call: what the Julia make_ray / make_beam shims ccall ------------------------------ */
int torj_trace(torj_ctx* ctx, const torj_plasma* p, const torj_options* opt, int64_t n_rays, const double* pos,
               const double* dir, const double* weight, const double* freq_hz, const int32_t* mode, int32_t per_ray_fm,
               double s_max, int32_t n_psi, const double* psi_edges, int32_t n_beams, const int32_t* beam_id /* or NULL */,
               /* out */ double* dP_dV, double* deposited_power, double* P_final, double* P_deposited_ray,
               int32_t* n_points, int32_t* status,
               /* optional trajectories */ int64_t traj_first, int64_t traj_count, int32_t traj_max_pts, double* traj_s,
               double* traj_xyz, double* traj_P, double* traj_dP_ds, double* traj_dP_dV_ray, torj_counters* counters);
/* torj_trace through a plasma set (torj_bundle_trace_plasmas): beam b of beam_id through plasmas[beam_plasma[b]]; the
 * trajectory window's dP_dV_ray rows use the volume of each ray's plasma. Same refusals; blocking like torj_trace. */
int torj_trace_plasmas(torj_ctx* ctx, int32_t n_plasmas, const torj_plasma* const* plasmas, const int32_t* beam_plasma,
                       const torj_options* opt, int64_t n_rays, const double* pos, const double* dir, const double* weight,
                       const double* freq_hz, const int32_t* mode, int32_t per_ray_fm, double s_max, int32_t n_psi,
                       const double* psi_edges, int32_t n_beams, const int32_t* beam_id, double* dP_dV, double* deposited_power,
                       double* P_final, double* P_deposited_ray, int32_t* n_points, int32_t* status, int64_t traj_first,
                       int64_t traj_count, int32_t traj_max_pts, double* traj_s, double* traj_xyz, double* traj_P,
                       double* traj_dP_ds, double* traj_dP_dV_ray, torj_counters* counters);

/* --- single-process multi-GPU front end ----------------------------------------------------------------------- */
/* For a host that is ONE process on a multi-GPU box (a Julia session calling make_beam): the same call as torj_trace,
 * sharded over the devices (one persistent worker thread, one context and pinned staging buffers per device, tables
 * replicated). The weighted sum of reference src/solve.jl:233-240 across devices is ONE ncclAllReduce(sum, double,
 * n_beams * (n_psi + 2)) over NVLink on the devices' profile buffers (communicators from ncclCommInitAll at
 * torj_multi_create; libnccl.so.2 is loaded at run time), or — reduction = 1, and whenever NCCL is unavailable — a
 * host sum in device order. Neither is bit-reproducible by default: each device's own profile carries the noise of its
 * floating-point atomics. With torj_multi_set_exact_sum(m, 1) both sum the devices' integer accumulators instead (an
 * ncclInt64 all-reduce or a host integer sum) and convert once, which gives the bits of one device tracing the whole
 * bundle, whatever the device count and sharding (at a fixed lanes_per_ray).
 * sharding: 0 = contiguous ray blocks; 1 = block-cyclic, blocks of `block_rays` consecutive rays (one beam) dealt
 * round-robin, which balances scans whose beams differ in ray length. */
typedef struct torj_multi torj_multi;
typedef struct torj_mplasma torj_mplasma;
int torj_multi_create(int32_t n_devices /* <= 0: all visible */, torj_multi** out);
void torj_multi_destroy(torj_multi* m);
int32_t torj_multi_device_count(const torj_multi* m);
int torj_multi_configure(torj_multi* m, int32_t sharding, int64_t block_rays, int32_t reduction);
/* 1 when the cross-device sum of the last torj_multi_trace(_plasmas) went through ncclAllReduce, 0 for the host sum */
int32_t torj_multi_used_nccl(const torj_multi* m);
int torj_multi_abs_init(torj_multi* m, int32_t n, const double* nodes, const double* weights);
/* torj_ctx_set_exact_sum on every device's context: exact sums for every later torj_multi_trace(_plasmas); 0 or 1 */
int torj_multi_set_exact_sum(torj_multi* m, int32_t on);
/* torj_ctx_last_trace_ms of device d's context: the k_trace time of its part of the last torj_multi_trace(_plasmas) */
int torj_multi_last_trace_ms(torj_multi* m, int32_t device, double* ms);
int torj_multi_plasma_create_from_data(torj_multi* m, const torj_grid* grid, const double* psi_norm, const double* psi_prof,
                                       const double* ne_prof, const double* Te_prof, int32_t n_prof, const double* BR,
                                       const double* BZ, const double* Bphi, const double* psi_1d, const double* vol_1d,
                                       int32_t n_1d, torj_mplasma** out);
void torj_multi_plasma_destroy(torj_mplasma* mp);
int torj_multi_trace(torj_multi* m, const torj_mplasma* mp, const torj_options* opt, int64_t n_rays, const double* pos,
                     const double* dir, const double* weight, const double* freq_hz, const int32_t* mode, int32_t per_ray_fm,
                     double s_max, int32_t n_psi, const double* psi_edges, int32_t n_beams, const int32_t* beam_id,
                     double* dP_dV, double* deposited_power, double* P_final, double* P_deposited_ray, int32_t* n_points,
                     int32_t* status, int64_t traj_first, int64_t traj_count, int32_t traj_max_pts, double* traj_s,
                     double* traj_xyz, double* traj_P, double* traj_dP_ds, double* traj_dP_dV_ray, torj_counters* counters);
/* torj_multi_trace through a plasma set (torj_trace_plasmas sharded over the devices): beam b of beam_id is traced through
 * plasmas[beam_plasma[b]] on whichever device holds its rays; device d traces through the copies {plasmas[k] on d}. Each
 * device's profile rows are already divided by their beam's plasma volume, so the one all-reduce (or host sum) of
 * n_beams * (n_psi + 2) doubles is the set's profile; a device holds zero rows for the beams it did not trace.
 * Block-cyclic sharding with block_rays = rays per beam deals whole beams. Refused before anything is enqueued (non-zero,
 * torj_last_error, every device's workspace left as it was): the refusals of torj_trace_plasmas on every device, and a
 * plasma created by another torj_multi. n_plasmas = 1 is torj_multi_trace (beam_plasma unused). */
int torj_multi_trace_plasmas(torj_multi* m, int32_t n_plasmas, const torj_mplasma* const* plasmas,
                             const int32_t* beam_plasma /* [n_beams] */, const torj_options* opt, int64_t n_rays,
                             const double* pos, const double* dir, const double* weight, const double* freq_hz,
                             const int32_t* mode, int32_t per_ray_fm, double s_max, int32_t n_psi, const double* psi_edges,
                             int32_t n_beams, const int32_t* beam_id, double* dP_dV, double* deposited_power, double* P_final,
                             double* P_deposited_ray, int32_t* n_points, int32_t* status, int64_t traj_first,
                             int64_t traj_count, int32_t traj_max_pts, double* traj_s, double* traj_xyz, double* traj_P,
                             double* traj_dP_ds, double* traj_dP_dV_ray, torj_counters* counters);

/* --- measurement ------------------------------------------------------------------------------------------- */
/* Register-resident DFMA-chain microbenchmark: the FP64 roofline denominator (MEASURED_PEAKS.json has none). */
int torj_fp64_peak(torj_ctx* ctx, int32_t iters, double* tflops, double* ms);
/* Dependent-issue latency of DFMA in cycles (one warp, one chain): how much ILP x TLP the FP64 pipe needs. */
int torj_fp64_latency(torj_ctx* ctx, int32_t iters, double* cycles_per_dfma);
/* The kernels' own reciprocal, reciprocal square root, square root and exp (MUFU seed + FMA correction; branch-free
   exp) on n host values x > 0 (exp: any |x| <= 708): out[4][n] in that order. For accuracy tests against libm. */
int torj_math_probe(torj_ctx* ctx, int64_t n, const double* x, double* out);

#ifdef __cplusplus
}
#endif
#endif /* TORJ_CUDA_H */
