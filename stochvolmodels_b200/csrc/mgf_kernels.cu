// mgf_kernels.cu -- Fourier / moment-generating-function hot path for sm_100a (B200).
//
// Replaces (paths under /root/reference/src/stochvolmodels):
//   func_a_ode_quadratic_terms, func_rhs            pricers/logsv/affine_expansion.py:67-205
//   solve_ode_for_a / solve_a_ode_grid (RK45)       pricers/logsv/affine_expansion.py:229-303, 492-529
//       -> scipy.integrate.solve_ivp(method="RK45", rtol=1e-3, atol=1e-6): scipy/integrate/_ivp/rk.py, common.py
//   compute_logsv_a_mgf_grid (log-MGF contraction)  pricers/logsv/affine_expansion.py:570-685
//   logsv_chain_pricer (LOG_RETURN)                 pricers/logsv_pricer.py:669-739
//   compute_heston_mgf_grid, heston_chain_pricer    pricers/heston_pricer.py:183-282
//   get_phi_grid, _compute_legacy_pricer_weights, vanilla_slice_pricer_with_mgf_grid   utils/mgf_pricer.py:11-34,157-221
//
// Design (DESIGN.md §4): the grid is P = 1000 independent ODE systems per maturity -- latency bound, no data reuse, no
// tensor-core shape.  One thread integrates one grid point through ALL maturities of the chain with the coefficient
// vector A in registers (the reference carries a_t0 across maturities the same way), using the exact step-size control
// law of SciPy's RK45 so that accepted steps -- and therefore prices -- match the reference to ~1e-13.  CTAs are kept
// tiny (8..64 threads) so the 1000 threads spread over as many SMs as possible and a warp waits for few slow lanes.
// A second kernel does the Simpson-weighted Fourier sums, one CTA per strike, fixed-order fp64 reduction.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "../../include/b200sv.h"
#include "common.cuh"
#include "black.cuh"
#include "fastmath64.cuh"

namespace b200sv {

struct cd {
  double re, im;
};
__host__ __device__ __forceinline__ cd mk(double re, double im = 0.0) { return cd{re, im}; }
__device__ __forceinline__ cd operator+(cd a, cd b) { return cd{a.re + b.re, a.im + b.im}; }
__device__ __forceinline__ cd operator-(cd a, cd b) { return cd{a.re - b.re, a.im - b.im}; }
__device__ __forceinline__ cd operator-(cd a) { return cd{-a.re, -a.im}; }
__device__ __forceinline__ cd operator*(cd a, cd b) { return cd{a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; }
__device__ __forceinline__ cd operator*(double s, cd a) { return cd{s * a.re, s * a.im}; }
__device__ __forceinline__ cd operator*(cd a, double s) { return cd{s * a.re, s * a.im}; }
__device__ __forceinline__ double cabs2(cd a) { return a.re * a.re + a.im * a.im; }
__device__ __forceinline__ double cabs_(cd a) { return hypot(a.re, a.im); }
// Smith's division (what numpy uses for complex128)
__device__ __forceinline__ cd operator/(cd a, cd b) {
  if (fabs(b.re) >= fabs(b.im)) {
    const double r = b.im / b.re, d = b.re + b.im * r;
    return cd{(a.re + a.im * r) / d, (a.im - a.re * r) / d};
  }
  const double r = b.re / b.im, d = b.re * r + b.im;
  return cd{(a.re * r + a.im) / d, (a.im * r - a.re) / d};
}
__device__ __forceinline__ cd csqrt_(cd z) {   // principal branch
  if (z.re == 0.0 && z.im == 0.0) return cd{0.0, z.im};
  const double t = sqrt(0.5 * (fabs(z.re) + hypot(z.re, z.im)));
  if (z.re >= 0.0) return cd{t, z.im / (2.0 * t)};
  return cd{fabs(z.im) / (2.0 * t), copysign(t, z.im)};
}
__device__ __forceinline__ cd cexp_(cd z) {
  double s, c;
  sincos(z.im, &s, &c);
  const double e = exp(z.re);
  return cd{e * c, e * s};
}
__device__ __forceinline__ cd clog_(cd z) { return cd{log(hypot(z.re, z.im)), atan2(z.im, z.re)}; }

// --------------------------------------------------------------------------------------------------------------------
// LogSV affine expansion: per-grid-point coefficients of A' = A^T M A + L A + H (sparse, hand-expanded)
// --------------------------------------------------------------------------------------------------------------------
struct LogsvModel {   // phi-independent reals, built on the host: affine_expansion.py:121-135
  double theta, th2, v2, qv, qv2, lam, k2p, kp, beta_eta, eta2;
  int spot;
};

static LogsvModel make_model(const b200sv_logsv_params& p, double eta, bool spot) {
  LogsvModel m;
  m.theta = p.theta;
  m.th2 = p.theta * p.theta;
  m.v2 = p.beta * p.beta + p.volvol * p.volvol;
  m.qv = p.theta * m.v2;
  m.qv2 = m.th2 * m.v2;
  m.eta2 = eta * eta;
  if (spot) {
    m.lam = 0.0;
    m.k2p = p.kappa2;
    m.kp = p.kappa1 + p.kappa2 * p.theta;
  } else {
    m.lam = p.beta * m.th2 * eta;
    m.k2p = p.kappa2 - p.beta * eta;
    m.kp = p.kappa1 + p.kappa2 * p.theta - 2 * p.beta * p.theta * eta;
  }
  m.beta_eta = p.beta * eta;
  m.spot = spot ? 1 : 0;
  return m;
}

struct Coef {   // the phi/psi-dependent entries of L and H (affine_expansion.py:166-183)
  cd l01, l11, l12, l21, l22, l23, l32, l33, l34, l43, l44, h0, h1, h2;
};

__device__ __forceinline__ Coef make_coef(const LogsvModel& m, cd phi, cd psi) {
  Coef c;
  const cd b = m.beta_eta * phi;
  c.l01 = mk(m.lam) - m.th2 * b;
  c.l11 = mk(-m.kp) - (2.0 * m.theta) * b;
  c.l12 = 2.0 * (mk(m.lam + m.qv) - m.th2 * b);
  c.l21 = mk(-m.k2p) - b;
  c.l22 = mk(m.v2 - 2.0 * m.kp) - (4.0 * m.theta) * b;
  c.l23 = 3.0 * (mk(2.0 * m.qv) - m.th2 * b);
  c.l32 = -2.0 * (mk(m.k2p) + b);
  c.l33 = 3.0 * (mk(m.v2 - m.kp) - (2.0 * m.theta) * b);
  c.l34 = 4.0 * (mk(3.0 * m.qv) - m.th2 * b);
  c.l43 = -3.0 * (mk(m.k2p) + b);
  c.l44 = 2.0 * (mk(m.v2 - 2.0 * m.kp) - (4.0 * m.theta) * b);
  const cd r = m.spot ? phi * (phi + mk(1.0)) - 2.0 * psi : phi * (phi - mk(1.0)) - 2.0 * psi;
  c.h0 = (0.5 * m.th2 * m.eta2) * r;
  c.h1 = (m.theta * m.eta2) * r;
  c.h2 = (0.5 * m.eta2) * r;
  return c;
}

// The 14 phi/psi-dependent coefficients of one thread, parked in shared memory ([coef][thread]) like the RK stages: the kernel is
// latency-bound, so register space is better spent on independent in-flight products than on long-lived constants.
template <int TPB>
struct CoefView {
  const cd* base;
  __device__ __forceinline__ cd at(int i) const { return base[i * TPB]; }
};
template <int TPB>
__device__ __forceinline__ void store_coef(cd* base, const Coef& c) {
  const cd v[14] = {c.l01, c.l11, c.l12, c.l21, c.l22, c.l23, c.l32, c.l33, c.l34, c.l43, c.l44, c.h0, c.h1, c.h2};
#pragma unroll
  for (int i = 0; i < 14; ++i) base[i * TPB] = v[i];
}

template <int N, int TPB>
__device__ __forceinline__ void rhs(const cd (&A)[N], const LogsvModel& m, const CoefView<TPB>& cv, cd (&out)[N]) {
  struct {
    cd l01, l11, l12, l21, l22, l23, l32, l33, l34, l43, l44, h0, h1, h2;
  } c;
  c.l01 = cv.at(0); c.l11 = cv.at(1); c.l12 = cv.at(2); c.l21 = cv.at(3); c.l22 = cv.at(4); c.h0 = cv.at(11); c.h1 = cv.at(12); c.h2 = cv.at(13);
  if constexpr (N == 5) {
    c.l23 = cv.at(5); c.l32 = cv.at(6); c.l33 = cv.at(7); c.l34 = cv.at(8); c.l43 = cv.at(9); c.l44 = cv.at(10);
  }
  const double v2 = m.v2, qv = m.qv, qv2 = m.qv2;
  const cd a1 = A[1], a2 = A[2];
  const cd a11 = a1 * a1, a12 = a1 * a2, a22 = a2 * a2;
  if constexpr (N == 5) {
    const cd a3 = A[3], a4 = A[4];
    const cd a13 = a1 * a3, a14 = a1 * a4, a23 = a2 * a3, a24 = a2 * a4, a33 = a3 * a3;
    out[0] = (0.5 * qv2) * a11 + c.l01 * a1 + qv2 * a2 + c.h0;
    out[1] = qv * a11 + (2.0 * qv2) * a12 + c.l11 * a1 + c.l12 * a2 + (3.0 * qv2) * a3 + c.h1;
    out[2] = (0.5 * v2) * a11 + (2.0 * qv2) * a22 + (4.0 * qv) * a12 + (3.0 * qv2) * a13 + c.l21 * a1 + c.l22 * a2 + c.l23 * a3 +
             (6.0 * qv2) * a4 + c.h2;
    out[3] = (4.0 * qv) * a22 + (2.0 * v2) * a12 + (6.0 * qv) * a13 + (4.0 * qv2) * a14 + (6.0 * qv2) * a23 + c.l32 * a2 +
             c.l33 * a3 + c.l34 * a4;
    out[4] = (2.0 * v2) * a22 + (4.5 * qv2) * a33 + (3.0 * v2) * a13 + (8.0 * qv) * a14 + (12.0 * qv) * a23 + (8.0 * qv2) * a24 +
             c.l43 * a3 + c.l44 * a4;
  } else {
    out[0] = (0.5 * qv2) * a11 + c.l01 * a1 + qv2 * a2 + c.h0;
    out[1] = qv * a11 + (2.0 * qv2) * a12 + c.l11 * a1 + c.l12 * a2 + c.h1;
    out[2] = (0.5 * v2) * a11 + (2.0 * qv2) * a22 + (4.0 * qv) * a12 + c.l21 * a1 + c.l22 * a2 + c.h2;
  }
}

// --------------------------------------------------------------------------------------------------------------------
// SciPy RK45 clone (scipy/integrate/_ivp/rk.py:111-170 step loop, :14-69 stages, :538-552 tableau;
//                   scipy/integrate/_ivp/common.py:63-65 norm, :109-134 select_initial_step)
// --------------------------------------------------------------------------------------------------------------------
__constant__ double c_A[6][5] = {{0, 0, 0, 0, 0},
                                 {1.0 / 5, 0, 0, 0, 0},
                                 {3.0 / 40, 9.0 / 40, 0, 0, 0},
                                 {44.0 / 45, -56.0 / 15, 32.0 / 9, 0, 0},
                                 {19372.0 / 6561, -25360.0 / 2187, 64448.0 / 6561, -212.0 / 729, 0},
                                 {9017.0 / 3168, -355.0 / 33, 46732.0 / 5247, 49.0 / 176, -5103.0 / 18656}};   // Dormand-Prince A (rk.py:542-549)
constexpr double kRtol = 1e-3, kAtol = 1e-6;   // solve_ivp defaults, affine_expansion.py:300-301 passes none

// Step-size control arithmetic of the RK45 clone (error scale, RMS norm): MUFU-seeded reciprocal / square root with Newton refinement
// (<= 2 ulp, fastmath64.cuh) instead of the IEEE sequences with their slow-path branches -- these sit on the dependent chain of every
// step attempt.  Moduli below 1e-145 count as 0 (the scale is atol + |a| rtol with atol = 1e-6: identical result).
__device__ __forceinline__ double ctrl_sqrt(double s) { return s < 1e-290 ? 0.0 : fast_sqrt(s); }
__device__ __forceinline__ double ctrl_rcp(double x) { return fast_div(1.0, x); }     // x >= atol
// RMS norm of v / scale over complex moduli (scipy/integrate/_ivp/common.py:63-65); inv_scale = 1 / scale.
template <int N>
__device__ __forceinline__ double rms_scaled(const cd (&v)[N], const double (&inv_scale)[N]) {
  double s = 0.0;
#pragma unroll
  for (int k = 0; k < N; ++k) {
    const double re = v[k].re * inv_scale[k], im = v[k].im * inv_scale[k];
    s += re * re + im * im;
  }
  return ctrl_sqrt(s) * (N == 5 ? 0.44721359549995793 : 0.57735026918962576);   // / sqrt(N)
}
__device__ __forceinline__ double cmod(cd a) { return ctrl_sqrt(a.re * a.re + a.im * a.im); }   // |a| (no overflow risk for these magnitudes)
// e^(-1/5), e > 0, for the step-size factor 0.9 e^(-1/5) clipped to [0.2, 10]: SFU single-precision seed + two Newton steps on x^-5 = e
// (x <- x (1.2 - 0.2 e x^5), quadratic: 1e-6 -> 3e-12 -> 1 ulp) instead of exp(-0.2 log e).  Outside [1e-30, 1e30] the clipped factor
// does not depend on e, so e is clamped for the float seed; NaN propagates (fmax(0.2, NaN) = 0.2 as before).
__device__ __forceinline__ double pow_m02(double e) {
  const double ec = e != e ? e : fmin(fmax(e, 1e-30), 1e30);
  double x = (double)__powf((float)ec, -0.2f);
  const double c = 0.2 * ec;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const double x2 = x * x;
    x = x * fma(-c, x2 * x2 * x, 1.2);
  }
  return x;
}

// Stage storage of one thread in shared memory: K[stage][component][thread] (16-byte elements, conflict-free across threads).
// Keeping the 7 x N complex stages out of the register file leaves ptxas room to schedule the independent products of the
// right-hand side in parallel: the kernel is latency-bound (one warp per SM), so ILP is what matters.
template <int N, int TPB>
struct StageStore {
  cd* base;
  __device__ __forceinline__ cd& at(int stage, int k) { return base[(stage * N + k) * TPB]; }
};

// returns 0 ok, 1 step size underflow (SciPy: TOO_SMALL_STEP -> solver fails, reference keeps the last accepted state)
// Rhs: functor ``void operator()(const cd (&A)[N], cd (&out)[N]) const`` -- the LogSV coefficient ODEs (LogsvRhsFn) or the Hawkes Riccati
// system (HawkesRhsFn); the control law does not depend on it.
template <int N, int TPB, typename Rhs>
__device__ int rk45_generic(cd (&y)[N], double T, const Rhs& rhs_fn, StageStore<N, TPB> K, int* nfev_out) {
  // stage coefficients: c_A in constant memory (indexed by the non-unrolled stage loop)
  constexpr double B[6] = {35.0 / 384, 0, 500.0 / 1113, 125.0 / 192, -2187.0 / 6784, 11.0 / 84};
  constexpr double E[7] = {-71.0 / 57600, 0, 71.0 / 16695, -71.0 / 1920, 17253.0 / 339200, -22.0 / 525, 1.0 / 40};

  cd f[N];                       // f(t, y): registers during the initial-step selection, then stage 0 of the shared-memory store
  rhs_fn(y, f);
  int nfev = 1;
  double inv_scale[N];
  // ---- select_initial_step (scipy/integrate/_ivp/common.py:109-134)
  double h_abs;
  {
#pragma unroll
    for (int k = 0; k < N; ++k) inv_scale[k] = ctrl_rcp(kAtol + cmod(y[k]) * kRtol);
    const double d0 = rms_scaled<N>(y, inv_scale), d1 = rms_scaled<N>(f, inv_scale);
    double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
    h0 = fmin(h0, T);
    cd y1[N], f1[N];
#pragma unroll
    for (int k = 0; k < N; ++k) y1[k] = y[k] + h0 * f[k];
    rhs_fn(y1, f1);
    ++nfev;
#pragma unroll
    for (int k = 0; k < N; ++k) f1[k] = f1[k] - f[k];
    const double d2 = rms_scaled<N>(f1, inv_scale) / h0;
    const double h1 = (d1 <= 1e-15 && d2 <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : exp(0.2 * log(0.01 / fmax(d1, d2)));
    h_abs = fmin(fmin(100.0 * h0, h1), T);
  }
  double t = 0.0;
  int status = 0;
#pragma unroll
  for (int k = 0; k < N; ++k) K.at(0, k) = f[k];
  // ONE loop over step ATTEMPTS (SciPy nests "while not accepted" inside the step loop): a lane that rejects an attempt simply goes round
  // again with the lanes that accepted theirs, so a warp runs max-over-lanes of the TOTAL attempts instead of the sum over steps of
  // the per-step maximum.  Same arithmetic per point.
  bool rejected = false;
  for (int guard = 0; t < T && guard < 400000; ++guard) {
    {
      const double min_step = 10.0 * (__longlong_as_double(__double_as_longlong(t) + 1) - t);   // 10*|nextafter(t, inf) - t|, t >= 0
      if (!rejected) {
        if (h_abs < min_step) h_abs = min_step;       // first attempt of a step (max_step = inf)
      } else if (h_abs < min_step) {
        status = 1;
        break;
      }
      double t_new = t + h_abs;
      if (t_new - T > 0.0) t_new = T;
      const double h = t_new - t;
      h_abs = fabs(h);
      cd yt[N], kn[N];
#pragma unroll 1
      for (int s = 1; s < 6; ++s) {            // rk_step (scipy/integrate/_ivp/rk.py:60-64): dy = (sum_j K_j a_sj) * h
        // not unrolled on purpose: the fully unrolled body (5 inlined right-hand sides) is ~70 KB of SASS and the single resident
        // warp per SM then stalls on instruction fetch; stages >= s still hold zeros / stale finite values and get coefficient 0
        // (skipping them with a warp-uniform trip count was measured: no gain, more spills)
#pragma unroll
        for (int k = 0; k < N; ++k) {
          cd acc = K.at(0, k) * c_A[s][0];
#pragma unroll
          for (int jj = 1; jj < 5; ++jj) acc = acc + K.at(jj, k) * c_A[s][jj];
          yt[k] = y[k] + acc * h;
        }
        rhs_fn(yt, kn);
#pragma unroll
        for (int k = 0; k < N; ++k) K.at(s, k) = kn[k];
      }
      cd yn[N];
#pragma unroll
      for (int k = 0; k < N; ++k) {
        cd acc = K.at(0, k) * B[0];
#pragma unroll
        for (int jj = 2; jj < 6; ++jj) acc = acc + K.at(jj, k) * B[jj];      // B[1] = 0
        yn[k] = y[k] + h * acc;
      }
      rhs_fn(yn, kn);                                                   // K[6] = f(t + h, y_new)
      nfev += 6;
      cd err[N];
#pragma unroll
      for (int k = 0; k < N; ++k) {
        inv_scale[k] = ctrl_rcp(kAtol + fmax(cmod(y[k]), cmod(yn[k])) * kRtol);
        cd acc = K.at(0, k) * E[0];
#pragma unroll
        for (int jj = 2; jj < 6; ++jj) acc = acc + K.at(jj, k) * E[jj];      // E[1] = 0
        err[k] = (acc + kn[k] * E[6]) * h;
      }
      const double en = rms_scaled<N>(err, inv_scale);
      const bool accepted = en < 1.0;
      const double pf = en == 0.0 ? 10.0 : 0.9 * pow_m02(en);
      double factor = fmin(10.0, pf);
      if (rejected) factor = fmin(1.0, factor);
      h_abs *= accepted ? factor : fmax(0.2, pf);
      if (accepted) {
        t = t_new;
#pragma unroll
        for (int k = 0; k < N; ++k) {
          y[k] = yn[k];
          K.at(0, k) = kn[k];     // FSAL: K[6] of this step is K[0] of the next
        }
      }
      rejected = !accepted;
    }
  }
  if (nfev_out) *nfev_out = nfev;
  return status;
}

template <int N, int TPB>
struct LogsvRhsFn {
  const LogsvModel& m;
  const CoefView<TPB>& c;
  __device__ __forceinline__ void operator()(const cd (&A)[N], cd (&out)[N]) const { rhs<N, TPB>(A, m, c, out); }
};
template <int N, int TPB>
__device__ __forceinline__ int rk45(cd (&y)[N], double T, const LogsvModel& m, const CoefView<TPB>& c, StageStore<N, TPB> K, int* nfev_out) {
  return rk45_generic<N, TPB>(y, T, LogsvRhsFn<N, TPB>{m, c}, K, nfev_out);
}

struct ChainSpec {   // per-maturity scalars (device array of M entries)
  double dtau;
  LogsvModel model;
};

// one thread = one grid point through all M maturities.  a_io: [P][N] in (A(0)) ; a_out: [M][P][N]; log_mgf: [M][P]
// blockIdx.y = parameter set of a batch (b200sv_logsv_price_chain_batch): spec[b][M], yb[b], phi[b][P] (phi_stride = P) or one shared
// grid (phi_stride = 0), outputs [b][M][P]...
template <int N, int TPB>
__global__ void __launch_bounds__(TPB) logsv_mgf_kernel(const cd* __restrict__ phi, const cd* __restrict__ psi, int P, int M,
                                 const ChainSpec* __restrict__ spec, const cd* __restrict__ a_in, cd* __restrict__ a_out,
                                 cd* __restrict__ log_mgf, double y, int* __restrict__ status, int* __restrict__ nfev,
                                 const double* __restrict__ yb = nullptr, int phi_stride = 0, int set_major_B = 0) {
  __shared__ cd stage_smem[6 * N * TPB];
  __shared__ cd coef_smem[14 * TPB];
  // Batches (set_major_B = B > 1): the parameter set is the FASTEST thread index, so the lanes of a warp integrate the same grid point
  // for 32 neighbouring sets -- the sets of a calibration batch are perturbations of one another and take (nearly) the same adaptive
  // steps, whereas neighbouring grid points of one set do not (24 of 32 lanes active with the point-major mapping, r01 profile).
  int p = blockIdx.x * TPB + threadIdx.x;
  size_t b = blockIdx.y;
  if (set_major_B > 1) {
    const long long t = (long long)blockIdx.x * TPB + threadIdx.x;
    if (t >= (long long)set_major_B * P) return;
    b = (size_t)(t % set_major_B);
    p = (int)(t / set_major_B);
  }
  if (p >= P) return;
  if (gridDim.y > 1 || yb) {
    spec += b * M;
    phi += b * (size_t)phi_stride;
    a_out += b * (size_t)M * P * N;
    log_mgf += b * (size_t)M * P;
    if (status) status += b * (size_t)P;
    if (yb) y = yb[b];
  }
  StageStore<N, TPB> K{stage_smem + threadIdx.x};
#pragma unroll
  for (int i = 0; i < 6 * N; ++i) stage_smem[threadIdx.x + i * TPB] = mk(0.0);      // stages read with coefficient 0 must be finite
  cd A[N];
#pragma unroll
  for (int k = 0; k < N; ++k) A[k] = a_in ? a_in[(size_t)p * N + k] : mk(0.0);
  const cd ph = phi[p], ps = psi ? psi[p] : mk(0.0);
  // ys = [1, y, y^2, y^3, y^4] (affine_expansion.py:674-681)
  const double y2 = y * y;
  const double ys[5] = {1.0, y, y2, y2 * y, y2 * y2};
  int st = 0, nf = 0;
  for (int mm = 0; mm < M; ++mm) {
    const LogsvModel model = spec[mm].model;
    store_coef<TPB>(coef_smem + threadIdx.x, make_coef(model, ph, ps));
    const CoefView<TPB> c{coef_smem + threadIdx.x};
    int nfe = 0;
    st |= rk45<N, TPB>(A, spec[mm].dtau, model, c, K, &nfe);
    nf += nfe;
    cd lm = mk(0.0);
#pragma unroll
    for (int k = 0; k < N; ++k) {
      a_out[((size_t)mm * P + p) * N + k] = A[k];
      lm = lm + A[k] * ys[k];
    }
    log_mgf[(size_t)mm * P + p] = lm;
  }
  if (status) status[p] = st;
  if (nfev) nfev[p] = nf;
}

// --------------------------------------------------------------------------------------------------------------------
// Lane-parallel variant for the latency regime (one chain, P = 1000): the N components of A are spread over N lanes of a group of LPP
// lanes (8 for N = 5, 4 for N = 3), so one Runge-Kutta stage costs each lane ONE row of A'MA + LA + H (<= 6 quadratic + 4 linear terms)
// instead of all N rows -- about a third of the dependent instruction stream of the thread-per-point kernel, which is what bounds a
// single chain pricing (one resident warp per SM).  The stage vector is exchanged through shared memory (one 16-byte store, <= 5 loads,
// __syncwarp); each lane keeps its own 7 stage derivatives in registers.  Step-size control is replicated in every lane of a point from
// an error norm summed in component order, i.e. the same accepted steps as the thread-per-point kernel; all points of a warp iterate
// together (finished points idle) so the warp-level barriers stay converged.  Row k accumulates its terms in the order of rhs<>().
// --------------------------------------------------------------------------------------------------------------------
template <int N>
struct LaneRow {        // row k of the right-hand side in table form
  cd l[4];              // linear coefficients (complex; real ones carry im = 0)
  double q[6];          // quadratic coefficients (already doubled for off-diagonal pairs)
  cd h;
  int li[4], qi[6], qj[6];
  int nl, nq;
};

template <int N>
__device__ __forceinline__ LaneRow<N> make_lane_row(int k, const LogsvModel& m, cd phi, cd psi) {
  const Coef c = make_coef(m, phi, psi);
  const double v2 = m.v2, qv = m.qv, qv2 = m.qv2;
  LaneRow<N> r;
  // padding entries: coefficient 0 on a component every row already depends on (rows 0-3: A1, row 4: A3), so that a non-finite value
  // cannot enter a row through a padded term unless the row is non-finite anyway
  const int pad = k == 4 ? 3 : 1;
#pragma unroll
  for (int t = 0; t < 4; ++t) { r.l[t] = mk(0.0); r.li[t] = pad; }
#pragma unroll
  for (int t = 0; t < 6; ++t) { r.q[t] = 0.0; r.qi[t] = pad; r.qj[t] = pad; }
  r.h = mk(0.0);
  r.nl = r.nq = 0;
  auto Q = [&](double coef, int i, int j) { r.q[r.nq] = coef; r.qi[r.nq] = i; r.qj[r.nq] = j; ++r.nq; };
  auto L = [&](cd coef, int i) { r.l[r.nl] = coef; r.li[r.nl] = i; ++r.nl; };
  // same term order as rhs<>() above (affine_expansion.py:139-183)
  if (k == 0) {
    Q(0.5 * qv2, 1, 1); L(c.l01, 1); L(mk(qv2), 2); r.h = c.h0;
  } else if (k == 1) {
    Q(qv, 1, 1); Q(2.0 * qv2, 1, 2); L(c.l11, 1); L(c.l12, 2);
    if (N == 5) L(mk(3.0 * qv2), 3);
    r.h = c.h1;
  } else if (k == 2) {
    Q(0.5 * v2, 1, 1); Q(2.0 * qv2, 2, 2); Q(4.0 * qv, 1, 2);
    if (N == 5) Q(3.0 * qv2, 1, 3);
    L(c.l21, 1); L(c.l22, 2);
    if (N == 5) { L(c.l23, 3); L(mk(6.0 * qv2), 4); }
    r.h = c.h2;
  } else if (k == 3) {
    Q(4.0 * qv, 2, 2); Q(2.0 * v2, 1, 2); Q(6.0 * qv, 1, 3); Q(4.0 * qv2, 1, 4); Q(6.0 * qv2, 2, 3);
    L(c.l32, 2); L(c.l33, 3); L(c.l34, 4);
  } else if (k == 4) {
    Q(2.0 * v2, 2, 2); Q(4.5 * qv2, 3, 3); Q(3.0 * v2, 1, 3); Q(8.0 * qv, 1, 4); Q(12.0 * qv, 2, 3); Q(8.0 * qv2, 2, 4);
    L(c.l43, 3); L(c.l44, 4);
  }
  return r;
}

// f_k(Y) for this lane's row; Y = the point's stage vector in shared memory.  Branch-free: rows shorter than 6 + 4 terms are padded with
// zero coefficients on an entry the row already reads (make_lane_row), so every lane of the warp runs the same instruction stream.
template <int N>
__device__ __forceinline__ cd lane_rhs(const LaneRow<N>& r, const cd* __restrict__ Y) {
  cd acc = r.q[0] * (Y[r.qi[0]] * Y[r.qj[0]]);
#pragma unroll
  for (int t = 1; t < (N == 5 ? 6 : 3); ++t) acc = acc + r.q[t] * (Y[r.qi[t]] * Y[r.qj[t]]);
#pragma unroll
  for (int t = 0; t < (N == 5 ? 4 : 2); ++t) acc = acc + r.l[t] * Y[r.li[t]];
  return acc + r.h;
}

constexpr int kLaneWarpsPerBlock = 1;

template <int N>
__global__ void __launch_bounds__(32 * kLaneWarpsPerBlock, 1) logsv_mgf_lanes_kernel(
    const cd* __restrict__ phi, const cd* __restrict__ psi, int P, int M, const ChainSpec* __restrict__ spec, const cd* __restrict__ a_in,
    cd* __restrict__ a_out, cd* __restrict__ log_mgf, double y, int* __restrict__ status_out, const double* __restrict__ yb, int phi_stride) {
  constexpr int LPP = N == 5 ? 8 : 4;             // lanes per grid point
  constexpr int PPW = 32 / LPP;                   // points per warp
  constexpr unsigned FULL = 0xffffffffu;
  constexpr double B[6] = {35.0 / 384, 0, 500.0 / 1113, 125.0 / 192, -2187.0 / 6784, 11.0 / 84};
  constexpr double E[7] = {-71.0 / 57600, 0, 71.0 / 16695, -71.0 / 1920, 17253.0 / 339200, -22.0 / 525, 1.0 / 40};
  constexpr double A[6][5] = {{0, 0, 0, 0, 0},
                              {1.0 / 5, 0, 0, 0, 0},
                              {3.0 / 40, 9.0 / 40, 0, 0, 0},
                              {44.0 / 45, -56.0 / 15, 32.0 / 9, 0, 0},
                              {19372.0 / 6561, -25360.0 / 2187, 64448.0 / 6561, -212.0 / 729, 0},
                              {9017.0 / 3168, -355.0 / 33, 46732.0 / 5247, 49.0 / 176, -5103.0 / 18656}};
  __shared__ cd Ysh[kLaneWarpsPerBlock][PPW][N];
  __shared__ double Nsh[kLaneWarpsPerBlock][PPW][N];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = lane / LPP, k = lane % LPP;        // point within the warp, component
  const int p = (blockIdx.x * kLaneWarpsPerBlock + wib) * PPW + g;
  {
    const size_t b = blockIdx.y;
    spec += b * M;
    phi += b * (size_t)phi_stride;
    a_out += b * (size_t)M * P * N;
    log_mgf += b * (size_t)M * P;
    if (status_out) status_out += b * (size_t)P;
    if (yb) y = yb[b];
  }
  const bool valid = p < P, comp = k < N, mine = valid && comp;
  const int pc = valid ? p : P - 1;                // out-of-range groups shadow the last point (never stored)
  const int kc = comp ? k : 0;
  cd* Y = &Ysh[wib][g][0];
  double* Nn = &Nsh[wib][g][0];
  const cd ph = phi[pc], ps = psi ? psi[pc] : mk(0.0);
  cd yk = a_in ? a_in[(size_t)pc * N + kc] : mk(0.0);
  const double y2 = y * y;
  const double ys[5] = {1.0, y, y2, y2 * y, y2 * y2};
  int st_all = 0;

  // sum over the point's components, in component order, of this lane's value (identical in every lane of the point)
  auto point_norm = [&](cd v, double inv_scale) -> double {
    const double re = v.re * inv_scale, im = v.im * inv_scale;
    __syncwarp(FULL);
    if (comp) Nn[k] = re * re + im * im;
    __syncwarp(FULL);
    double s = 0.0;
#pragma unroll
    for (int c = 0; c < N; ++c) s += Nn[c];
    return ctrl_sqrt(s) * (N == 5 ? 0.44721359549995793 : 0.57735026918962576);   // / sqrt(N)
  };
  // f_k at the point's vector whose k-th entry is `mine_k`
  auto eval = [&](const LaneRow<N>& row, cd mine_k) -> cd {
    __syncwarp(FULL);
    if (comp) Y[k] = mine_k;
    __syncwarp(FULL);
    return lane_rhs<N>(row, Y);
  };

  for (int mm = 0; mm < M; ++mm) {
    const LogsvModel model = spec[mm].model;
    const double T = spec[mm].dtau;
    const LaneRow<N> row = make_lane_row<N>(kc, model, ph, ps);
    cd K[7];
    K[0] = eval(row, yk);
    double h_abs;
    {   // select_initial_step (scipy/integrate/_ivp/common.py:109-134)
      const double inv_scale = ctrl_rcp(kAtol + cmod(yk) * kRtol);
      const double d0 = point_norm(yk, inv_scale), d1 = point_norm(K[0], inv_scale);
      double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
      h0 = fmin(h0, T);
      const cd f1 = eval(row, yk + h0 * K[0]);
      const double d2 = point_norm(f1 - K[0], inv_scale) / h0;
      const double h1 = (d1 <= 1e-15 && d2 <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : exp(0.2 * log(0.01 / fmax(d1, d2)));
      h_abs = fmin(fmin(100.0 * h0, h1), T);
    }
    double t = 0.0, min_step = 0.0;
    bool done = !(t < T), in_step = false, rejected = false;
    int status = 0;
    for (int guard = 0; guard < 1000000 && __any_sync(FULL, !done); ++guard) {
      if (!done && !in_step) {                      // head of the outer loop of rk.py:111-170
        min_step = 10.0 * (__longlong_as_double(__double_as_longlong(t) + 1) - t);
        if (h_abs < min_step) h_abs = min_step;
        rejected = false;
        in_step = true;
      }
      if (!done && h_abs < min_step) {
        status = 1;
        done = true;
      }
      double t_new = t + h_abs;
      if (t_new - T > 0.0) t_new = T;
      const double h = t_new - t;
      if (!done) h_abs = fabs(h);
#pragma unroll
      for (int s = 1; s < 6; ++s) {
        cd acc = K[0] * A[s][0];
#pragma unroll
        for (int jj = 1; jj < 5; ++jj)
          if (jj < s) acc = acc + K[jj] * A[s][jj];
        K[s] = eval(row, yk + acc * h);
      }
      cd acc = K[0] * B[0];
#pragma unroll
      for (int jj = 2; jj < 6; ++jj) acc = acc + K[jj] * B[jj];
      const cd yn = yk + h * acc;
      K[6] = eval(row, yn);
      const double inv_scale = ctrl_rcp(kAtol + fmax(cmod(yk), cmod(yn)) * kRtol);
      cd e = K[0] * E[0];
#pragma unroll
      for (int jj = 2; jj < 6; ++jj) e = e + K[jj] * E[jj];
      const cd err = (e + K[6] * E[6]) * h;
      const double en = point_norm(err, inv_scale);
      if (!done) {
        if (en < 1.0) {
          double factor = en == 0.0 ? 10.0 : fmin(10.0, 0.9 * pow_m02(en));
          if (rejected) factor = fmin(1.0, factor);
          h_abs *= factor;
          t = t_new;
          yk = yn;
          K[0] = K[6];                               // FSAL
          in_step = false;
          done = !(t < T);
        } else {
          h_abs *= fmax(0.2, 0.9 * pow_m02(en));
          rejected = true;
        }
      }
    }
    st_all |= status;
    // outputs of this maturity: a_t1 and log_mgf = sum_k A_k ys_k in component order (affine_expansion.py:674-685)
    __syncwarp(FULL);
    if (comp) Y[k] = yk;
    __syncwarp(FULL);
    if (mine) a_out[((size_t)mm * P + p) * N + k] = yk;
    if (valid && k == 0) {
      cd lm = mk(0.0);
#pragma unroll
      for (int c = 0; c < N; ++c) lm = lm + Y[c] * ys[c];
      log_mgf[(size_t)mm * P + p] = lm;
    }
  }
  if (status_out && valid && k == 0) status_out[p] = st_all;
}

// --------------------------------------------------------------------------------------------------------------------
// Heston closed form: pricers/heston_pricer.py:199-214, chained over maturities with (a, b) carried in registers
// --------------------------------------------------------------------------------------------------------------------
__global__ void heston_mgf_kernel(const cd* __restrict__ phi, const cd* __restrict__ psi, int P, int M,
                                  const double* __restrict__ dtaus, b200sv_heston_params hp, const cd* __restrict__ a_in,
                                  const cd* __restrict__ b_in, cd* __restrict__ a_out, cd* __restrict__ b_out,
                                  cd* __restrict__ log_mgf, const b200sv_heston_params* __restrict__ hpb = nullptr, int phi_stride = 0) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  if (hpb) {                                       // batch of parameter sets (b200sv_heston_price_chain_batch): blockIdx.y = set
    const size_t b = blockIdx.y;
    hp = hpb[b];
    phi += b * (size_t)phi_stride;
    log_mgf += b * (size_t)M * P;
  }
  const cd ph = phi[p], ps = psi ? psi[p] : mk(0.0);
  cd a = a_in ? a_in[p] : mk(0.0), b = b_in ? b_in[p] : mk(0.0);
  const double vv2 = hp.volvol * hp.volvol;
  const cd b1 = mk(hp.kappa) + (hp.rho * hp.volvol) * ph;
  const cd b0 = (0.5 * ph) * (ph + mk(1.0)) - ps;
  const cd zeta = csqrt_(b1 * b1 - (2.0 * b0) * vv2);
  const cd psi_p = zeta - b1, psi_m = b1 + zeta;
  const cd two_zeta = 2.0 * zeta;
  for (int mm = 0; mm < M; ++mm) {
    const double tau = dtaus[mm];
    const cd ez = cexp_(-(zeta * tau));
    const cd c_p = (psi_p + vv2 * b) / two_zeta, c_m = (psi_m - vv2 * b) / two_zeta;
    const cd den = c_p * ez + c_m;
    const cd b_new = -((-(psi_m * c_p)) * ez + psi_p * c_m) / (vv2 * den);
    const cd a_new = (-(hp.theta * hp.kappa / vv2)) * (psi_p * tau + 2.0 * clog_(den)) + a;
    a = a_new;
    b = b_new;
    if (a_out) a_out[(size_t)mm * P + p] = a;
    if (b_out) b_out[(size_t)mm * P + p] = b;
    log_mgf[(size_t)mm * P + p] = a + b * hp.v0;
  }
}

// --------------------------------------------------------------------------------------------------------------------
// Fourier sums: utils/mgf_pricer.py:190-219.  One CTA per strike.
// --------------------------------------------------------------------------------------------------------------------
struct StrikeSpec {
  double strike, forward, discfactor;
  int type;     // B200SV_CALL ..
  int slice;    // which log_mgf row
  double ttm;   // only for the fused Black inversion of the batched pricers
  int grid;     // which phi row (batched pricers with per-set grids), else 0
};

constexpr int kFourierThreads = 256;

__global__ void __launch_bounds__(kFourierThreads) fourier_vanilla_kernel(const cd* __restrict__ log_mgf, const cd* __restrict__ phi,
                                                                         int P, const StrikeSpec* __restrict__ specs,
                                                                         int is_spot, int half_re, double* __restrict__ prices,
                                                                         double* __restrict__ ivols = nullptr) {
  __shared__ double red[kFourierThreads / 32];
  const StrikeSpec sp = specs[blockIdx.x];
  const cd* lm = log_mgf + (size_t)sp.slice * P;
  phi += (size_t)sp.grid * P;
  const double x = log(sp.forward / sp.strike);
  const double h3 = (phi[1].im - phi[0].im) / 3.0;
  double acc[1] = {0.0};
  for (int j = threadIdx.x; j < P; j += kFourierThreads) {
    // legacy Simpson weights (utils/mgf_pricer.py:163-170): 1,4,2,4,... with first/last = 1 and THEN every odd index = 4
    double wq = (j & 1) ? 4.0 : ((j == 0 || j == P - 1) ? 1.0 : 2.0);
    const double dp = h3 * wq;
    const cd ph = phi[j];
    cd w;
    if (half_re) {
      w = mk((dp / M_PI) / (ph.im * ph.im + 0.25));
    } else {
      const cd den = is_spot ? (ph + mk(1.0)) * ph : (ph - mk(1.0)) * ph;
      w = -(mk(dp / M_PI) / den);
    }
    const cd z = lm[j] - x * ph;
    const cd term = w * cexp_(z);
    if (term.re == term.re) acc[0] += term.re;     // np.nansum(np.real(...))
  }
  block_sum<1, kFourierThreads>(acc, red);
  if (threadIdx.x == 0) {
    const double capped = acc[0], F = sp.forward, K = sp.strike, df = sp.discfactor;
    double price;
    if (is_spot)
      price = sp.type == B200SV_CALL ? df * (F - K * capped) : df * (K - K * capped);
    else
      price = (sp.type == B200SV_CALL || sp.type == B200SV_INV_CALL) ? F * df * (1.0 - capped) : F * df * (exp(-x) - capped);
    prices[blockIdx.x] = price;
    // calibration objective: the Black inversion that follows every chain pricing (option_chain.py:327-346), fused
    if (ivols) ivols[blockIdx.x] = black_implied_vol(F, K, sp.ttm, df, price, sp.type);
  }
}

// Generic Fourier sum  S = nansum_j Re( w_j * exp(coef * g_j + log_mgf_j) )  for the other inversion formulas of
// utils/mgf_pricer.py: options on quadratic variance (:323-358), densities (:361-384), digitals (:224-269).
enum { kModeQvar = 1, kModePdf = 2, kModeDigital = 3 };
struct SumSpec {
  double coef;        // QVAR: strike*ttm ; PDF: z = (x - shift)/scale ; DIGITAL: -ln(F/K)
  double a, b;        // QVAR: a = discfactor, b = ttm ; DIGITAL: a = discfactor
  int type, slice;
};
static_assert(sizeof(SumSpec) <= sizeof(StrikeSpec), "the chain pricers stage either kind of spec in one StrikeSpec buffer");

__global__ void __launch_bounds__(kFourierThreads) fourier_sum_kernel(const cd* __restrict__ log_mgf, const cd* __restrict__ grid, int P,
                                                                     const SumSpec* __restrict__ specs, int mode, int all_calls,
                                                                     double* __restrict__ out) {
  __shared__ double red[kFourierThreads / 32];
  const SumSpec sp = specs[blockIdx.x];
  const cd* lm = log_mgf + (size_t)sp.slice * P;
  const double h3 = (grid[1].im - grid[0].im) / 3.0;
  double acc[1] = {0.0};
  for (int j = threadIdx.x; j < P; j += kFourierThreads) {
    const double wq = (j & 1) ? 4.0 : ((j == 0 || j == P - 1) ? 1.0 : 2.0);   // legacy Simpson, mgf_pricer.py:163-170
    const double dp = h3 * wq;
    const cd g = grid[j];
    cd w;
    if (mode == kModeQvar)
      w = mk(dp / M_PI) / (g * g);                              // (dp/pi)/(psi*psi), :344
    else if (mode == kModePdf)
      w = mk(dp / M_PI);                                        // dp/pi, :374-376
    else
      w = all_calls ? -(mk(dp / M_PI) / g) : (mk(dp / M_PI) / g);   // -/+ (dp/pi)/phi, :241-246
    const cd term = w * cexp_(sp.coef * g + lm[j]);
    if (term.re == term.re) acc[0] += term.re;
  }
  block_sum<1, kFourierThreads>(acc, red);
  if (threadIdx.x == 0) {
    const double S = acc[0];
    double r;
    if (mode == kModeQvar)
      r = fmax(sp.a * S / sp.b, 1e-10);                         // np.maximum(discfactor*option_price/ttm, 1e-10), :347
    else if (mode == kModePdf)
      r = S;
    else {
      const bool is_call = sp.type == B200SV_CALL;
      r = sp.a * ((is_call == (all_calls != 0)) ? S : 1.0 - S);  // :251-264
    }
    out[blockIdx.x] = r;
  }
}

// --------------------------------------------------------------------------------------------------------------------
// Hawkes jump-diffusion Fourier route (pricers/hawkes_jd_pricer.py:365-641): Riccati system for (a0, a_p, a_m) per transform point,
//   a0' = kappa_p theta_p a_p + kappa_m theta_m a_m + sigma^2 ((phi + 1) phi / 2 - psi)
//   a_p' = E_p(phi - beta1_p a_p - beta1_m a_m) - 1 - kappa_p a_p + comp_p phi        E(z) = exp(-shift z) / (1 + mean z): the jump-size MGF
//   a_m' = E_m(phi - beta2_p a_p - beta2_m a_m) - 1 - kappa_m a_m + comp_m phi        comp = exp(shift) / (1 - mean) - 1
// integrated per maturity by the SAME SciPy-RK45 clone as the LogSV coefficient ODEs (solve_ivp defaults, :636-639), A carried over the
// maturities (:396-416); log-MGF = a0 + a_p lambda_p + a_m lambda_m (:546).  One thread = one transform point.
// --------------------------------------------------------------------------------------------------------------------
struct HawkesMgfConsts {
  double sigma2, shift_p, mean_p, shift_m, mean_m, comp_p, comp_m;
  double kt_p, kt_m, kappa_p, kappa_m, beta1_p, beta1_m, beta2_p, beta2_m, lambda_p, lambda_m;
};

static HawkesMgfConsts make_hawkes_mgf_consts(const b200sv_hawkes_params& p) {
  HawkesMgfConsts c;
  c.sigma2 = p.sigma * p.sigma;
  c.shift_p = p.shift_p;
  c.mean_p = p.mean_p;
  c.shift_m = p.shift_m;
  c.mean_m = p.mean_m;
  c.comp_p = std::exp(p.shift_p) / (1.0 - p.mean_p) - 1.0;
  c.comp_m = std::exp(p.shift_m) / (1.0 - p.mean_m) - 1.0;
  c.kt_p = p.kappa_p * p.theta_p;
  c.kt_m = p.kappa_m * p.theta_m;
  c.kappa_p = p.kappa_p;
  c.kappa_m = p.kappa_m;
  c.beta1_p = p.beta1_p;
  c.beta1_m = p.beta1_m;
  c.beta2_p = p.beta2_p;
  c.beta2_m = p.beta2_m;
  c.lambda_p = p.lambda_p;
  c.lambda_m = p.lambda_m;
  return c;
}

struct HawkesRhsFn {
  const HawkesMgfConsts& c;
  cd phi, drift0;          // drift0 = sigma^2 ((phi + 1) phi / 2 - psi)
  __device__ __forceinline__ void operator()(const cd (&A)[3], cd (&out)[3]) const {
    const cd zp = (phi - c.beta1_p * A[1]) - c.beta1_m * A[2], zm = (phi - c.beta2_p * A[1]) - c.beta2_m * A[2];
    const cd jp = cexp_(-c.shift_p * zp) / (mk(1.0) + c.mean_p * zp) - mk(1.0);
    const cd jm = cexp_(-c.shift_m * zm) / (mk(1.0) + c.mean_m * zm) - mk(1.0);
    out[0] = (c.kt_p * A[1] + c.kt_m * A[2]) + drift0;
    out[1] = (jp - c.kappa_p * A[1]) + c.comp_p * phi;
    out[2] = (jm - c.kappa_m * A[2]) + c.comp_m * phi;
  }
};

// a_io: A(0) per point or nullptr (zeros); restart != 0: every maturity starts from A = 0 and integrates over ITS ttm (the risk-kernel
// normalisers, :498-509) instead of carrying A over the increments
template <int TPB>
__global__ void __launch_bounds__(TPB) hawkes_mgf_kernel(const cd* __restrict__ phi, const cd* __restrict__ psi, int P, int M,
                                                         const double* __restrict__ dtaus, HawkesMgfConsts c, const cd* __restrict__ a_in,
                                                         cd* __restrict__ a_out, cd* __restrict__ log_mgf, int restart, int* __restrict__ status) {
  __shared__ cd stage_smem[6 * 3 * TPB];
  const int p = blockIdx.x * TPB + threadIdx.x;
  if (p >= P) return;
  StageStore<3, TPB> K{stage_smem + threadIdx.x};
#pragma unroll
  for (int i = 0; i < 18; ++i) stage_smem[threadIdx.x + i * TPB] = mk(0.0);
  cd A[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) A[k] = a_in ? a_in[(size_t)p * 3 + k] : mk(0.0);
  const cd ph = phi[p], ps = psi ? psi[p] : mk(0.0);
  const HawkesRhsFn f{c, ph, c.sigma2 * (0.5 * ((ph + mk(1.0)) * ph) - ps)};
  int st = 0;
  for (int m = 0; m < M; ++m) {
    if (restart) {
#pragma unroll
      for (int k = 0; k < 3; ++k) A[k] = mk(0.0);
    }
    st |= rk45_generic<3, TPB>(A, dtaus[m], f, K, nullptr);
    if (a_out) {
#pragma unroll
      for (int k = 0; k < 3; ++k) a_out[((size_t)m * P + p) * 3 + k] = A[k];
    }
    log_mgf[(size_t)m * P + p] = (A[0] + A[1] * c.lambda_p) + A[2] * c.lambda_m;
  }
  if (status) status[p] = st;
}

// slice_pricer_with_mgf_grid_with_gamma (utils/mgf_pricer.py:273-320): general weights -(dp/pi) / ((phi + g + 1)(phi + g)) (its fast branch
// compares Re(phi) with +(1/2 + g) while the grid sits on -(1/2 + g), so it never runs), calls gamma_forward - n K^(1+g) S, puts K - n K^(1+g) S;
// no discount factor (both as in the reference).  spec.forward = forward, spec.discfactor = normalizer n, spec.ttm = gamma_forward.
__global__ void __launch_bounds__(kFourierThreads) fourier_gamma_kernel(const cd* __restrict__ log_mgf, const cd* __restrict__ phi, int P,
                                                                       const StrikeSpec* __restrict__ specs, double gamma,
                                                                       double* __restrict__ prices) {
  __shared__ double red[kFourierThreads / 32];
  const StrikeSpec sp = specs[blockIdx.x];
  const cd* lm = log_mgf + (size_t)sp.slice * P;
  const double x = log(sp.forward / sp.strike);
  const double h3 = (phi[1].im - phi[0].im) / 3.0;
  const bool fast = fabs(phi[0].re - (0.5 + gamma)) < 1e-10;
  double acc[1] = {0.0};
  for (int j = threadIdx.x; j < P; j += kFourierThreads) {
    const double wq = (j & 1) ? 4.0 : ((j == 0 || j == P - 1) ? 1.0 : 2.0);
    const double dp = h3 * wq;
    const cd ph = phi[j];
    const cd pg = ph + mk(gamma);
    const cd w = fast ? mk((dp / M_PI) / (ph.im * ph.im + 0.25)) : -(mk(dp / M_PI) / ((pg + mk(1.0)) * pg));
    const cd term = w * cexp_(lm[j] - x * ph);
    if (term.re == term.re) acc[0] += term.re;
  }
  block_sum<1, kFourierThreads>(acc, red);
  if (threadIdx.x == 0) {
    const double gk = pow(sp.strike, 1.0 + gamma);
    prices[blockIdx.x] = (sp.type == B200SV_CALL ? sp.ttm : sp.strike) - sp.discfactor * gk * acc[0];
  }
}

// --------------------------------------------------------------------------------------------------------------------
// host side
// --------------------------------------------------------------------------------------------------------------------
// Latency regime (few grid points in total): lane-parallel kernel; throughput regime (batches, the 40000-point psi grid): one thread per
// point.  B200SV_MGF_LANES=0/1 overrides the choice (A/B timing in tools/bench_mgf.py).
static bool use_lane_kernel(long long points) {
  static const int forced = [] {
    const char* e = getenv("B200SV_MGF_LANES");
    return e ? atoi(e) : -1;
  }();
  if (forced >= 0) return forced != 0;
  return points <= 8192;
}

template <int N>
static void launch_logsv_mgf(int tpb, int nb, cudaStream_t st, const cd* phi, const cd* psi, int P, int M, const ChainSpec* spec,
                             const cd* a_in, cd* a_out, cd* lm, double y, int* status, int B = 1, const double* yb = nullptr,
                             int phi_stride = 0) {
  if (use_lane_kernel((long long)P * B)) {
    constexpr int PPW = 32 / (N == 5 ? 8 : 4);
    const int per_block = PPW * kLaneWarpsPerBlock;
    logsv_mgf_lanes_kernel<N><<<dim3((P + per_block - 1) / per_block, B), 32 * kLaneWarpsPerBlock, 0, st>>>(phi, psi, P, M, spec, a_in, a_out, lm, y,
                                                                                                      status, yb, phi_stride);
    return;
  }
  static const bool set_major = [] {
    const char* e = getenv("B200SV_MGF_SET_MAJOR");      // A/B timing switch (tools/bench_calibration.py); default on
    return !e || atoi(e) != 0;
  }();
  const int smB = (B > 1 && set_major) ? B : 0;
  const dim3 grid = smB ? dim3((unsigned)(((long long)B * P + tpb - 1) / tpb), 1) : dim3(nb, B);
  switch (tpb) {
    case 4: logsv_mgf_kernel<N, 4><<<grid, 4, 0, st>>>(phi, psi, P, M, spec, a_in, a_out, lm, y, status, nullptr, yb, phi_stride, smB); break;
    case 8: logsv_mgf_kernel<N, 8><<<grid, 8, 0, st>>>(phi, psi, P, M, spec, a_in, a_out, lm, y, status, nullptr, yb, phi_stride, smB); break;
    case 16: logsv_mgf_kernel<N, 16><<<grid, 16, 0, st>>>(phi, psi, P, M, spec, a_in, a_out, lm, y, status, nullptr, yb, phi_stride, smB); break;
    case 32: logsv_mgf_kernel<N, 32><<<grid, 32, 0, st>>>(phi, psi, P, M, spec, a_in, a_out, lm, y, status, nullptr, yb, phi_stride, smB); break;
    default: logsv_mgf_kernel<N, 64><<<grid, 64, 0, st>>>(phi, psi, P, M, spec, a_in, a_out, lm, y, status, nullptr, yb, phi_stride, smB); break;
  }
}

// dense M / L / H of affine_expansion.py:139-184 from the row tables (parity entry b200sv_logsv_ode_terms)
template <int N>
__global__ void logsv_ode_terms_kernel(const cd* __restrict__ phi, const cd* __restrict__ psi, int P, LogsvModel m, cd* __restrict__ M_out,
                                       cd* __restrict__ L_out, cd* __restrict__ H_out) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const cd ph = phi[p], ps = psi ? psi[p] : mk(0.0);
  cd* Mo = M_out + (size_t)p * N * N * N;
  cd* Lo = L_out + (size_t)p * N * N;
  for (int i = 0; i < N * N * N; ++i) Mo[i] = mk(0.0);
  for (int i = 0; i < N * N; ++i) Lo[i] = mk(0.0);
  for (int k = 0; k < N; ++k) {
    const LaneRow<N> r = make_lane_row<N>(k, m, ph, ps);
    for (int t = 0; t < r.nq; ++t) {
      const int i = r.qi[t], j = r.qj[t];
      if (i == j) {
        Mo[(k * N + i) * N + i] = mk(r.q[t]);
      } else {          // the row tables carry off-diagonal pairs doubled: A_i A_j (M_ij + M_ji)
        Mo[(k * N + i) * N + j] = mk(0.5 * r.q[t]);
        Mo[(k * N + j) * N + i] = mk(0.5 * r.q[t]);
      }
    }
    for (int t = 0; t < r.nl; ++t) Lo[k * N + r.li[t]] = r.l[t];
    H_out[(size_t)p * N + k] = r.h;
  }
}

// func_rhs (affine_expansion.py:187-205) through the production right-hand side
template <int N>
__global__ void logsv_ode_rhs_kernel(const cd* __restrict__ phi, const cd* __restrict__ psi, int P, LogsvModel m, const cd* __restrict__ A_in,
                                     cd* __restrict__ rhs_out) {
  __shared__ cd coef_smem[14 * 64];
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  store_coef<64>(coef_smem + threadIdx.x, make_coef(m, phi[p], psi ? psi[p] : mk(0.0)));
  const CoefView<64> c{coef_smem + threadIdx.x};
  cd A[N], out[N];
#pragma unroll
  for (int k = 0; k < N; ++k) A[k] = A_in[(size_t)p * N + k];
  rhs<N, 64>(A, m, c, out);
#pragma unroll
  for (int k = 0; k < N; ++k) rhs_out[(size_t)p * N + k] = out[k];
}

// func_rhs with caller-supplied dense tensors (the reference signature): rhs[p][k] = A_p^T M[k] A_p + (L A_p)[k] + H[k]
__global__ void ode_rhs_dense_kernel(const cd* __restrict__ A, int P, int n, const cd* __restrict__ M, const cd* __restrict__ L,
                                     const cd* __restrict__ H, cd* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P * n) return;
  const int p = idx / n, k = idx % n;
  const cd* a = A + (size_t)p * n;
  cd acc = mk(0.0);
  for (int i = 0; i < n; ++i) {          // A^T M[k] A: row-by-row, as numpy's A0.T @ M[n_] @ A0 contracts (vector-matrix, then dot)
    cd row = mk(0.0);
    for (int j = 0; j < n; ++j) row = row + a[j] * M[((size_t)k * n + j) * n + i];
    acc = acc + row * a[i];
  }
  cd lin = mk(0.0);
  for (int j = 0; j < n; ++j) lin = lin + L[(size_t)k * n + j] * a[j];
  out[idx] = (acc + lin) + H[k];
}

// --------------------------------------------------------------------------------------------------------------------
// semi-analytic branch: solve_analytic_ode_for_a (pricers/logsv/affine_expansion.py:306-384), is_analytic=True
// --------------------------------------------------------------------------------------------------------------------
// The reference steps A' = A^T M A + L A + H on a business-day grid (nb_steps = ceil(260 dtau)): the linear part exactly -- through
// eig(L), v diag(exp(w dt)) v^-1 and v diag((exp(w dt) - 1)/w) v^-1 with the zero eigenvalue's entry set to 0 -- and the quadratic part by
// 10 unchecked fixed-point sweeps per step, quadratic term times plain dt; row 0 of the right-hand side is (H_0 + quad_0) dt.
// Here the two matrices are formed WITHOUT an eigendecomposition: v diag(e^{w dt}) v^-1 = expm(L dt) =: E, and because column 0 of L is zero
// (nothing depends on A_0) the null eigenvector is e_0, so rows 1.. of the second matrix equal rows 1.. of Psi = int_0^dt e^{L s} ds
// (the projector that the reference removes has only row 0, and row 0 is overwritten anyway).  E and Psi come from a degree-18 Taylor series
// of the scaled matrix and s doublings  Psi_{2h} = (I + E_h) Psi_h,  E_{2h} = E_h^2  -- 5x5 complex products in thread-local memory, once per
// (grid point, maturity).  Agreement with the reference's LAPACK route is limited by the conditioning of ITS eigenvector matrix (1e-10 on
// the goldens).  vol_backbone_eta is ignored on this branch as in the reference (:340-348: not passed to func_a_ode_quadratic_terms).
template <int N>
__device__ void cmat_mul(const cd (&A)[N][N], const cd (&B)[N][N], cd (&C)[N][N]) {
  for (int i = 0; i < N; ++i)
    for (int j = 0; j < N; ++j) {
      cd acc = mk(0.0);
      for (int k = 0; k < N; ++k) acc = acc + A[i][k] * B[k][j];
      C[i][j] = acc;
    }
}

template <int N>
__global__ void __launch_bounds__(64) logsv_mgf_analytic_kernel(const cd* __restrict__ phi, const cd* __restrict__ psi, int P, LogsvModel m, double dtau,
                                                                int year_days, const cd* __restrict__ a_in, cd* __restrict__ a_out,
                                                                cd* __restrict__ log_mgf, double y) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const cd ph = phi[p], ps = psi ? psi[p] : mk(0.0);
  const int nb_steps = (int)ceil((double)year_days * dtau);
  const double dt = dtau / (double)nb_steps;
  // rows of the system (the same tables the RK45 kernels integrate) -> dense L, H
  LaneRow<N> rows[N];
  cd L[N][N], H[N];
  for (int i = 0; i < N; ++i)
    for (int j = 0; j < N; ++j) L[i][j] = mk(0.0);
  double nrm = 0.0;
  for (int k = 0; k < N; ++k) {
    rows[k] = make_lane_row<N>(k, m, ph, ps);
    for (int t = 0; t < rows[k].nl; ++t) L[k][rows[k].li[t]] = rows[k].l[t];
    H[k] = rows[k].h;
    double rs = 0.0;
    for (int j = 0; j < N; ++j) rs += cabs_(L[k][j]);
    nrm = fmax(nrm, rs);
  }
  // scaling: ||L h||_inf <= 1/2
  int sq = 0;
  double h = dt;
  while (nrm * h > 0.5 && sq < 40) {
    h *= 0.5;
    ++sq;
  }
  cd X[N][N], E[N][N], Psi[N][N], T1[N][N], T2[N][N];
  for (int i = 0; i < N; ++i)
    for (int j = 0; j < N; ++j) {
      X[i][j] = h * L[i][j];
      E[i][j] = mk(i == j ? 1.0 : 0.0);
      Psi[i][j] = mk(i == j ? h : 0.0);
      T1[i][j] = E[i][j];                     // running term X^k / k!
    }
  for (int k = 1; k <= 18; ++k) {             // E = sum X^k/k!,  Psi = h sum X^k/(k+1)!
    cmat_mul<N>(T1, X, T2);
    for (int i = 0; i < N; ++i)
      for (int j = 0; j < N; ++j) {
        T1[i][j] = (1.0 / k) * T2[i][j];
        E[i][j] = E[i][j] + T1[i][j];
        Psi[i][j] = Psi[i][j] + (h / (k + 1)) * T1[i][j];
      }
  }
  for (int d = 0; d < sq; ++d) {              // doubling
    for (int i = 0; i < N; ++i)
      for (int j = 0; j < N; ++j) T1[i][j] = E[i][j] + mk(i == j ? 1.0 : 0.0);
    cmat_mul<N>(T1, Psi, T2);
    cmat_mul<N>(E, E, T1);
    for (int i = 0; i < N; ++i)
      for (int j = 0; j < N; ++j) {
        Psi[i][j] = T2[i][j];
        E[i][j] = T1[i][j];
      }
  }
  cd g[N];                                    // rows 1.. of (m_rhs @ H)
  for (int k = 0; k < N; ++k) {
    cd acc = mk(0.0);
    for (int j = 0; j < N; ++j) acc = acc + Psi[k][j] * H[j];
    g[k] = acc;
  }
  cd a[N], fp[N], q[N];
  for (int k = 0; k < N; ++k) a[k] = a_in[(size_t)p * N + k];
  for (int t = 0; t < nb_steps; ++t) {
    for (int k = 0; k < N; ++k) fp[k] = a[k];
    cd Ea[N];
    for (int k = 0; k < N; ++k) {
      cd acc = mk(0.0);
      for (int j = 0; j < N; ++j) acc = acc + E[k][j] * a[j];
      Ea[k] = acc;
    }
    for (int it = 0; it < 10; ++it) {         // nfp = 10, no convergence test (:365)
      for (int k = 0; k < N; ++k) {
        cd acc = mk(0.0);
        for (int u = 0; u < rows[k].nq; ++u) acc = acc + rows[k].q[u] * (fp[rows[k].qi[u]] * fp[rows[k].qj[u]]);
        q[k] = acc;
      }
      fp[0] = Ea[0] + dt * (H[0] + q[0]);
      for (int k = 1; k < N; ++k) fp[k] = Ea[k] + (g[k] + dt * q[k]);
    }
    for (int k = 0; k < N; ++k) a[k] = fp[k];
  }
  double yk = 1.0;
  cd lm = mk(0.0);
  for (int k = 0; k < N; ++k) {
    a_out[(size_t)p * N + k] = a[k];
    lm = lm + yk * a[k];
    yk *= y;
  }
  log_mgf[p] = lm;
}

// --------------------------------------------------------------------------------------------------------------------
// stiff branch: solve_ivp(method="BDF", jac=func_rhs_jac) as used by solve_ode_for_a(is_stiff_solver=True) (affine_expansion.py:229-303)
// --------------------------------------------------------------------------------------------------------------------
// A clone of the CONTROL LAW of scipy.integrate.BDF (scipy 1.18.1, scipy/integrate/_ivp/bdf.py:14-60, 186-230, 317-455; select_initial_step
// with order 1, common.py:68-134; rtol 1e-3 / atol 1e-6): variable order 1..5 NDF with quasi-constant step size, the differences array D and
// its rescaling matrices (change_D), simplified Newton with at most 4 iterations on an LU of I - c J that is KEPT across steps and across
// error rejections (bdf.py resets it only when the step size changes for other reasons), Jacobian refreshed only after a failed Newton
// solve, order selection from the three error norms after order + 1 equal steps.  Parity with the reference means reproducing its accepted
// steps, so every branch of the step routine is mirrored; floating-point differences (LAPACK's blocked zgetrf / BLAS dot products vs the
// scalar loops here) stay at the 1e-15 level because the decisions are thresholds on norms (tests: 1e-10 against the reference goldens).
// One thread = one grid point; D (8 x N complex), J and LU live in thread-local memory -- this is the reference's non-default branch, 1000
// independent stiff solves of ~30 steps each, not a throughput path.
template <int N>
struct BdfState {
  cd D[8][N];
  cd J[N][N], LU[N][N];
  int piv[N];
  bool lu_valid;
};

__device__ __forceinline__ double cabs1(cd a) { return fabs(a.re) + fabs(a.im); }     // LAPACK izamax's magnitude

template <int N>
__device__ void bdf_lu_factor(BdfState<N>& s, double c) {             // LU of I - c J, partial pivoting (zgetrf semantics)
  for (int i = 0; i < N; ++i)
    for (int j = 0; j < N; ++j) s.LU[i][j] = mk(i == j ? 1.0 : 0.0) - c * s.J[i][j];
  for (int k = 0; k < N; ++k) {
    int p = k;
    double best = cabs1(s.LU[k][k]);
    for (int i = k + 1; i < N; ++i) {
      const double v = cabs1(s.LU[i][k]);
      if (v > best) {
        best = v;
        p = i;
      }
    }
    s.piv[k] = p;
    if (p != k)
      for (int j = 0; j < N; ++j) {
        const cd t = s.LU[k][j];
        s.LU[k][j] = s.LU[p][j];
        s.LU[p][j] = t;
      }
    const cd inv = mk(1.0) / s.LU[k][k];
    for (int i = k + 1; i < N; ++i) {
      s.LU[i][k] = s.LU[i][k] * inv;
      for (int j = k + 1; j < N; ++j) s.LU[i][j] = s.LU[i][j] - s.LU[i][k] * s.LU[k][j];
    }
  }
  s.lu_valid = true;
}

template <int N>
__device__ void bdf_lu_solve(const BdfState<N>& s, cd (&b)[N]) {
  for (int k = 0; k < N; ++k) {
    const int p = s.piv[k];
    if (p != k) {
      const cd t = b[k];
      b[k] = b[p];
      b[p] = t;
    }
  }
  for (int i = 1; i < N; ++i)
    for (int j = 0; j < i; ++j) b[i] = b[i] - s.LU[i][j] * b[j];
  for (int i = N - 1; i >= 0; --i) {
    for (int j = i + 1; j < N; ++j) b[i] = b[i] - s.LU[i][j] * b[j];
    b[i] = b[i] / s.LU[i][i];
  }
}

// func_rhs_jac (affine_expansion.py:208-225): J = 2 M[k] A + L, from the row tables
template <int N>
__device__ void bdf_jacobian(BdfState<N>& s, const cd (&A)[N], const LogsvModel& m, cd phi, cd psi) {
  for (int k = 0; k < N; ++k) {
    for (int j = 0; j < N; ++j) s.J[k][j] = mk(0.0);
    const LaneRow<N> r = make_lane_row<N>(k, m, phi, psi);
    for (int t = 0; t < r.nq; ++t) {
      const int i = r.qi[t], j = r.qj[t];
      if (i == j) {
        s.J[k][i] = s.J[k][i] + (2.0 * r.q[t]) * A[i];
      } else {                       // the tables carry off-diagonal pairs doubled: q A_i A_j with q = M_ij + M_ji
        s.J[k][i] = s.J[k][i] + r.q[t] * A[j];
        s.J[k][j] = s.J[k][j] + r.q[t] * A[i];
      }
    }
    for (int t = 0; t < r.nl; ++t) s.J[k][r.li[t]] = s.J[k][r.li[t]] + r.l[t];
  }
}

// change_D (bdf.py:28-33): D[:order+1] <- (R U)^T D[:order+1],  R = compute_R(order, factor), U = compute_R(order, 1)
template <int N>
__device__ void bdf_change_D(BdfState<N>& s, int order, double factor) {
  double R[6][6], U[6][6], RU[6][6];
  for (int j = 0; j <= order; ++j) {
    R[0][j] = 1.0;
    U[0][j] = 1.0;
  }
  for (int i = 1; i <= order; ++i) {
    R[i][0] = 0.0;                  // M[i][0] = 0 => cumprod is 0 from row 1 on
    U[i][0] = 0.0;
    for (int j = 1; j <= order; ++j) {
      R[i][j] = R[i - 1][j] * (((double)(i - 1) - factor * (double)j) / (double)i);
      U[i][j] = U[i - 1][j] * (((double)(i - 1) - (double)j) / (double)i);
    }
  }
  for (int i = 0; i <= order; ++i)
    for (int j = 0; j <= order; ++j) {
      double acc = 0.0;
      for (int k = 0; k <= order; ++k) acc += R[i][k] * U[k][j];
      RU[i][j] = acc;
    }
  cd Dn[6][N];
  for (int i = 0; i <= order; ++i)
    for (int c = 0; c < N; ++c) {
      cd acc = mk(0.0);
      for (int k = 0; k <= order; ++k) acc = acc + RU[k][i] * s.D[k][c];
      Dn[i][c] = acc;
    }
  for (int i = 0; i <= order; ++i)
    for (int c = 0; c < N; ++c) s.D[i][c] = Dn[i][c];
}

template <int N>
__device__ double bdf_norm_scaled(const cd (&v)[N], const double (&scale)[N]) {       // norm(v / scale) = ||.||_2 / sqrt(n)
  double acc = 0.0;
  for (int k = 0; k < N; ++k) {
    const double re = v[k].re / scale[k], im = v[k].im / scale[k];
    acc += re * re + im * im;
  }
  return sqrt(acc) / sqrt((double)N);
}

// returns 0 ok, 1 step size underflow (TOO_SMALL_STEP: the reference keeps the last accepted state)
template <int N, int TPB>
__device__ int bdf_integrate(cd (&y)[N], double T, const LogsvModel& m, const CoefView<TPB>& c, cd phi, cd psi, BdfState<N>& s) {
  const double gamma[6] = {0.0, 1.0, 1.5, 1.5 + 1.0 / 3.0, 1.5 + 1.0 / 3.0 + 0.25, 1.5 + 1.0 / 3.0 + 0.25 + 0.2};
  const double kappa[6] = {0.0, -0.1850, -1.0 / 9.0, -0.0823, -0.0415, 0.0};
  double alpha[6], error_const[7];
  for (int i = 0; i < 6; ++i) {
    alpha[i] = (1.0 - kappa[i]) * gamma[i];
    error_const[i] = kappa[i] * gamma[i] + 1.0 / (double)(i + 1);
  }
  const double newton_tol = 0.03;       // max(10 EPS / rtol, min(0.03, sqrt(rtol)))
  cd f[N];
  rhs<N, TPB>(y, m, c, f);
  double h_abs;
  {  // select_initial_step(order = 1)
    double scale[N];
    for (int k = 0; k < N; ++k) scale[k] = kAtol + cmod(y[k]) * kRtol;
    const double d0 = bdf_norm_scaled<N>(y, scale), d1 = bdf_norm_scaled<N>(f, scale);
    double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
    h0 = fmin(h0, T);
    cd y1[N], f1[N];
    for (int k = 0; k < N; ++k) y1[k] = y[k] + h0 * f[k];
    rhs<N, TPB>(y1, m, c, f1);
    for (int k = 0; k < N; ++k) f1[k] = f1[k] - f[k];
    const double d2 = bdf_norm_scaled<N>(f1, scale) / h0;
    const double h1 = (d1 <= 1e-15 && d2 <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : sqrt(0.01 / fmax(d1, d2));
    h_abs = fmin(fmin(100.0 * h0, h1), T);
  }
  bdf_jacobian<N>(s, y, m, phi, psi);
  for (int i = 0; i < 8; ++i)
    for (int k = 0; k < N; ++k) s.D[i][k] = mk(0.0);
  for (int k = 0; k < N; ++k) {
    s.D[0][k] = y[k];
    s.D[1][k] = h_abs * f[k];
  }
  int order = 1, n_equal_steps = 0;
  s.lu_valid = false;
  double t = 0.0;
  for (int guard = 0; t < T && guard < 100000; ++guard) {
    // ---- _step_impl (bdf.py:317-455)
    const double min_step = 10.0 * (__longlong_as_double(__double_as_longlong(t) + 1) - t);
    if (h_abs < min_step) {
      bdf_change_D<N>(s, order, min_step / h_abs);
      h_abs = min_step;
      n_equal_steps = 0;
    }
    bool current_jac = false;
    bool accepted = false;
    double t_new = t, safety = 0.0, error_norm = 0.0;
    double scale[N];
    cd y_new[N], d[N];
    while (!accepted) {
      if (h_abs < min_step) return 1;
      t_new = t + h_abs;
      if (t_new - T > 0.0) {
        t_new = T;
        bdf_change_D<N>(s, order, fabs(t_new - t) / h_abs);
        n_equal_steps = 0;
        s.lu_valid = false;
      }
      const double h = t_new - t;
      h_abs = fabs(h);
      cd y_predict[N], psi_v[N];
      for (int k = 0; k < N; ++k) {
        cd acc = s.D[0][k];
        for (int i = 1; i <= order; ++i) acc = acc + s.D[i][k];
        y_predict[k] = acc;
        scale[k] = kAtol + kRtol * cmod(acc);
        cd ps = mk(0.0);
        for (int i = 1; i <= order; ++i) ps = ps + gamma[i] * s.D[i][k];
        psi_v[k] = mk(ps.re / alpha[order], ps.im / alpha[order]);      // numpy divides (dot(...) / alpha[order]): no reciprocal multiply
      }
      const double cc = h / alpha[order];
      bool converged = false;
      int n_iter = 0;
      while (!converged) {
        if (!s.lu_valid) bdf_lu_factor<N>(s, cc);
        // ---- solve_bdf_system (bdf.py:36-72)
        for (int k = 0; k < N; ++k) {
          d[k] = mk(0.0);
          y_new[k] = y_predict[k];
        }
        double dy_norm_old = -1.0;
        for (int k_it = 0; k_it < 4; ++k_it) {
          cd fn[N];
          rhs<N, TPB>(y_new, m, c, fn);
          bool finite = true;
          for (int k = 0; k < N; ++k) finite = finite && isfinite(fn[k].re) && isfinite(fn[k].im);
          if (!finite) break;
          cd dy[N];
          for (int k = 0; k < N; ++k) dy[k] = (cc * fn[k] - psi_v[k]) - d[k];
          bdf_lu_solve<N>(s, dy);
          const double dy_norm = bdf_norm_scaled<N>(dy, scale);
          const bool have_rate = dy_norm_old >= 0.0;
          const double rate = have_rate ? dy_norm / dy_norm_old : 0.0;
          if (have_rate && (rate >= 1.0 || pow(rate, (double)(4 - k_it)) / (1.0 - rate) * dy_norm > newton_tol)) break;
          for (int k = 0; k < N; ++k) {
            y_new[k] = y_new[k] + dy[k];
            d[k] = d[k] + dy[k];
          }
          n_iter = k_it + 1;
          if (dy_norm == 0.0 || (have_rate && rate / (1.0 - rate) * dy_norm < newton_tol)) {
            converged = true;
            break;
          }
          dy_norm_old = dy_norm;
        }
        if (!converged) {
          if (current_jac) break;
          bdf_jacobian<N>(s, y_predict, m, phi, psi);
          s.lu_valid = false;
          current_jac = true;
        }
      }
      if (!converged) {
        h_abs *= 0.5;
        bdf_change_D<N>(s, order, 0.5);
        n_equal_steps = 0;
        s.lu_valid = false;
        continue;
      }
      safety = 0.9 * (2.0 * 4.0 + 1.0) / (2.0 * 4.0 + (double)n_iter);
      for (int k = 0; k < N; ++k) scale[k] = kAtol + kRtol * cmod(y_new[k]);
      cd err[N];
      for (int k = 0; k < N; ++k) err[k] = error_const[order] * d[k];
      error_norm = bdf_norm_scaled<N>(err, scale);
      if (error_norm > 1.0) {
        const double factor = fmax(0.2, safety * pow(error_norm, -1.0 / (double)(order + 1)));
        h_abs *= factor;
        bdf_change_D<N>(s, order, factor);
        n_equal_steps = 0;            // LU is deliberately NOT invalidated here (bdf.py:398-403)
      } else {
        accepted = true;
      }
    }
    ++n_equal_steps;
    t = t_new;
    for (int k = 0; k < N; ++k) {
      y[k] = y_new[k];
      s.D[order + 2][k] = d[k] - s.D[order + 1][k];
      s.D[order + 1][k] = d[k];
    }
    for (int i = order; i >= 0; --i)
      for (int k = 0; k < N; ++k) s.D[i][k] = s.D[i][k] + s.D[i + 1][k];
    if (n_equal_steps < order + 1) continue;
    double en[3];
    {
      cd e[N];
      if (order > 1) {
        for (int k = 0; k < N; ++k) e[k] = error_const[order - 1] * s.D[order][k];
        en[0] = bdf_norm_scaled<N>(e, scale);
      } else {
        en[0] = INFINITY;
      }
      en[1] = error_norm;
      if (order < 5) {
        for (int k = 0; k < N; ++k) e[k] = error_const[order + 1] * s.D[order + 2][k];
        en[2] = bdf_norm_scaled<N>(e, scale);
      } else {
        en[2] = INFINITY;
      }
    }
    double factors[3], best = -1.0;
    int arg = 0;
    for (int i = 0; i < 3; ++i) {
      factors[i] = pow(en[i], -1.0 / (double)(order + i));     // 0 -> inf, inf -> 0 (numpy with divide='ignore')
      if (factors[i] > best) {                                   // np.argmax: first maximum
        best = factors[i];
        arg = i;
      }
    }
    order += arg - 1;
    const double factor = fmin(10.0, safety * best);
    h_abs *= factor;
    bdf_change_D<N>(s, order, factor);
    n_equal_steps = 0;
    s.lu_valid = false;
  }
  return 0;
}

template <int N>
__global__ void __launch_bounds__(64) logsv_mgf_bdf_kernel(const cd* __restrict__ phi, const cd* __restrict__ psi, int P, LogsvModel m, double dtau,
                                                           const cd* __restrict__ a_in, cd* __restrict__ a_out, cd* __restrict__ log_mgf, double y,
                                                           int* __restrict__ status) {
  __shared__ cd coef_smem[14 * 64];
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const cd ph = phi[p], ps = psi ? psi[p] : mk(0.0);
  store_coef<64>(coef_smem + threadIdx.x, make_coef(m, ph, ps));
  const CoefView<64> c{coef_smem + threadIdx.x};
  cd A[N];
  for (int k = 0; k < N; ++k) A[k] = a_in[(size_t)p * N + k];
  BdfState<N> st;
  const int rc = bdf_integrate<N, 64>(A, dtau, m, c, ph, ps, st);
  if (status) status[p] = rc;
  double yk = 1.0;
  cd lm = mk(0.0);
  for (int k = 0; k < N; ++k) {
    a_out[(size_t)p * N + k] = A[k];
    lm = lm + yk * A[k];
    yk *= y;
  }
  log_mgf[p] = lm;
}

static int mgf_block_threads(int P) {
  int t = 4;
  while (t < 64 && t * 148 < P) t <<= 1;
  return t;
}

// np.linspace(0, stop, P): y[i] = i*step, step = stop/(P-1), last = stop; phi = re + 1j*p (utils/mgf_pricer.py:22-33)
static void build_phi(double vol_scaler, bool spot, int P, std::vector<double>& phi) {
  phi.resize(2 * (size_t)P);
  const double stop = 5.6 / vol_scaler, step = stop / (double)(P - 1);
  for (int i = 0; i < P; ++i) {
    phi[2 * i] = spot ? -0.5 : 0.5;
    phi[2 * i + 1] = (double)i * step;
  }
  phi[2 * (size_t)(P - 1) + 1] = stop;
}

// re + 1j*linspace(0, stop, P)  (get_psi_grid: -0.5 + 1j*linspace(0, 4000, 40000), utils/mgf_pricer.py:37-47)
static void build_grid(double re, double stop, int P, std::vector<double>& g) {
  g.resize(2 * (size_t)P);
  const double step = stop / (double)(P - 1);
  for (int i = 0; i < P; ++i) {
    g[2 * i] = re;
    g[2 * i + 1] = (double)i * step;
  }
  g[2 * (size_t)(P - 1) + 1] = stop;
}

static int check_qvar_types(const int8_t* types, int n) {
  for (int j = 0; j < n; ++j)
    if (types[j] != B200SV_CALL) return fail(-5, "not implemented");      // utils/mgf_pricer.py:349-358: only 'C'
  return 0;
}

static int check_fourier_types(const int8_t* types, int n, bool spot) {
  for (int j = 0; j < n; ++j) {
    if (types[j] < 0 || types[j] > 3) return fail(-5, "not implemented");
    // MMA measure rejects inverse payoffs (utils/mgf_pricer.py:206-212); the inverse measure accepts C == IC, P == IP (:214-217)
    if (spot && types[j] >= 2) return fail(-5, "not implemented");
  }
  return 0;
}

static bool all_half_re(const double* phi, int P) {
  for (int i = 0; i < P; ++i)
    if (std::fabs(phi[2 * i]) != 0.5) return false;
  return true;
}

}  // namespace b200sv

using namespace b200sv;

extern "C" {

int b200sv_logsv_price_chain(const b200sv_logsv_params* params, int M, const double* ttms, const double* forwards,
                             const double* discfactors, const double* etas, const int* offsets, const double* strikes,
                             const int8_t* types, int is_spot_measure, int variable_type, int expansion_order,
                             double vol_scaler, int P, double* prices_out, double* a_out, double* log_mgf_out) {
  B200SV_REQUIRE(params && ttms && forwards && discfactors && offsets && prices_out, "null pointer");
  if (variable_type != B200SV_LOG_RETURN && variable_type != B200SV_Q_VAR) return fail(-4, "variable_type not implemented");   // logsv_pricer.py:733-734
  const bool qvar = variable_type == B200SV_Q_VAR;
  if (P <= 0) P = qvar ? 40000 : 1000;                                     // utils/mgf_pricer.py:13, :44
  B200SV_REQUIRE(M >= 1 && P >= 3, "M >= 1, P >= 3");
  if (expansion_order != B200SV_ORDER_FIRST && expansion_order != B200SV_ORDER_SECOND)
    return fail(-4, "expansion_order not implemented");                    // affine_expansion.py:680-681
  const bool spot = is_spot_measure != 0;
  const int Jtot = offsets[M] - offsets[0];
  if (int rc = qvar ? check_qvar_types(types + offsets[0], Jtot) : check_fourier_types(types + offsets[0], Jtot, spot)) return rc;
  double t0 = 0.0, tmin = ttms[0];
  for (int m = 0; m < M; ++m) {
    B200SV_REQUIRE(ttms[m] > t0, "ttms must be positive and strictly increasing");
    t0 = ttms[m];
    tmin = std::min(tmin, ttms[m]);
  }
  if (!(vol_scaler > 0.0)) vol_scaler = params->sigma0 * std::sqrt(std::min(tmin, 0.5 / 12.0));   // logsv_pricer.py:664-666
  const int N = expansion_order == B200SV_ORDER_FIRST ? 3 : 5;
  std::vector<double> phi, psi;
  if (!qvar) {
    build_phi(vol_scaler, spot, P, phi);
  } else {                                                                 // utils/mgf_pricer.py:79-85: psi grid, phi = 0 (MMA) | 1 (inverse)
    build_grid(-0.5, 4000.0, P, psi);
    phi.assign(2 * (size_t)P, 0.0);
    if (!spot)
      for (int i = 0; i < P; ++i) phi[2 * i] = 1.0;
  }
  std::vector<ChainSpec> spec(M);
  t0 = 0.0;
  for (int m = 0; m < M; ++m) {
    spec[m].dtau = ttms[m] - t0;
    spec[m].model = make_model(*params, etas ? etas[m] : 1.0, spot);
    t0 = ttms[m];
  }
  std::vector<StrikeSpec> ss(std::max(Jtot, 1));
  std::vector<SumSpec> qs(std::max(Jtot, 1));
  for (int m = 0; m < M; ++m)
    for (int j = offsets[m]; j < offsets[m + 1]; ++j) {
      B200SV_REQUIRE(strikes[j] > 0.0, "strikes must be positive");
      ss[j - offsets[0]] = StrikeSpec{strikes[j], forwards[m], discfactors[m], (int)types[j], m, ttms[m], 0};
      qs[j - offsets[0]] = SumSpec{strikes[j] * ttms[m], discfactors[m], ttms[m], (int)types[j], m};
    }
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_phi(st), d_psi(st), d_a(st), d_lm(st);
    DevBuf<ChainSpec> d_spec(st);
    DevBuf<StrikeSpec> d_ss(st);      // the StrikeSpecs, or the (smaller) SumSpecs for Q_VAR
    DevBuf<double> d_pr(st);
    DevBuf<int> d_stat(st);
    B200SV_CUDA(d_phi.upload(phi.data(), P));
    B200SV_CUDA(qvar ? d_psi.upload(psi.data(), P) : d_psi.alloc(P));
    B200SV_CUDA(d_spec.upload(spec.data(), M));
    B200SV_CUDA(d_a.alloc((size_t)M * P * N));
    B200SV_CUDA(d_lm.alloc((size_t)M * P));
    B200SV_CUDA(d_ss.alloc(ss.size()));
    B200SV_CUDA(d_pr.alloc(ss.size()));
    B200SV_CUDA(d_stat.alloc(P));
    B200SV_CUDA(qvar ? cudaMemcpyAsync(d_ss.p, qs.data(), sizeof(SumSpec) * qs.size(), cudaMemcpyHostToDevice, st)
                     : cudaMemcpyAsync(d_ss.p, ss.data(), sizeof(StrikeSpec) * ss.size(), cudaMemcpyHostToDevice, st));
    const int tpb = mgf_block_threads(P), nb = (P + tpb - 1) / tpb;
    const double y = params->sigma0 - params->theta;
    const cd* dpsi = qvar ? d_psi.p : nullptr;
    if (N == 5)
      launch_logsv_mgf<5>(tpb, nb, st, d_phi.p, dpsi, P, M, d_spec.p, nullptr, d_a.p, d_lm.p, y, d_stat.p);
    else
      launch_logsv_mgf<3>(tpb, nb, st, d_phi.p, dpsi, P, M, d_spec.p, nullptr, d_a.p, d_lm.p, y, d_stat.p);
    if (int rc = launched("logsv_mgf_kernel")) return rc;
    if (Jtot > 0) {
      if (qvar)
        fourier_sum_kernel<<<Jtot, kFourierThreads, 0, st>>>(d_lm.p, d_psi.p, P, (const SumSpec*)d_ss.p, kModeQvar, 0, d_pr.p);
      else
        fourier_vanilla_kernel<<<Jtot, kFourierThreads, 0, st>>>(d_lm.p, d_phi.p, P, d_ss.p, spot ? 1 : 0, 1, d_pr.p);
      if (int rc = launched("fourier_vanilla_kernel")) return rc;
      B200SV_CUDA(cudaMemcpyAsync(prices_out, d_pr.p, sizeof(double) * Jtot, cudaMemcpyDeviceToHost, st));
    }
    if (a_out) B200SV_CUDA(cudaMemcpyAsync(a_out, d_a.p, sizeof(cd) * (size_t)M * P * N, cudaMemcpyDeviceToHost, st));
    if (log_mgf_out) B200SV_CUDA(cudaMemcpyAsync(log_mgf_out, d_lm.p, sizeof(cd) * (size_t)M * P, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

int b200sv_heston_price_chain(const b200sv_heston_params* params, int M, const double* ttms, const double* forwards,
                              const double* discfactors, const int* offsets, const double* strikes, const int8_t* types,
                              int variable_type, double vol_scaler, int P, double* prices_out, double* log_mgf_out) {
  B200SV_REQUIRE(params && ttms && forwards && discfactors && offsets && prices_out, "null pointer");
  if (variable_type != B200SV_LOG_RETURN && variable_type != B200SV_Q_VAR) return fail(-4, "variable_type not implemented");   // heston_pricer.py:276-277
  const bool qvar = variable_type == B200SV_Q_VAR;
  if (P <= 0) P = qvar ? 40000 : 1000;
  B200SV_REQUIRE(M >= 1 && P >= 3, "M >= 1, P >= 3");
  const int Jtot = offsets[M] - offsets[0];
  if (int rc = qvar ? check_qvar_types(types + offsets[0], Jtot) : check_fourier_types(types + offsets[0], Jtot, true)) return rc;
  if (!(vol_scaler > 0.0)) vol_scaler = std::min(0.3, std::sqrt(params->v0 * ttms[0]));   // heston_pricer.py:234-235
  std::vector<double> phi, psi;
  if (!qvar) {
    build_phi(vol_scaler, true, P, phi);
  } else {
    build_grid(-0.5, 4000.0, P, psi);
    phi.assign(2 * (size_t)P, 0.0);
  }
  std::vector<double> dtaus(M);
  double t0 = 0.0;
  for (int m = 0; m < M; ++m) {
    B200SV_REQUIRE(ttms[m] > t0, "ttms must be positive and strictly increasing");
    dtaus[m] = ttms[m] - t0;
    t0 = ttms[m];
  }
  std::vector<StrikeSpec> ss(std::max(Jtot, 1));
  std::vector<SumSpec> qs(std::max(Jtot, 1));
  for (int m = 0; m < M; ++m)
    for (int j = offsets[m]; j < offsets[m + 1]; ++j) {
      B200SV_REQUIRE(strikes[j] > 0.0, "strikes must be positive");
      ss[j - offsets[0]] = StrikeSpec{strikes[j], forwards[m], discfactors[m], (int)types[j], m, ttms[m], 0};
      qs[j - offsets[0]] = SumSpec{strikes[j] * ttms[m], discfactors[m], ttms[m], (int)types[j], m};
    }
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_phi(st), d_psi(st), d_lm(st);
    DevBuf<double> d_dt(st), d_pr(st);
    DevBuf<StrikeSpec> d_ss(st);      // the StrikeSpecs, or the (smaller) SumSpecs for Q_VAR
    B200SV_CUDA(d_phi.upload(phi.data(), P));
    B200SV_CUDA(qvar ? d_psi.upload(psi.data(), P) : d_psi.alloc(P));
    B200SV_CUDA(d_dt.upload(dtaus.data(), M));
    B200SV_CUDA(d_lm.alloc((size_t)M * P));
    B200SV_CUDA(d_ss.alloc(ss.size()));
    B200SV_CUDA(d_pr.alloc(ss.size()));
    B200SV_CUDA(qvar ? cudaMemcpyAsync(d_ss.p, qs.data(), sizeof(SumSpec) * qs.size(), cudaMemcpyHostToDevice, st)
                     : cudaMemcpyAsync(d_ss.p, ss.data(), sizeof(StrikeSpec) * ss.size(), cudaMemcpyHostToDevice, st));
    const int tpb = mgf_block_threads(P), nb = (P + tpb - 1) / tpb;
    heston_mgf_kernel<<<nb, tpb, 0, st>>>(d_phi.p, qvar ? d_psi.p : nullptr, P, M, d_dt.p, *params, nullptr, nullptr, nullptr, nullptr, d_lm.p);
    if (int rc = launched("heston_mgf_kernel")) return rc;
    if (Jtot > 0) {
      if (qvar)
        fourier_sum_kernel<<<Jtot, kFourierThreads, 0, st>>>(d_lm.p, d_psi.p, P, (const SumSpec*)d_ss.p, kModeQvar, 0, d_pr.p);
      else
        fourier_vanilla_kernel<<<Jtot, kFourierThreads, 0, st>>>(d_lm.p, d_phi.p, P, d_ss.p, 1, 1, d_pr.p);
      if (int rc = launched("fourier_vanilla_kernel")) return rc;
      B200SV_CUDA(cudaMemcpyAsync(prices_out, d_pr.p, sizeof(double) * Jtot, cudaMemcpyDeviceToHost, st));
    }
    if (log_mgf_out) B200SV_CUDA(cudaMemcpyAsync(log_mgf_out, d_lm.p, sizeof(cd) * (size_t)M * P, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

/* ---- batched chain pricers: B parameter sets on one chain in one pass (calibration objective + its finite-difference gradient) ---- */
static int chain_batch_common(int B, int M, const double* ttms, const double* forwards, const double* discfactors, const int* offsets,
                              const double* strikes, const int8_t* types, bool spot, int P, std::vector<double>& dtaus,
                              std::vector<StrikeSpec>& ss, bool per_set_grid) {
  B200SV_REQUIRE(B >= 1 && B <= 65535 && M >= 1 && P >= 3, "1 <= B <= 65535, M >= 1, P >= 3");
  const int Jtot = offsets[M] - offsets[0];
  B200SV_REQUIRE(Jtot >= 1, "the chain has no strikes");
  if (int rc = check_fourier_types(types + offsets[0], Jtot, spot)) return rc;
  dtaus.resize(M);
  double t0 = 0.0;
  for (int m = 0; m < M; ++m) {
    B200SV_REQUIRE(ttms[m] > t0, "ttms must be positive and strictly increasing");
    dtaus[m] = ttms[m] - t0;
    t0 = ttms[m];
  }
  ss.resize((size_t)B * Jtot);
  for (int b = 0; b < B; ++b)
    for (int m = 0; m < M; ++m)
      for (int j = offsets[m]; j < offsets[m + 1]; ++j) {
        B200SV_REQUIRE(strikes[j] > 0.0, "strikes must be positive");
        ss[(size_t)b * Jtot + (j - offsets[0])] = StrikeSpec{strikes[j], forwards[m], discfactors[m], (int)types[j], b * M + m, ttms[m], per_set_grid ? b : 0};
      }
  return 0;
}

int b200sv_logsv_price_chain_batch(const b200sv_logsv_params* params, int B, int M, const double* ttms, const double* forwards,
                                   const double* discfactors, const double* etas, const int* offsets, const double* strikes,
                                   const int8_t* types, int is_spot_measure, int expansion_order, double vol_scaler, int P,
                                   double* prices_out, double* ivols_out) {
  B200SV_REQUIRE(params && ttms && forwards && discfactors && offsets && strikes && types && prices_out, "null pointer");
  if (P <= 0) P = 1000;
  if (expansion_order != B200SV_ORDER_FIRST && expansion_order != B200SV_ORDER_SECOND) return fail(-4, "expansion_order not implemented");
  const bool spot = is_spot_measure != 0;
  const bool per_set_grid = !(vol_scaler > 0.0);      // default scaler depends on sigma0 of each set (logsv_pricer.py:664-666)
  std::vector<double> dtaus;
  std::vector<StrikeSpec> ss;
  if (int rc = chain_batch_common(B, M, ttms, forwards, discfactors, offsets, strikes, types, spot, P, dtaus, ss, per_set_grid)) return rc;
  const int Jtot = offsets[M] - offsets[0], N = expansion_order == B200SV_ORDER_FIRST ? 3 : 5;
  const double tmin = *std::min_element(ttms, ttms + M);
  const int G = per_set_grid ? B : 1;
  std::vector<double> phi, one;
  for (int g = 0; g < G; ++g) {
    build_phi(per_set_grid ? params[g].sigma0 * std::sqrt(std::min(tmin, 0.5 / 12.0)) : vol_scaler, spot, P, one);
    phi.insert(phi.end(), one.begin(), one.end());
  }
  std::vector<ChainSpec> spec((size_t)B * M);
  std::vector<double> yb(B);
  for (int b = 0; b < B; ++b) {
    yb[b] = params[b].sigma0 - params[b].theta;
    for (int m = 0; m < M; ++m) spec[(size_t)b * M + m] = ChainSpec{dtaus[m], make_model(params[b], etas ? etas[(size_t)b * M + m] : 1.0, spot)};
  }
  const size_t nq = (size_t)B * Jtot;
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_phi(st), d_a(st), d_lm(st);
    DevBuf<ChainSpec> d_spec(st);
    DevBuf<double> d_y(st), d_pr(st), d_iv(st);
    DevBuf<StrikeSpec> d_ss(st);
    B200SV_CUDA(d_phi.upload(phi.data(), (size_t)G * P));
    B200SV_CUDA(d_spec.upload(spec.data(), spec.size()));
    B200SV_CUDA(d_y.upload(yb.data(), B));
    B200SV_CUDA(d_a.alloc((size_t)B * M * P * N));
    B200SV_CUDA(d_lm.alloc((size_t)B * M * P));
    B200SV_CUDA(d_ss.upload(ss.data(), nq));
    B200SV_CUDA(d_pr.alloc(nq));
    B200SV_CUDA(d_iv.alloc(nq));
    const long long threads = (long long)B * P;
    const int tpb = mgf_block_threads((int)std::min<long long>(threads, 1 << 30)), nb = (P + tpb - 1) / tpb;
    if (N == 5)
      launch_logsv_mgf<5>(tpb, nb, st, d_phi.p, nullptr, P, M, d_spec.p, nullptr, d_a.p, d_lm.p, 0.0, nullptr, B, d_y.p, per_set_grid ? P : 0);
    else
      launch_logsv_mgf<3>(tpb, nb, st, d_phi.p, nullptr, P, M, d_spec.p, nullptr, d_a.p, d_lm.p, 0.0, nullptr, B, d_y.p, per_set_grid ? P : 0);
    if (int rc = launched("logsv_mgf_kernel")) return rc;
    fourier_vanilla_kernel<<<(unsigned)nq, kFourierThreads, 0, st>>>(d_lm.p, d_phi.p, P, d_ss.p, spot ? 1 : 0, 1, d_pr.p, ivols_out ? d_iv.p : nullptr);
    if (int rc = launched("fourier_vanilla_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(prices_out, d_pr.p, sizeof(double) * nq, cudaMemcpyDeviceToHost, st));
    if (ivols_out) B200SV_CUDA(cudaMemcpyAsync(ivols_out, d_iv.p, sizeof(double) * nq, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

int b200sv_heston_price_chain_batch(const b200sv_heston_params* params, int B, int M, const double* ttms, const double* forwards,
                                    const double* discfactors, const int* offsets, const double* strikes, const int8_t* types,
                                    double vol_scaler, int P, double* prices_out, double* ivols_out) {
  B200SV_REQUIRE(params && ttms && forwards && discfactors && offsets && strikes && types && prices_out, "null pointer");
  if (P <= 0) P = 1000;
  const bool per_set_grid = !(vol_scaler > 0.0);      // default scaler depends on v0 of each set (heston_pricer.py:234-235)
  std::vector<double> dtaus;
  std::vector<StrikeSpec> ss;
  if (int rc = chain_batch_common(B, M, ttms, forwards, discfactors, offsets, strikes, types, true, P, dtaus, ss, per_set_grid)) return rc;
  const int Jtot = offsets[M] - offsets[0];
  const int G = per_set_grid ? B : 1;
  std::vector<double> phi, one;
  for (int g = 0; g < G; ++g) {
    build_phi(per_set_grid ? std::min(0.3, std::sqrt(params[g].v0 * ttms[0])) : vol_scaler, true, P, one);
    phi.insert(phi.end(), one.begin(), one.end());
  }
  const size_t nq = (size_t)B * Jtot;
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_phi(st), d_lm(st);
    DevBuf<b200sv_heston_params> d_hp(st);
    DevBuf<double> d_dt(st), d_pr(st), d_iv(st);
    DevBuf<StrikeSpec> d_ss(st);
    B200SV_CUDA(d_phi.upload(phi.data(), (size_t)G * P));
    B200SV_CUDA(d_hp.upload(params, B));
    B200SV_CUDA(d_dt.upload(dtaus.data(), M));
    B200SV_CUDA(d_lm.alloc((size_t)B * M * P));
    B200SV_CUDA(d_ss.upload(ss.data(), nq));
    B200SV_CUDA(d_pr.alloc(nq));
    B200SV_CUDA(d_iv.alloc(nq));
    const int tpb = 64, nb = (P + tpb - 1) / tpb;
    heston_mgf_kernel<<<dim3(nb, B), tpb, 0, st>>>(d_phi.p, nullptr, P, M, d_dt.p, params[0], nullptr, nullptr, nullptr, nullptr, d_lm.p, d_hp.p,
                                                   per_set_grid ? P : 0);
    if (int rc = launched("heston_mgf_kernel")) return rc;
    fourier_vanilla_kernel<<<(unsigned)nq, kFourierThreads, 0, st>>>(d_lm.p, d_phi.p, P, d_ss.p, 1, 1, d_pr.p, ivols_out ? d_iv.p : nullptr);
    if (int rc = launched("fourier_vanilla_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(prices_out, d_pr.p, sizeof(double) * nq, cudaMemcpyDeviceToHost, st));
    if (ivols_out) B200SV_CUDA(cudaMemcpyAsync(ivols_out, d_iv.p, sizeof(double) * nq, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

/* Hawkes jump-diffusion Fourier chain (hawkesjd_chain_pricer / hawkesjd_chain_pricer_with_risk_premia, hawkes_jd_pricer.py:365-515).
 * risk_premia_gamma = NaN: no risk kernel.  Otherwise the grid sits on Re = -1/2 - gamma, the normalisers / forwards under the risk kernel
 * come from two single-point solves per maturity (each restarted from A = 0) and the gamma slice pricer assembles the prices;
 * normalizers_out / gamma_forwards_out (M each, optional) return them. */
int b200sv_hawkesjd_price_chain(const b200sv_hawkes_params* params, int M, const double* ttms, const double* forwards, const double* discfactors,
                                const int* offsets, const double* strikes, const int8_t* types, int is_spot_measure, double vol_scaler, int P,
                                double risk_premia_gamma, double* prices_out, double* a_out, double* log_mgf_out, double* normalizers_out,
                                double* gamma_forwards_out) {
  B200SV_REQUIRE(params && ttms && forwards && discfactors && offsets && prices_out, "null pointer");
  if (P <= 0) P = 500;                                                        // MAX_PHI, hawkes_jd_pricer.py:37
  B200SV_REQUIRE(M >= 1 && P >= 3, "M >= 1, P >= 3");
  const bool with_gamma = risk_premia_gamma == risk_premia_gamma;
  const bool spot = is_spot_measure != 0;
  const int Jtot = offsets[M] - offsets[0];
  if (with_gamma) {                                                            // utils/mgf_pricer.py:310-318: 'C' / 'P' under the spot measure only
    if (!spot) return fail(-5, "not implemented");
    for (int j = offsets[0]; j < offsets[M]; ++j)
      if (types[j] != B200SV_CALL && types[j] != B200SV_PUT) return fail(-5, "not implemented");
  } else if (int rc = check_fourier_types(types + offsets[0], Jtot, spot)) {
    return rc;
  }
  std::vector<double> dts(2 * (size_t)M);                                      // [increments | full maturities]
  double t0 = 0.0, tmin = ttms[0];
  for (int m = 0; m < M; ++m) {
    B200SV_REQUIRE(ttms[m] > t0, "ttms must be positive and strictly increasing");
    dts[m] = ttms[m] - t0;
    dts[M + m] = ttms[m];
    t0 = ttms[m];
    tmin = std::min(tmin, ttms[m]);
  }
  for (int m = 0; m < M; ++m)
    for (int j = offsets[m]; j < offsets[m + 1]; ++j) B200SV_REQUIRE(strikes[j] > 0.0, "strikes must be positive");
  if (!(vol_scaler > 0.0)) vol_scaler = std::min(std::max(params->sigma, 0.2), 0.5) * std::sqrt(std::min(tmin, 1.0 / 12.0));   // :360-362
  std::vector<double> phi;
  build_phi(vol_scaler, true, P, phi);                                         // get_transform_var_grid default is_spot_measure=True (:385)
  if (with_gamma)
    for (int i = 0; i < P; ++i) phi[2 * i] = -0.5 - risk_premia_gamma;           // real_phi (:451)
  const HawkesMgfConsts c = make_hawkes_mgf_consts(*params);
  std::vector<double> normalizers(M, 1.0), gamma_forwards(M, 1.0);
  const int rc = host_call([&](cudaStream_t st) {
    DevBuf<cd> d_phi(st), d_a(st), d_lm(st), d_g(st);
    DevBuf<double> d_dt(st), d_pr(st);
    DevBuf<StrikeSpec> d_ss(st);
    B200SV_CUDA(d_phi.upload(phi.data(), P));
    B200SV_CUDA(d_dt.upload(dts.data(), 2 * (size_t)M));
    B200SV_CUDA(d_a.alloc((size_t)M * P * 3));
    B200SV_CUDA(d_lm.alloc((size_t)M * P));
    if (with_gamma) {                                                            // hawkesjd_forwards_under_risk_kernel (:487-515)
      const double two[4] = {-risk_premia_gamma, 0.0, -risk_premia_gamma - 1.0, 0.0};
      B200SV_CUDA(d_g.alloc(2 + 2 * (size_t)M));
      B200SV_CUDA(cudaMemcpyAsync(d_g.p, two, sizeof(two), cudaMemcpyHostToDevice, st));
      hawkes_mgf_kernel<4><<<1, 4, 0, st>>>(d_g.p, nullptr, 2, M, d_dt.p + M, c, nullptr, nullptr, d_g.p + 2, 1, nullptr);
      if (int rc = launched("hawkes_mgf_kernel")) return rc;
      std::vector<double> lm2(4 * (size_t)M);
      B200SV_CUDA(cudaMemcpyAsync(lm2.data(), d_g.p + 2, sizeof(cd) * 2 * M, cudaMemcpyDeviceToHost, st));
      B200SV_CUDA(cudaStreamSynchronize(st));                                    // the strike specs below need these on the host
      for (int m = 0; m < M; ++m) {                                              // log_mgf layout [m][point]
        normalizers[m] = 1.0 / std::exp(lm2[2 * (2 * (size_t)m + 0)]);
        gamma_forwards[m] = forwards[m] * std::exp(lm2[2 * (2 * (size_t)m + 1)]) * normalizers[m];
      }
    }
    std::vector<StrikeSpec> ss(std::max(Jtot, 1));
    for (int m = 0; m < M; ++m)
      for (int j = offsets[m]; j < offsets[m + 1]; ++j)
        ss[j - offsets[0]] = with_gamma ? StrikeSpec{strikes[j], forwards[m], normalizers[m], (int)types[j], m, gamma_forwards[m], 0}
                                        : StrikeSpec{strikes[j], forwards[m], discfactors[m], (int)types[j], m, ttms[m], 0};
    B200SV_CUDA(d_ss.upload(ss.data(), ss.size()));
    B200SV_CUDA(d_pr.alloc(ss.size()));
    const int tpb = mgf_block_threads(P), nb = (P + tpb - 1) / tpb;
    switch (tpb) {
      case 4: hawkes_mgf_kernel<4><<<nb, 4, 0, st>>>(d_phi.p, nullptr, P, M, d_dt.p, c, nullptr, d_a.p, d_lm.p, 0, nullptr); break;
      case 8: hawkes_mgf_kernel<8><<<nb, 8, 0, st>>>(d_phi.p, nullptr, P, M, d_dt.p, c, nullptr, d_a.p, d_lm.p, 0, nullptr); break;
      case 16: hawkes_mgf_kernel<16><<<nb, 16, 0, st>>>(d_phi.p, nullptr, P, M, d_dt.p, c, nullptr, d_a.p, d_lm.p, 0, nullptr); break;
      case 32: hawkes_mgf_kernel<32><<<nb, 32, 0, st>>>(d_phi.p, nullptr, P, M, d_dt.p, c, nullptr, d_a.p, d_lm.p, 0, nullptr); break;
      default: hawkes_mgf_kernel<64><<<nb, 64, 0, st>>>(d_phi.p, nullptr, P, M, d_dt.p, c, nullptr, d_a.p, d_lm.p, 0, nullptr); break;
    }
    if (int rc = launched("hawkes_mgf_kernel")) return rc;
    if (Jtot > 0) {
      if (with_gamma)
        fourier_gamma_kernel<<<Jtot, kFourierThreads, 0, st>>>(d_lm.p, d_phi.p, P, d_ss.p, risk_premia_gamma, d_pr.p);
      else
        fourier_vanilla_kernel<<<Jtot, kFourierThreads, 0, st>>>(d_lm.p, d_phi.p, P, d_ss.p, spot ? 1 : 0, 1, d_pr.p);
      if (int rc = launched("fourier kernel")) return rc;
      B200SV_CUDA(cudaMemcpyAsync(prices_out, d_pr.p, sizeof(double) * Jtot, cudaMemcpyDeviceToHost, st));
    }
    if (a_out) B200SV_CUDA(cudaMemcpyAsync(a_out, d_a.p, sizeof(cd) * (size_t)M * P * 3, cudaMemcpyDeviceToHost, st));
    if (log_mgf_out) B200SV_CUDA(cudaMemcpyAsync(log_mgf_out, d_lm.p, sizeof(cd) * (size_t)M * P, cudaMemcpyDeviceToHost, st));
    return 0;
  });
  if (rc) return rc;
  if (normalizers_out) std::copy(normalizers.begin(), normalizers.end(), normalizers_out);
  if (gamma_forwards_out) std::copy(gamma_forwards.begin(), gamma_forwards.end(), gamma_forwards_out);
  return 0;
}

/* compute_hawkes_a_mgf_grid (hawkes_jd_pricer.py:518-547) on caller-supplied grids: A(0) = a_inout [P][3] -> A(dtau) in place, log_mgf_out [P] */
int b200sv_hawkesjd_mgf_grid(const double* phi, const double* psi, int P, double dtau, double* a_inout, const b200sv_hawkes_params* params,
                             double* log_mgf_out) {
  B200SV_REQUIRE(phi && a_inout && params && log_mgf_out, "null pointer");
  B200SV_REQUIRE(P >= 1 && dtau > 0.0, "P >= 1, dtau > 0");
  const HawkesMgfConsts c = make_hawkes_mgf_consts(*params);
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_phi(st), d_psi(st), d_a0(st), d_a1(st), d_lm(st);
    DevBuf<double> d_dt(st);
    B200SV_CUDA(d_phi.upload(phi, P));
    B200SV_CUDA(psi ? d_psi.upload(psi, P) : d_psi.alloc(P));
    B200SV_CUDA(d_dt.upload(&dtau, 1));
    B200SV_CUDA(d_a0.upload(a_inout, (size_t)P * 3));
    B200SV_CUDA(d_a1.alloc((size_t)P * 3));
    B200SV_CUDA(d_lm.alloc(P));
    const cd* dpsi = psi ? d_psi.p : nullptr;
    const int tpb = mgf_block_threads(P), nb = (P + tpb - 1) / tpb;
    switch (tpb) {
      case 4: hawkes_mgf_kernel<4><<<nb, 4, 0, st>>>(d_phi.p, dpsi, P, 1, d_dt.p, c, d_a0.p, d_a1.p, d_lm.p, 0, nullptr); break;
      case 8: hawkes_mgf_kernel<8><<<nb, 8, 0, st>>>(d_phi.p, dpsi, P, 1, d_dt.p, c, d_a0.p, d_a1.p, d_lm.p, 0, nullptr); break;
      case 16: hawkes_mgf_kernel<16><<<nb, 16, 0, st>>>(d_phi.p, dpsi, P, 1, d_dt.p, c, d_a0.p, d_a1.p, d_lm.p, 0, nullptr); break;
      case 32: hawkes_mgf_kernel<32><<<nb, 32, 0, st>>>(d_phi.p, dpsi, P, 1, d_dt.p, c, d_a0.p, d_a1.p, d_lm.p, 0, nullptr); break;
      default: hawkes_mgf_kernel<64><<<nb, 64, 0, st>>>(d_phi.p, dpsi, P, 1, d_dt.p, c, d_a0.p, d_a1.p, d_lm.p, 0, nullptr); break;
    }
    if (int rc = launched("hawkes_mgf_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(a_inout, d_a1.p, sizeof(cd) * (size_t)P * 3, cudaMemcpyDeviceToHost, st));
    B200SV_CUDA(cudaMemcpyAsync(log_mgf_out, d_lm.p, sizeof(cd) * P, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

int b200sv_logsv_mgf_grid(const double* phi, const double* psi, int P, double dtau, double* a_inout,
                          const b200sv_logsv_params* params, double eta, int is_spot_measure, int expansion_order,
                          double* log_mgf_out) {
  B200SV_REQUIRE(phi && a_inout && params && log_mgf_out, "null pointer");
  B200SV_REQUIRE(P >= 1 && dtau > 0.0, "P >= 1, dtau > 0");
  if (expansion_order != B200SV_ORDER_FIRST && expansion_order != B200SV_ORDER_SECOND)
    return fail(-4, "expansion_order not implemented");
  const int N = expansion_order == B200SV_ORDER_FIRST ? 3 : 5;
  ChainSpec spec{dtau, make_model(*params, eta, is_spot_measure != 0)};
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_phi(st), d_psi(st), d_a0(st), d_a1(st), d_lm(st);
    DevBuf<ChainSpec> d_spec(st);
    B200SV_CUDA(d_phi.upload(phi, P));
    B200SV_CUDA(psi ? d_psi.upload(psi, P) : d_psi.alloc(P));
    B200SV_CUDA(d_spec.upload(&spec, 1));
    B200SV_CUDA(d_a0.upload(a_inout, (size_t)P * N));
    B200SV_CUDA(d_a1.alloc((size_t)P * N));
    B200SV_CUDA(d_lm.alloc(P));
    const int tpb = mgf_block_threads(P), nb = (P + tpb - 1) / tpb;
    const double y = params->sigma0 - params->theta;
    const cd* dpsi = psi ? d_psi.p : nullptr;
    if (N == 5)
      launch_logsv_mgf<5>(tpb, nb, st, d_phi.p, dpsi, P, 1, d_spec.p, d_a0.p, d_a1.p, d_lm.p, y, nullptr);
    else
      launch_logsv_mgf<3>(tpb, nb, st, d_phi.p, dpsi, P, 1, d_spec.p, d_a0.p, d_a1.p, d_lm.p, y, nullptr);
    if (int rc = launched("logsv_mgf_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(a_inout, d_a1.p, sizeof(cd) * (size_t)P * N, cudaMemcpyDeviceToHost, st));
    B200SV_CUDA(cudaMemcpyAsync(log_mgf_out, d_lm.p, sizeof(cd) * P, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

// func_a_ode_quadratic_terms (pricers/logsv/affine_expansion.py:67-184) for a grid of transform points: the dense tensors the reference
// builds per point -- M [n][n][n] (symmetric in the last two indices), L [n][n], H [n], complex -- written from the SAME row tables
// (make_lane_row / make_coef) the ODE kernels integrate with, and func_rhs (:187-205) evaluated with the production rhs<>() at given A.
// Parity entry points: nothing on the pricing path needs the dense tensors.
int b200sv_logsv_ode_terms(const double* phi, const double* psi, int P, const b200sv_logsv_params* params, double eta, int is_spot_measure,
                           int expansion_order, double* M_out, double* L_out, double* H_out) {
  B200SV_REQUIRE(phi && params && M_out && L_out && H_out, "null pointer");
  B200SV_REQUIRE(P >= 1, "P >= 1");
  if (expansion_order != B200SV_ORDER_FIRST && expansion_order != B200SV_ORDER_SECOND) return fail(-4, "expansion_order not implemented");
  const int N = expansion_order == B200SV_ORDER_FIRST ? 3 : 5;
  const LogsvModel model = make_model(*params, eta, is_spot_measure != 0);
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_phi(st), d_psi(st), d_M(st), d_L(st), d_H(st);
    const size_t nM = (size_t)P * N * N * N, nL = (size_t)P * N * N, nH = (size_t)P * N;
    B200SV_CUDA(d_phi.upload(phi, P));
    B200SV_CUDA(psi ? d_psi.upload(psi, P) : d_psi.alloc(P));
    B200SV_CUDA(d_M.alloc(nM));
    B200SV_CUDA(d_L.alloc(nL));
    B200SV_CUDA(d_H.alloc(nH));
    const cd* dpsi = psi ? d_psi.p : nullptr;
    if (N == 5)
      logsv_ode_terms_kernel<5><<<(P + 63) / 64, 64, 0, st>>>(d_phi.p, dpsi, P, model, d_M.p, d_L.p, d_H.p);
    else
      logsv_ode_terms_kernel<3><<<(P + 63) / 64, 64, 0, st>>>(d_phi.p, dpsi, P, model, d_M.p, d_L.p, d_H.p);
    if (int rc = launched("logsv_ode_terms_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(M_out, d_M.p, sizeof(cd) * nM, cudaMemcpyDeviceToHost, st));
    B200SV_CUDA(cudaMemcpyAsync(L_out, d_L.p, sizeof(cd) * nL, cudaMemcpyDeviceToHost, st));
    B200SV_CUDA(cudaMemcpyAsync(H_out, d_H.p, sizeof(cd) * nH, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

int b200sv_logsv_ode_rhs(const double* phi, const double* psi, int P, const double* A, const b200sv_logsv_params* params, double eta,
                         int is_spot_measure, int expansion_order, double* rhs_out) {
  B200SV_REQUIRE(phi && A && params && rhs_out, "null pointer");
  B200SV_REQUIRE(P >= 1, "P >= 1");
  if (expansion_order != B200SV_ORDER_FIRST && expansion_order != B200SV_ORDER_SECOND) return fail(-4, "expansion_order not implemented");
  const int N = expansion_order == B200SV_ORDER_FIRST ? 3 : 5;
  const LogsvModel model = make_model(*params, eta, is_spot_measure != 0);
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_phi(st), d_psi(st), d_A(st), d_R(st);
    B200SV_CUDA(d_phi.upload(phi, P));
    B200SV_CUDA(psi ? d_psi.upload(psi, P) : d_psi.alloc(P));
    B200SV_CUDA(d_A.upload(A, (size_t)P * N));
    B200SV_CUDA(d_R.alloc((size_t)P * N));
    const cd* dpsi = psi ? d_psi.p : nullptr;
    if (N == 5)
      logsv_ode_rhs_kernel<5><<<(P + 63) / 64, 64, 0, st>>>(d_phi.p, dpsi, P, model, d_A.p, d_R.p);
    else
      logsv_ode_rhs_kernel<3><<<(P + 63) / 64, 64, 0, st>>>(d_phi.p, dpsi, P, model, d_A.p, d_R.p);
    if (int rc = launched("logsv_ode_rhs_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(rhs_out, d_R.p, sizeof(cd) * (size_t)P * N, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

int b200sv_ode_rhs_dense(const double* A, int P, int n, const double* M, const double* L, const double* H, double* rhs_out) {
  B200SV_REQUIRE(A && M && L && H && rhs_out, "null pointer");
  B200SV_REQUIRE(P >= 1 && n >= 1 && n <= 16, "P >= 1, 1 <= n <= 16");
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_A(st), d_M(st), d_L(st), d_H(st), d_R(st);
    B200SV_CUDA(d_A.upload(A, (size_t)P * n));
    B200SV_CUDA(d_M.upload(M, (size_t)n * n * n));
    B200SV_CUDA(d_L.upload(L, (size_t)n * n));
    B200SV_CUDA(d_H.upload(H, n));
    B200SV_CUDA(d_R.alloc((size_t)P * n));
    ode_rhs_dense_kernel<<<(P * n + 127) / 128, 128, 0, st>>>(d_A.p, P, n, d_M.p, d_L.p, d_H.p, d_R.p);
    if (int rc = launched("ode_rhs_dense_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(rhs_out, d_R.p, sizeof(cd) * (size_t)P * n, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

// compute_logsv_a_mgf_grid(is_analytic=True): the semi-analytic branch over a transform grid (affine_expansion.py:388-470 -> :306-384)
int b200sv_logsv_mgf_grid_analytic(const double* phi, const double* psi, int P, double dtau, double* a_inout, const b200sv_logsv_params* params,
                                   int is_spot_measure, int expansion_order, int year_days, double* log_mgf_out) {
  B200SV_REQUIRE(phi && a_inout && params && log_mgf_out, "null pointer");
  B200SV_REQUIRE(P >= 1 && dtau > 0.0 && year_days >= 1, "P >= 1, dtau > 0, year_days >= 1");
  if (expansion_order != B200SV_ORDER_FIRST && expansion_order != B200SV_ORDER_SECOND) return fail(-4, "expansion_order not implemented");
  const int N = expansion_order == B200SV_ORDER_FIRST ? 3 : 5;
  const LogsvModel model = make_model(*params, 1.0, is_spot_measure != 0);      // eta is ignored on this branch (reference :340-348)
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_phi(st), d_psi(st), d_a0(st), d_a1(st), d_lm(st);
    B200SV_CUDA(d_phi.upload(phi, P));
    B200SV_CUDA(psi ? d_psi.upload(psi, P) : d_psi.alloc(P));
    B200SV_CUDA(d_a0.upload(a_inout, (size_t)P * N));
    B200SV_CUDA(d_a1.alloc((size_t)P * N));
    B200SV_CUDA(d_lm.alloc(P));
    const cd* dpsi = psi ? d_psi.p : nullptr;
    const double y = params->sigma0 - params->theta;
    if (N == 5)
      logsv_mgf_analytic_kernel<5><<<(P + 63) / 64, 64, 0, st>>>(d_phi.p, dpsi, P, model, dtau, year_days, d_a0.p, d_a1.p, d_lm.p, y);
    else
      logsv_mgf_analytic_kernel<3><<<(P + 63) / 64, 64, 0, st>>>(d_phi.p, dpsi, P, model, dtau, year_days, d_a0.p, d_a1.p, d_lm.p, y);
    if (int rc = launched("logsv_mgf_analytic_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(a_inout, d_a1.p, sizeof(cd) * (size_t)P * N, cudaMemcpyDeviceToHost, st));
    B200SV_CUDA(cudaMemcpyAsync(log_mgf_out, d_lm.p, sizeof(cd) * P, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

// compute_logsv_a_mgf_grid(is_stiff_solver=True): SciPy's BDF control law per grid point (affine_expansion.py:229-303)
int b200sv_logsv_mgf_grid_bdf(const double* phi, const double* psi, int P, double dtau, double* a_inout, const b200sv_logsv_params* params,
                              double eta, int is_spot_measure, int expansion_order, double* log_mgf_out) {
  B200SV_REQUIRE(phi && a_inout && params && log_mgf_out, "null pointer");
  B200SV_REQUIRE(P >= 1 && dtau > 0.0, "P >= 1, dtau > 0");
  if (expansion_order != B200SV_ORDER_FIRST && expansion_order != B200SV_ORDER_SECOND) return fail(-4, "expansion_order not implemented");
  const int N = expansion_order == B200SV_ORDER_FIRST ? 3 : 5;
  const LogsvModel model = make_model(*params, eta, is_spot_measure != 0);
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_phi(st), d_psi(st), d_a0(st), d_a1(st), d_lm(st);
    B200SV_CUDA(d_phi.upload(phi, P));
    B200SV_CUDA(psi ? d_psi.upload(psi, P) : d_psi.alloc(P));
    B200SV_CUDA(d_a0.upload(a_inout, (size_t)P * N));
    B200SV_CUDA(d_a1.alloc((size_t)P * N));
    B200SV_CUDA(d_lm.alloc(P));
    const cd* dpsi = psi ? d_psi.p : nullptr;
    const double y = params->sigma0 - params->theta;
    if (N == 5)
      logsv_mgf_bdf_kernel<5><<<(P + 63) / 64, 64, 0, st>>>(d_phi.p, dpsi, P, model, dtau, d_a0.p, d_a1.p, d_lm.p, y, nullptr);
    else
      logsv_mgf_bdf_kernel<3><<<(P + 63) / 64, 64, 0, st>>>(d_phi.p, dpsi, P, model, dtau, d_a0.p, d_a1.p, d_lm.p, y, nullptr);
    if (int rc = launched("logsv_mgf_bdf_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(a_inout, d_a1.p, sizeof(cd) * (size_t)P * N, cudaMemcpyDeviceToHost, st));
    B200SV_CUDA(cudaMemcpyAsync(log_mgf_out, d_lm.p, sizeof(cd) * P, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

int b200sv_heston_mgf_grid(const double* phi, const double* psi, int P, double dtau, double* a_inout, double* b_inout,
                           const b200sv_heston_params* params, double* log_mgf_out) {
  B200SV_REQUIRE(phi && a_inout && b_inout && params && log_mgf_out, "null pointer");
  B200SV_REQUIRE(P >= 1 && dtau > 0.0, "P >= 1, dtau > 0");
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_phi(st), d_psi(st), d_a(st), d_b(st), d_a1(st), d_b1(st), d_lm(st);
    DevBuf<double> d_dt(st);
    B200SV_CUDA(d_phi.upload(phi, P));
    B200SV_CUDA(psi ? d_psi.upload(psi, P) : d_psi.alloc(P));
    B200SV_CUDA(d_dt.upload(&dtau, 1));
    B200SV_CUDA(d_a.upload(a_inout, P));
    B200SV_CUDA(d_b.upload(b_inout, P));
    B200SV_CUDA(d_a1.alloc(P));
    B200SV_CUDA(d_b1.alloc(P));
    B200SV_CUDA(d_lm.alloc(P));
    const int tpb = mgf_block_threads(P), nb = (P + tpb - 1) / tpb;
    heston_mgf_kernel<<<nb, tpb, 0, st>>>(d_phi.p, psi ? d_psi.p : nullptr, P, 1, d_dt.p, *params,
                                          d_a.p, d_b.p, d_a1.p, d_b1.p, d_lm.p);
    if (int rc = launched("heston_mgf_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(a_inout, d_a1.p, sizeof(cd) * P, cudaMemcpyDeviceToHost, st));
    B200SV_CUDA(cudaMemcpyAsync(b_inout, d_b1.p, sizeof(cd) * P, cudaMemcpyDeviceToHost, st));
    B200SV_CUDA(cudaMemcpyAsync(log_mgf_out, d_lm.p, sizeof(cd) * P, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

int b200sv_fourier_vanilla(const double* log_mgf, const double* phi, int P, double forward, const double* strikes,
                           const int8_t* types, int J, double discfactor, int is_spot_measure, double* prices_out) {
  B200SV_REQUIRE(log_mgf && phi && strikes && types && prices_out, "null pointer");
  B200SV_REQUIRE(P >= 3 && J >= 1, "P >= 3, J >= 1");
  const bool spot = is_spot_measure != 0;
  if (int rc = check_fourier_types(types, J, spot)) return rc;
  std::vector<StrikeSpec> ss(J);
  for (int j = 0; j < J; ++j) ss[j] = StrikeSpec{strikes[j], forward, discfactor, (int)types[j], 0, 1.0, 0};
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_phi(st), d_lm(st);
    DevBuf<StrikeSpec> d_ss(st);
    DevBuf<double> d_pr(st);
    B200SV_CUDA(d_phi.upload(phi, P));
    B200SV_CUDA(d_lm.upload(log_mgf, P));
    B200SV_CUDA(d_ss.upload(ss.data(), J));
    B200SV_CUDA(d_pr.alloc(J));
    fourier_vanilla_kernel<<<J, kFourierThreads, 0, st>>>(d_lm.p, d_phi.p, P, d_ss.p, spot ? 1 : 0,
                                                          all_half_re(phi, P) ? 1 : 0, d_pr.p);
    if (int rc = launched("fourier_vanilla_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(prices_out, d_pr.p, sizeof(double) * J, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

/* slice_pricer_with_mgf_grid_with_gamma (utils/mgf_pricer.py:273-320) on caller-supplied log-MGF / transform grids: 'C' / 'P' under the spot
 * measure, everything else is ValueError("not implemented") there (-5 here) */
int b200sv_fourier_gamma(const double* log_mgf, const double* phi, int P, double risk_premia_gamma, double forward, double normalizer,
                         double gamma_forward, const double* strikes, const int8_t* types, int J, int is_spot_measure, double* prices_out) {
  B200SV_REQUIRE(log_mgf && phi && strikes && types && prices_out, "null pointer");
  B200SV_REQUIRE(P >= 3 && J >= 1, "P >= 3, J >= 1");
  if (!is_spot_measure) return fail(-5, "not implemented");
  std::vector<StrikeSpec> ss(J);
  for (int j = 0; j < J; ++j) {
    if (types[j] != B200SV_CALL && types[j] != B200SV_PUT) return fail(-5, "not implemented");
    ss[j] = StrikeSpec{strikes[j], forward, normalizer, (int)types[j], 0, gamma_forward, 0};
  }
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_phi(st), d_lm(st);
    DevBuf<StrikeSpec> d_ss(st);
    DevBuf<double> d_pr(st);
    B200SV_CUDA(d_phi.upload(phi, P));
    B200SV_CUDA(d_lm.upload(log_mgf, P));
    B200SV_CUDA(d_ss.upload(ss.data(), J));
    B200SV_CUDA(d_pr.alloc(J));
    fourier_gamma_kernel<<<J, kFourierThreads, 0, st>>>(d_lm.p, d_phi.p, P, d_ss.p, risk_premia_gamma, d_pr.p);
    if (int rc = launched("fourier_gamma_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(prices_out, d_pr.p, sizeof(double) * J, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

// shared driver of the generic sums
static int fourier_sum_host(const double* log_mgf, const double* grid, int P, const std::vector<SumSpec>& specs, int mode, int all_calls,
                            double* out) {
  const int J = (int)specs.size();
  return host_call([&](cudaStream_t st) {
    DevBuf<cd> d_g(st), d_lm(st);
    DevBuf<SumSpec> d_ss(st);
    DevBuf<double> d_pr(st);
    B200SV_CUDA(d_g.upload(grid, P));
    B200SV_CUDA(d_lm.upload(log_mgf, P));
    B200SV_CUDA(d_ss.upload(specs.data(), J));
    B200SV_CUDA(d_pr.alloc(J));
    fourier_sum_kernel<<<J, kFourierThreads, 0, st>>>(d_lm.p, d_g.p, P, d_ss.p, mode, all_calls, d_pr.p);
    if (int rc = launched("fourier_sum_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(out, d_pr.p, sizeof(double) * J, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

int b200sv_fourier_qvar(const double* log_mgf, const double* psi, int P, double ttm, const double* strikes, const int8_t* types, int J,
                        double discfactor, double* prices_out) {
  B200SV_REQUIRE(log_mgf && psi && strikes && types && prices_out, "null pointer");
  B200SV_REQUIRE(P >= 3 && J >= 1 && ttm > 0.0, "P >= 3, J >= 1, ttm > 0");
  if (int rc = check_qvar_types(types, J)) return rc;
  std::vector<SumSpec> specs(J);
  for (int j = 0; j < J; ++j) specs[j] = SumSpec{strikes[j] * ttm, discfactor, ttm, (int)types[j], 0};
  return fourier_sum_host(log_mgf, psi, P, specs, kModeQvar, 0, prices_out);
}

int b200sv_fourier_pdf(const double* log_mgf, const double* grid, int P, const double* z, int J, double* out) {
  B200SV_REQUIRE(log_mgf && grid && z && out, "null pointer");
  B200SV_REQUIRE(P >= 3 && J >= 1, "P >= 3, J >= 1");
  std::vector<SumSpec> specs(J);
  for (int j = 0; j < J; ++j) specs[j] = SumSpec{z[j], 1.0, 1.0, 0, 0};
  return fourier_sum_host(log_mgf, grid, P, specs, kModePdf, 0, out);
}

int b200sv_fourier_digital(const double* log_mgf, const double* phi, int P, double forward, const double* strikes, const int8_t* types,
                           int J, double discfactor, double* prices_out) {
  B200SV_REQUIRE(log_mgf && phi && strikes && types && prices_out, "null pointer");
  B200SV_REQUIRE(P >= 3 && J >= 1, "P >= 3, J >= 1");
  for (int j = 0; j < J; ++j)
    if (types[j] != B200SV_CALL && types[j] != B200SV_PUT) return fail(-5, "not implemented");   // utils/mgf_pricer.py:265-266
  bool all_neg = true;                                             // np.all(np.real(phi_grid) < 0.0), :241
  for (int i = 0; i < P; ++i) all_neg = all_neg && (phi[2 * i] < 0.0);
  std::vector<SumSpec> specs(J);
  for (int j = 0; j < J; ++j) specs[j] = SumSpec{-std::log(forward / strikes[j]), discfactor, 1.0, (int)types[j], 0};
  return fourier_sum_host(log_mgf, phi, P, specs, kModeDigital, all_neg ? 1 : 0, prices_out);
}

}  // extern "C"
