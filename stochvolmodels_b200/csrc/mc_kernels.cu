// mc_kernels.cu -- fused Monte Carlo hot path for sm_100a (B200).
//
// Replaces, behind the C ABI of include/b200sv.h, the reference functions (paths under
// /root/reference/src/stochvolmodels):
//   simulate_logsv_x_vol_terminal     pricers/logsv_pricer.py:950-1047
//   logsv_mc_chain_pricer             pricers/logsv_pricer.py:806-867
//   logsv_mc_chain_pricer_fixed_randoms (stepping part)  pricers/logsv_pricer.py:1100-1162
//   simulate_heston_x_vol_terminal    pricers/heston_pricer.py:334-381
//   heston_mc_chain_pricer            pricers/heston_pricer.py:285-331
//   compute_mc_vars_payoff            utils/mc_payoffs.py:10-88
//   set_time_grid                     utils/funcs.py:24-47
//
// Design (DESIGN.md §3): one persistent wave of CTAs; a thread owns one path at a time, keeps (x, log sigma, sigma,
// sigma^2, qvar) in registers for the whole maturity slice, draws its Gaussians in-kernel (Philox4x32-10 keyed by the
// GLOBAL path id), and touches HBM only to load / store the SoA state at slice boundaries (24 B + 24 B per path per slice
// in fp64).  The forward re-centring of the payoffs needs the mean over ALL paths first, hence two phases per slice:
//   slice kernel  -> per-CTA (sum F e^x, count) partials -> fixed-order reduction            [all-reduce #1 if multi-GPU]
//   payoff kernel -> per-CTA per-strike (sum, sum^2, count) partials -> fixed-order reduction [all-reduce #2 if multi-GPU]
// All moment arithmetic is fp64 and every reduction has a fixed order => bitwise reproducible for a given launch shape.
#include <cooperative_groups.h>

#include <algorithm>
#include <cmath>
#include <type_traits>
#include <cstdlib>
#include <vector>

#include "../../include/b200sv.h"
#include "common.cuh"
#include "fastmath64.cuh"
#include "p2p.cuh"
#include "black.cuh"
#include "philox.cuh"

namespace b200sv {

cudaStream_t& current_stream_ref() {
  static thread_local cudaStream_t st = nullptr;
  return st;
}
long long& launch_count() {
  static thread_local long long n = 0;
  return n;
}
constexpr int kThreads = 256;
#ifndef B200SV_SLICE_PREFETCH
#define B200SV_SLICE_PREFETCH 1     // issue the next Philox/Box-Muller call before the two fp64 steps of the current one
#endif
#ifndef B200SV_SLICE_THREADS
#define B200SV_SLICE_THREADS 256
#endif
constexpr int kSliceThreads = B200SV_SLICE_THREADS;
#ifndef B200SV_SLICE_MINBLOCKS
#define B200SV_SLICE_MINBLOCKS 2   // resident CTAs / SM the slice kernel is register-budgeted for.  Tuned on B200 (profiles/r02_occupancy.txt):
#endif                             // 16 warps/SM as 2 x 256 threads 352 Gpath-steps/s, 4 x 128 345, 3 x 128 345, 5 x 128 (96 regs) 330, 6 x 128 319
constexpr int kStrikeChunk = 8;

// --------------------------------------------------------------------------------------------------------------------
// per-step model updates
// --------------------------------------------------------------------------------------------------------------------
struct LogsvConsts {   // all dt / sqrt(dt) factors folded in on the host (fp64)
  double cx;    // alpha * 0.5 * eta^2 * dt          x  += cx * sigma^2 + ce * sigma * z0
  double ce;    // eta * sqrt(dt)
  double a0;    // (-kappa1 + kappa2*theta - 0.5*vartheta^2) * dt
  double a1;    // kappa1 * theta * dt               L  += a0 + a1 / sigma + a2 * sigma + b0 z0 + b1 z1
  double a2;    // (adj - kappa2) * dt
  double b0;    // beta * sqrt(dt)
  double b1;    // volvol * sqrt(dt)
  double cq;    // 0.5 * eta^2 * dt                  q  += cq * (sigma_old^2 + sigma_new^2)
  double a0s, a1s, a2s, b0s, b1s;   // a0..b1 in table units (x 256/ln2): the fp64 stepper carries Ls = L * 256/ln2 (fastmath64.cuh)
};

struct HestonConsts {
  double hx;    // -0.5 * dt                         x += hx * v + sdt * sqrt(v) * z0
  double sdt;   // sqrt(dt)
  double dt;    //                                   q += dt * v
  double kdt;   // kappa * dt                        v += kdt * (theta - v) + sqrt(v) * (c0 z0 + c1 z1);  v = max(v, 1e-4)
  double theta;
  double c0;    // volvol * rho * sqrt(dt)
  double c1;    // volvol * sqrt(1 - rho^2) * sqrt(dt)
  // opt-in Andersen (2008) quadratic-exponential scheme (B200SV_HESTON_QE), central discretisation gamma1 = gamma2 = 1/2
  int qe;
  double e;     // exp(-kappa dt)                     m  = v e + m0,  m0 = theta (1 - e)
  double m0;
  double s1;    // volvol^2 e (1 - e) / kappa         s2 = v s1 + s0
  double s0;    // theta volvol^2 (1 - e)^2 / (2 kappa)
  double K0, K1, K2, K3, K4;   // x' = x + K0 + K1 v + K2 v' + sqrt(K3 v + K4 v') Zx
};

static LogsvConsts make_logsv_consts(const b200sv_logsv_params& p, double eta, bool spot, double dt) {
  // measure switch: pricers/logsv_pricer.py:1032-1035
  const double alpha = spot ? -1.0 : 1.0, adj = spot ? 0.0 : p.beta * eta;
  const double vt2 = p.beta * p.beta + p.volvol * p.volvol, sdt = std::sqrt(dt);
  LogsvConsts c;
  c.cx = alpha * 0.5 * eta * eta * dt;
  c.ce = eta * sdt;
  c.a0 = (-p.kappa1 + p.kappa2 * p.theta - 0.5 * vt2) * dt;
  c.a1 = p.kappa1 * p.theta * dt;
  c.a2 = (adj - p.kappa2) * dt;
  c.b0 = p.beta * sdt;
  c.b1 = p.volvol * sdt;
  c.cq = 0.5 * eta * eta * dt;
  c.a0s = c.a0 * kLogScale;
  c.a1s = c.a1 * kLogScale;
  c.a2s = c.a2 * kLogScale;
  c.b0s = c.b0 * kLogScale;
  c.b1s = c.b1 * kLogScale;
  return c;
}

static HestonConsts make_heston_consts(const b200sv_heston_params& p, double dt, int scheme = B200SV_HESTON_EULER_FLOOR) {
  const double sdt = std::sqrt(dt);
  HestonConsts c;
  c.qe = scheme == B200SV_HESTON_QE;
  c.e = std::exp(-p.kappa * dt);
  c.m0 = p.theta * (1.0 - c.e);
  c.s1 = p.volvol * p.volvol * c.e * (1.0 - c.e) / p.kappa;
  c.s0 = p.theta * p.volvol * p.volvol * (1.0 - c.e) * (1.0 - c.e) / (2.0 * p.kappa);
  const double kre = p.kappa * p.rho / p.volvol;
  c.K0 = -p.rho * p.kappa * p.theta * dt / p.volvol;
  c.K1 = 0.5 * dt * (kre - 0.5) - p.rho / p.volvol;
  c.K2 = 0.5 * dt * (kre - 0.5) + p.rho / p.volvol;
  c.K3 = 0.5 * dt * (1.0 - p.rho * p.rho);
  c.K4 = c.K3;
  c.hx = -0.5 * dt;
  c.sdt = sdt;
  c.dt = dt;
  c.kdt = p.kappa * dt;
  c.theta = p.theta;
  c.c0 = p.volvol * p.rho * sdt;
  c.c1 = p.volvol * std::sqrt(1.0 - p.rho * p.rho) * sdt;
  return c;
}

template <typename Real>
struct LogsvPath;

// fp64 state: same scheme, reformulated so that the per-step work is the log-vol recursion plus two running sums:
//   A  = sum_{k=1..S} sigma_k^2      (new sigma of every step)
//   XM = sum_{k=0..S-1} sigma_k z0_k (martingale part of x, old sigma)
// from which  x_S = x_0 + cx*(sigma_0^2 + A - sigma_S^2) + ce*XM          [sum_k cx*sigma_k^2 + ce*sigma_k*z0_k]
//             q_S = q_0 + cq*(sigma_0^2 + 2A - sigma_S^2)                 [sum_k cq*(sigma_k^2 + sigma_{k+1}^2)]
// (logsv_pricer.py:1041-1045 summed over the slice).  The log-vol is carried in table units Ls = L * 256/ln2 so that sigma = exp(L) and
// 1/sigma = exp(-L) come out of exp_pair_scaled (11 fp64 instructions, fastmath64.cuh); 18 fp64-pipe instructions per step in all.
// Range guard: step<false> only RECORDS |Ls| > kLogScaledMax (|L| > 699.997: one LOP3 + one ISETP.OR per step); a path that ever trips
// it is re-run by the kernel with step<true>, which clamps every step -- the result is the clamped recursion for every path, the common
// case pays 2 integer instructions instead of 5 + 2.
template <>
struct LogsvPath<double> {
  double Ls, s, inv, A, XM, x0, q0, s2_first;
  double cx, ce, a0, a1, a2, b0, b1, cq;
  bool bad;
  __device__ __forceinline__ LogsvPath(const LogsvConsts& c)
      : cx(c.cx), ce(c.ce), a0(c.a0s), a1(c.a1s), a2(c.a2s), b0(c.b0s), b1(c.b1s), cq(c.cq), bad(false) {}
  __device__ __forceinline__ void load(double x_, double sigma0, double q_) {
    x0 = x_;
    q0 = q_;
    Ls = clamp_log_scaled(clamp_log(log(sigma0)) * kLogScale);    // vol_var = np.log(sigma0), logsv_pricer.py:1039
    exp_pair_scaled(Ls, s, inv);
    s = sigma0;                    // keep the loaded sigma itself for the first step
    s2_first = s * s;
    A = 0.0;
    XM = 0.0;
    bad = false;
  }
  template <bool SAFE>
  __device__ __forceinline__ void step(double z0, double z1) {
#if defined(B200SV_ABLATE) && (B200SV_ABLATE & 4)   // tuning only: no fp64 recursion, just consume the normals
    XM = fma(z1, z0, XM);
    return;
#endif
    XM = fma(s, z0, XM);
    // noise + constant drift first (independent of sigma: off the critical path), then the two state-dependent terms
    double l = Ls + fma(b0, z0, fma(b1, z1, a0));
    l = fma(a2, s, l);
    l = fma(a1, inv, l);
    if constexpr (SAFE)
      l = clamp_log_scaled(l);
    else
      bad |= log_scaled_out_of_range(l);
    Ls = l;
    exp_pair_scaled(Ls, s, inv);
    A = fma(s, s, A);
  }
  __device__ __forceinline__ bool overflowed() const { return bad; }
  __device__ __forceinline__ double sigma() const { return s; }
  __device__ __forceinline__ double x() const { return fma(ce, XM, fma(cx, (s2_first - s * s) + A, x0)); }
  __device__ __forceinline__ double q() const { return fma(cq, (s2_first - s * s) + 2.0 * A, q0); }
};

// fp32 state (opt-in B200SV_STATE_F32): same structure, SFU exp / reciprocal
template <>
struct LogsvPath<float> {
  float L, s, inv, A, XM, x0, q0, s2_first;
  float cx, ce, a0, a1, a2, b0, b1, cq;
  __device__ __forceinline__ LogsvPath(const LogsvConsts& c)
      : cx((float)c.cx), ce((float)c.ce), a0((float)c.a0), a1((float)c.a1), a2((float)c.a2), b0((float)c.b0),
        b1((float)c.b1), cq((float)c.cq) {}
  __device__ __forceinline__ void load(float x_, float sigma0, float q_) {
    x0 = x_;
    q0 = q_;
    L = __logf(sigma0);
    s = sigma0;
    s2_first = s * s;
    inv = __frcp_rn(s);
    A = 0.0f;
    XM = 0.0f;
  }
  template <bool SAFE>
  __device__ __forceinline__ void step(float z0, float z1) {
    XM = fmaf(s, z0, XM);
    float l = L + fmaf(b0, z0, fmaf(b1, z1, a0));
    l = fmaf(a2, s, l);
    l = fmaf(a1, inv, l);
    L = fminf(fmaxf(l, -80.0f), 80.0f);
    s = __expf(L);
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(s));
    A = fmaf(s, s, A);
  }
  __device__ __forceinline__ bool overflowed() const { return false; }   // L is clamped every step
  __device__ __forceinline__ float sigma() const { return s; }
  __device__ __forceinline__ float x() const { return fmaf(ce, XM, fmaf(cx, (s2_first - s * s) + A, x0)); }
  __device__ __forceinline__ float q() const { return fmaf(cq, (s2_first - s * s) + 2.0f * A, q0); }
};

// QE = compile-time scheme switch: the floor-Euler kernel carries none of the quadratic-exponential code (a runtime flag inside the step
// cost the reference scheme 6 % through registers and instruction-cache footprint)
template <typename Real, bool QE = false>
struct HestonPath {
  Real v, V, XM, x0, q0, xacc, qacc;
  Real hx, sdt, dt, kdt, theta, c0, c1;
  Real e, m0, s1, s0, K0, K1, K2, K3, K4;
  int qe;
  __device__ __forceinline__ HestonPath(const HestonConsts& c)
      : hx((Real)c.hx), sdt((Real)c.sdt), dt((Real)c.dt), kdt((Real)c.kdt), theta((Real)c.theta), c0((Real)c.c0), c1((Real)c.c1),
        e((Real)c.e), m0((Real)c.m0), s1((Real)c.s1), s0((Real)c.s0), K0((Real)c.K0), K1((Real)c.K1), K2((Real)c.K2), K3((Real)c.K3),
        K4((Real)c.K4), qe(c.qe) {}
  __device__ __forceinline__ void load(Real x_, Real v_, Real q_) {
    x0 = x_;
    v = v_;
    q0 = q_;
    V = (Real)0;
    XM = (Real)0;
    xacc = (Real)0;
    qacc = (Real)0;
  }
  // Andersen's QE step: moment-matched quadratic (psi <= 1.5) or exponential (psi > 1.5) variance draw, then the log-spot with the
  // central discretisation.  z0 drives the spot, z1 the variance (U = Phi(z1) in the exponential branch).  Not in the reference
  // (BASELINE.json names it; SURVEY.md §0.1): validated against the Heston Fourier price and the oracle restatement.
  __device__ __forceinline__ void step_qe(Real zx, Real zv) {
    const Real m = fma(v, e, m0);
    const Real s2 = fma(v, s1, s0);
    const Real mm = m * m;
    Real vn;
    if (s2 <= (Real)1.5 * mm) {          // psi = s2 / m^2 <= 1.5, tested without the division
      // 2/psi = 2 m^2 / s2;  b^2 = 2/psi - 1 + sqrt(2/psi) sqrt(2/psi - 1) with the two roots merged (2/psi >= 4/3: both factors positive);
      // fp64 divisions and square roots through MUFU seeds + Newton / Householder steps (fastmath64.cuh, gauss64.cuh): <= 2 ulp, a third of
      // the instructions of the IEEE routines -- the QE step is 3 divisions + 4 roots in its textbook form, 2 + 3 here
      const Real ip = (Real)2 * fast_div(mm, s2);
      const Real t = ip - (Real)1;
      const Real b2 = t + fast_sqrt(ip * t);
      const Real a = fast_div(m, (Real)1 + b2);
      const Real r = fast_sqrt(b2) + zv;
      vn = a * r * r;
    } else {
      const Real psi = s2 / mm;
      const Real p = (psi - (Real)1) / (psi + (Real)1);
      const Real beta = ((Real)1 - p) / m;
      const Real u = (Real)normcdf((double)zv);
      vn = u <= p ? (Real)0 : (Real)log((double)(((Real)1 - p) / ((Real)1 - u))) / beta;
    }
    const Real arg = K3 * v + K4 * vn;
    xacc += K0 + K1 * v + K2 * vn + (arg > (Real)0 ? fast_sqrt(arg) : (Real)0) * zx;
    qacc += (Real)0.5 * dt * (v + vn);
    v = vn;
  }
  // pricers/heston_pricer.py:372-379 (floor-Euler): everything on the OLD variance, then v = max(v, 1e-4).
  // V = sum v_k, XM = sum sqrt(v_k) z0_k  =>  x_S = x_0 - 0.5*dt*V + sqrt(dt)*XM,  q_S = q_0 + dt*V.
  template <bool SAFE>
  __device__ __forceinline__ void step(Real z0, Real z1) {
    if constexpr (QE) {
      step_qe(z0, z1);
      return;
    }
    const Real sig = sqrt(v);
    V += v;
    XM = fma(sig, z0, XM);
    Real vn = fma(kdt, theta - v, v);
    vn = fma(sig, fma(c0, z0, c1 * z1), vn);
    v = vn > (Real)1e-4 ? vn : (Real)1e-4;     // np.maximum(var0, 1e-4)
  }
  __device__ __forceinline__ bool overflowed() const { return false; }
  __device__ __forceinline__ Real sigma() const { return v; }
  __device__ __forceinline__ Real x() const { return fma(sdt, XM, fma(hx, V, x0)) + xacc; }
  __device__ __forceinline__ Real q() const { return fma(dt, V, q0) + qacc; }
};

// --------------------------------------------------------------------------------------------------------------------
// fused slice kernel
// --------------------------------------------------------------------------------------------------------------------
template <typename Real>
struct SliceArgs {
  Real* x;
  Real* v;      // sigma (LogSV) or variance (Heston)
  Real* q;
  long long n;
  unsigned long long path_offset;
  int init;
  double v_init;
  int nsteps;
  unsigned int slice;
  unsigned long long seed;
  double forward;
  double* partials;   // [gridDim.x][2]
};

// advance one path through the slice, drawing its normals in the order philox.cuh defines.  SAFE = clamp the log-vol every step (re-run
// of a path whose fast pass left the representable range); !SAFE = the production loop with the generator software-pipelined one call
// ahead of the fp64 recursion (the integer / SFU stream of call c+1 overlaps the fp64 stream of call c inside a warp).
template <bool SAFE, typename Path, typename Real, int GAUSS>
__device__ __forceinline__ void run_slice_steps(Path& p, StepNormals<Real, GAUSS>& rng, int nsteps) {
  if constexpr (GAUSS == kGaussF64) {
    if constexpr (SAFE || !B200SV_SLICE_PREFETCH) {
      for (int s = 0; s < nsteps; ++s) {
        Real z0, z1;
        rng.get((uint32_t)s, z0, z1);
        p.template step<SAFE>(z0, z1);
      }
    } else {
      Real n0, n1;
      rng.get(0u, n0, n1);
#pragma unroll 1
      for (int s = 0; s < nsteps; ++s) {
        Real m0, m1;
        rng.get((uint32_t)(s + 1), m0, m1);
        p.template step<SAFE>(n0, n1);
        n0 = m0;
        n1 = m1;
      }
    }
  } else {
    // one Philox call feeds two steps
    const int ncalls = nsteps >> 1;
    if constexpr (SAFE || !B200SV_SLICE_PREFETCH) {
      for (int c = 0; c < ncalls; ++c) {
        Real n0, n1, n2, n3;
        rng.get2((uint32_t)c, n0, n1, n2, n3);
        p.template step<SAFE>(n0, n1);
        p.template step<SAFE>(n2, n3);
      }
      if (nsteps & 1) {
        Real n0, n1, n2, n3;
        rng.get2((uint32_t)ncalls, n0, n1, n2, n3);
        p.template step<SAFE>(n0, n1);
      }
    } else {
      Real n0, n1, n2, n3, m0, m1, m2, m3;
      rng.get2(0u, n0, n1, n2, n3);
      int c = 0;
#pragma unroll 1
      for (; c + 2 <= ncalls; c += 2) {     // two calls = four steps per iteration: the n / m register sets swap roles, no moves
        rng.get2((uint32_t)(c + 1), m0, m1, m2, m3);
        p.template step<SAFE>(n0, n1);
        p.template step<SAFE>(n2, n3);
        rng.get2((uint32_t)(c + 2), n0, n1, n2, n3);
        p.template step<SAFE>(m0, m1);
        p.template step<SAFE>(m2, m3);
      }
      if (c < ncalls) {
        rng.get2((uint32_t)(c + 1), m0, m1, m2, m3);
        p.template step<SAFE>(n0, n1);
        p.template step<SAFE>(n2, n3);
        n0 = m0;
        n1 = m1;
      }
      if (nsteps & 1) p.template step<SAFE>(n0, n1);
    }
  }
}

template <typename Path, typename Consts, typename Real, int GAUSS>
__global__ void __launch_bounds__(kSliceThreads, B200SV_SLICE_MINBLOCKS) mc_slice_kernel(SliceArgs<Real> a, Consts consts) {
  __shared__ double red[2 * kSliceThreads / 32];
  exp_table_init();
  if constexpr (GAUSS != kGaussF32) gauss64_table_init();
  double acc[2] = {0.0, 0.0};
  Path p(consts);
  const long long stride = (long long)gridDim.x * kSliceThreads;
  for (long long i = (long long)blockIdx.x * kSliceThreads + threadIdx.x; i < a.n; i += stride) {
    Real xi = (Real)0, vi = (Real)a.v_init, qi = (Real)0;
    if (!a.init) {
      xi = a.x[i];
      vi = a.v[i];
      qi = a.q[i];
    }
    p.load(xi, vi, qi);
    StepNormals<Real, GAUSS> rng(a.seed, a.path_offset + (unsigned long long)i, a.slice);
    run_slice_steps<false>(p, rng, a.nsteps);
    if (p.overflowed()) {      // rare: |log sigma| left [-700, 700] somewhere on this path -> redo it with the per-step clamp
      p.load(xi, vi, qi);
      run_slice_steps<true>(p, rng, a.nsteps);
    }
    const Real xT = p.x();
    a.x[i] = xT;
    a.v[i] = p.sigma();
    a.q[i] = p.q();
    // spots_t = forward*np.exp(x0); nanmean over all paths (utils/mc_payoffs.py:61-62)
    const double spot = a.forward * exp((double)xT);
    if (spot == spot) {
      acc[0] += spot;
      acc[1] += 1.0;
    }
  }
  block_sum<2, kSliceThreads>(acc, red);
  if (threadIdx.x == 0) {
    a.partials[2 * blockIdx.x + 0] = acc[0];
    a.partials[2 * blockIdx.x + 1] = acc[1];
  }
}

// out[k] = sum_b partials[b*K + k] for k < K_out, fixed order: one warp per k, lanes stride over b, shuffle tree.
// With a P2P context the same kernel PUBLISHES the K_out values into every peer's mailbox (stores to NVLink-mapped peer memory)
// and then signals the epoch -- the producer half of the exchange, fused into the reduction that produces the values (p2p.cuh).
__global__ void __launch_bounds__(256) reduce_partials_kernel(const double* __restrict__ partials, int nblk, int K, int K_out,
                                                              double* __restrict__ out, P2pPublish pub) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int k = warp; k < K_out; k += nw) {
    double s = 0.0;
    for (int b = lane; b < nblk; b += 32) s += partials[(size_t)b * K + k];
    s = warp_sum(s);
    if (lane == 0) {
      out[k] = s;
      if (pub.world) p2p_store(pub, k, s);
    }
  }
  if (pub.world) {
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) p2p_signal(pub);
  }
}

// publish K values that are already final on this rank (ranks without local paths, tests)
__global__ void p2p_publish_kernel(const double* __restrict__ vals, int K, P2pPublish pub) {
  for (int k = threadIdx.x; k < K; k += blockDim.x) p2p_store(pub, k, vals ? vals[k] : 0.0);
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) p2p_signal(pub);
}

// gather K values of the current epoch into out[] (tests; the product consumes them inside the payoff / finalize kernels)
__global__ void p2p_gather_kernel(P2pGather gat, int K, double* __restrict__ out) {
  for (int k = threadIdx.x; k < K; k += blockDim.x) out[k] = p2p_gather(gat, k);
}

// --------------------------------------------------------------------------------------------------------------------
// strict fixed-random steppers (parity entry points): reference evaluation order, no FMA contraction
// --------------------------------------------------------------------------------------------------------------------
struct LogsvRaw {
  double theta, kappa1, kappa2, beta, volvol, eta, alpha, adj, dt;
};

__global__ void __launch_bounds__(kThreads) logsv_step_fixed_kernel(double* __restrict__ x, double* __restrict__ sigma,
                                                                   double* __restrict__ qvar, const double* __restrict__ W0,
                                                                   const double* __restrict__ W1, int S, long long N, LogsvRaw r) {
  // pricers/logsv_pricer.py:1027-1047, expression by expression (fastmath=False in the reference)
  const double sdt = __dsqrt_rn(r.dt);
  const double vartheta2 = __dadd_rn(__dmul_rn(r.beta, r.beta), __dmul_rn(r.volvol, r.volvol));
  const double eta2 = __dmul_rn(r.eta, r.eta);
  const double k1theta = __dmul_rn(r.kappa1, r.theta);
  const double half_alpha = __dmul_rn(r.alpha, 0.5);
  const double half_vt2 = __dmul_rn(0.5, vartheta2);
  const long long stride = (long long)gridDim.x * kThreads;
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < N; i += stride) {
    double xi = x[i], si = sigma[i], qi = qvar[i];
    double L = log(si);
    for (int s = 0; s < S; ++s) {
      const double w0 = __dmul_rn(sdt, __ldg(W0 + (size_t)s * N + i));
      const double w1 = __dmul_rn(sdt, __ldg(W1 + (size_t)s * N + i));
      const double s2dt = __dmul_rn(__dmul_rn(__dmul_rn(eta2, si), si), r.dt);
      xi = __dadd_rn(__dadd_rn(xi, __dmul_rn(half_alpha, s2dt)), __dmul_rn(__dmul_rn(r.eta, si), w0));
      double d = __dadd_rn(__dadd_rn(__ddiv_rn(k1theta, si), -r.kappa1), __dmul_rn(r.kappa2, __dadd_rn(r.theta, -si)));
      d = __dadd_rn(__dadd_rn(d, __dmul_rn(r.adj, si)), -half_vt2);
      L = __dadd_rn(__dadd_rn(__dadd_rn(L, __dmul_rn(d, r.dt)), __dmul_rn(r.beta, w0)), __dmul_rn(r.volvol, w1));
      si = exp(L);
      qi = __dadd_rn(qi, __dmul_rn(0.5, __dadd_rn(s2dt, __dmul_rn(__dmul_rn(__dmul_rn(eta2, si), si), r.dt))));
    }
    x[i] = xi;
    sigma[i] = si;
    qvar[i] = qi;
  }
}

// Throughput variant of the fixed-random stepper for the device-resident calibration loop: same normals from HBM, but the
// per-step update of the fused kernel (LogsvPath<double>: folded constants, shared-polynomial exp pair, FMA) -- about half the
// fp64 instructions of the strict kernel, so the 16 B/path-step HBM stream becomes the bound.  Agrees with the strict kernel to
// ~1e-14 (tests/test_gpu_mc.py::test_device_resident_fixed_randoms_chain).
__global__ void __launch_bounds__(kThreads) logsv_step_fixed_fast_kernel(double* __restrict__ x, double* __restrict__ sigma,
                                                                        double* __restrict__ qvar, const double* __restrict__ W0,
                                                                        const double* __restrict__ W1, int S, long long N,
                                                                        LogsvConsts consts) {
  exp_table_init();
  LogsvPath<double> p(consts);
  const long long stride = (long long)gridDim.x * kThreads;
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < N; i += stride) {
    p.load(x[i], sigma[i], qvar[i]);
    for (int s = 0; s < S; ++s) p.step<true>(__ldg(W0 + (size_t)s * N + i), __ldg(W1 + (size_t)s * N + i));
    x[i] = p.x();
    sigma[i] = p.sigma();
    qvar[i] = p.q();
  }
}

__global__ void __launch_bounds__(kThreads) heston_step_fixed_kernel(double* __restrict__ x, double* __restrict__ var,
                                                                    double* __restrict__ qvar, const double* __restrict__ W0,
                                                                    const double* __restrict__ W1, int S, long long N,
                                                                    b200sv_heston_params p, double dt) {
  // pricers/heston_pricer.py:366-379
  const double sdt = __dsqrt_rn(dt);
  const double rho_1 = __dsqrt_rn(__dadd_rn(1.0, -__dmul_rn(p.rho, p.rho)));
  const long long stride = (long long)gridDim.x * kThreads;
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < N; i += stride) {
    double xi = x[i], vi = var[i], qi = qvar[i];
    for (int s = 0; s < S; ++s) {
      const double w0 = __dmul_rn(sdt, __ldg(W0 + (size_t)s * N + i));
      const double w1 = __dmul_rn(sdt, __ldg(W1 + (size_t)s * N + i));
      const double sig = __dsqrt_rn(vi);
      const double vdt = __dmul_rn(vi, dt);
      xi = __dadd_rn(__dadd_rn(xi, -__dmul_rn(0.5, vdt)), __dmul_rn(sig, w0));
      qi = __dadd_rn(qi, vdt);
      const double drift = __dmul_rn(__dmul_rn(p.kappa, __dadd_rn(p.theta, -vi)), dt);
      const double diff = __dmul_rn(__dmul_rn(sig, p.volvol), __dadd_rn(__dmul_rn(p.rho, w0), __dmul_rn(rho_1, w1)));
      vi = __dadd_rn(__dadd_rn(vi, drift), diff);
      vi = vi < 1e-4 ? 1e-4 : vi;   // np.maximum(var0, 1e-4): NaN stays NaN
    }
    x[i] = xi;
    var[i] = vi;
    qvar[i] = qi;
  }
}

// Full volatility paths sigma_t[(S+1)][N]: simulate_vol_paths (pricers/logsv_pricer.py:870-947).  One normal per step
// (vartheta * w1), drift evaluated at the current step, reference evaluation order (it is plain numpy, no fastmath).
// W != nullptr: caller-supplied SCALED increments [S][N] ("brownians"); else sqrt(dt) * Z0 of the device Philox stream
// (gauss f64: call = step, first normal of the pair).  Output-bandwidth bound: 8 B written per path-step.
__global__ void __launch_bounds__(kThreads) logsv_vol_paths_kernel(double* __restrict__ sigma_t, const double* __restrict__ W, int S,
                                                                  long long N, LogsvRaw r, double v0, unsigned long long seed,
                                                                  unsigned long long path_offset) {
  const double sdt = __dsqrt_rn(r.dt);
  const double vartheta2 = __dadd_rn(__dmul_rn(r.beta, r.beta), __dmul_rn(r.volvol, r.volvol));
  const double vartheta = __dsqrt_rn(vartheta2);
  const double k1theta = __dmul_rn(r.kappa1, r.theta);
  const double half_vt2 = __dmul_rn(0.5, vartheta2);
  gauss64_table_init();
  const long long stride = (long long)gridDim.x * kThreads;
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < N; i += stride) {
    double si = v0;
    double L = log(si);
    sigma_t[i] = si;
    StepNormals<double, kGaussF64> rng(seed, path_offset + (unsigned long long)i, 0u);
    for (int s = 0; s < S; ++s) {
      double w1;
      if (W) {
        w1 = __ldg(W + (size_t)s * N + i);
      } else {
        double z0, z1;
        rng.get((uint32_t)s, z0, z1);
        w1 = __dmul_rn(sdt, z0);
      }
      double d = __dadd_rn(__dadd_rn(__ddiv_rn(k1theta, si), -r.kappa1), __dmul_rn(r.kappa2, __dadd_rn(r.theta, -si)));
      d = __dadd_rn(__dadd_rn(d, __dmul_rn(r.adj, si)), -half_vt2);
      L = __dadd_rn(__dadd_rn(L, __dmul_rn(d, r.dt)), __dmul_rn(vartheta, w1));
      si = exp(L);
      sigma_t[(size_t)(s + 1) * N + i] = si;
    }
  }
}

// (sum F e^x over non-NaN, count) partials for externally supplied states (b200sv_mc_payoffs)
__global__ void __launch_bounds__(kThreads) spot_moments_kernel(const double* __restrict__ x, long long n, double forward,
                                                               double* __restrict__ partials) {
  __shared__ double red[2 * kThreads / 32];
  double acc[2] = {0.0, 0.0};
  const long long stride = (long long)gridDim.x * kThreads;
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += stride) {
    const double spot = forward * exp(x[i]);
    if (spot == spot) {
      acc[0] += spot;
      acc[1] += 1.0;
    }
  }
  block_sum<2, kThreads>(acc, red);
  if (threadIdx.x == 0) {
    partials[2 * blockIdx.x + 0] = acc[0];
    partials[2 * blockIdx.x + 1] = acc[1];
  }
}

// --------------------------------------------------------------------------------------------------------------------
// payoff sums: utils/mc_payoffs.py:61-88
// --------------------------------------------------------------------------------------------------------------------
// General payoffs (any mix of C / P / IC / IP): per-strike NaN-skipping counts, IEEE division for the inverse payoffs.
// payoff_general_block / payoff_vanilla_block: the work of ONE CTA for the strike chunk starting at j0 -- grid-stride over the paths with
// `nblocks` CTAs, block-reduce, write this CTA's partial row.  Called by the stand-alone payoff kernels (blockIdx.y = chunk) and by the
// cooperative whole-chain kernel (chunks looped inside).
template <typename Real>
__device__ __forceinline__ void payoff_general_block(const Real* __restrict__ x, const Real* __restrict__ q, long long n, double ttm, double forward,
                                                     const double* __restrict__ strikes, const int8_t* __restrict__ types, int J, int variable_type,
                                                     double corr, double* __restrict__ partials, int Kpad, int j0, int block, int nblocks) {
  __shared__ double red[3 * kStrikeChunk * kThreads / 32];
  double kk[kStrikeChunk];
  int ty[kStrikeChunk];
#pragma unroll
  for (int c = 0; c < kStrikeChunk; ++c) {
    const int j = j0 + c;
    kk[c] = j < J ? strikes[j] : 0.0;
    ty[c] = j < J ? (int)types[j] : -1;
  }
  const bool is_qvar = variable_type == B200SV_Q_VAR;
  double acc[3 * kStrikeChunk];
#pragma unroll
  for (int c = 0; c < 3 * kStrikeChunk; ++c) acc[c] = 0.0;
  const long long stride = (long long)nblocks * kThreads;
  for (long long i = (long long)block * kThreads + threadIdx.x; i < n; i += stride) {
    const double spot = forward * exp((double)x[i]) - corr;
    const double under = is_qvar ? (double)q[i] / ttm : spot;
#pragma unroll
    for (int c = 0; c < kStrikeChunk; ++c) {
      if (ty[c] >= 0) {
        const bool is_put = (ty[c] & 1);
        double pay = is_put ? (under < kk[c] ? kk[c] - under : 0.0) : (under > kk[c] ? under - kk[c] : 0.0);
        // np.where(np.greater(nan, k), ..., 0.0) == 0.0: a NaN underlying pays 0 for C/P and 0/NaN = NaN (skipped) for IC/IP
        if (ty[c] >= 2) pay = pay / spot;
        if (pay == pay) {
          acc[3 * c + 0] += pay;
          acc[3 * c + 1] += pay * pay;
          acc[3 * c + 2] += 1.0;
        }
      }
    }
  }
  block_sum<3 * kStrikeChunk, kThreads>(acc, red);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int c = 0; c < 3 * kStrikeChunk; ++c) partials[(size_t)block * Kpad + 3 * j0 + c] = acc[c];
  }
}

// Vanilla-only payoffs ('C' / 'P' in every slot of the slice): pay = max(+-(U - K), 0) is never NaN (numpy's
// where(greater(nan, K), ., 0.0) is 0.0 as well), so every path counts and the count is simply n; no division, no branches.
// ~6 instructions per (path, strike) + one exp per (path, chunk); kPayoffUnroll loads in flight per thread.
constexpr int kPayoffUnroll = 4;
template <typename Real>
__device__ __forceinline__ void payoff_vanilla_block(const Real* __restrict__ x, const Real* __restrict__ q, long long n, double ttm, double forward,
                                                     const double* __restrict__ strikes, const int8_t* __restrict__ types, int J, int variable_type,
                                                     double corr, double* __restrict__ partials, int Kpad, int j0, int block, int nblocks) {
  __shared__ double red[2 * kStrikeChunk * kThreads / 32];
  double sg[kStrikeChunk], nk[kStrikeChunk];      // pay = max(sg*U + nk, 0), nk = -sg*K
#pragma unroll
  for (int c = 0; c < kStrikeChunk; ++c) {
    const int j = j0 + c;
    const double sgn = (j < J && (types[j] & 1)) ? -1.0 : 1.0;
    sg[c] = sgn;
    nk[c] = j < J ? -sgn * strikes[j] : -INFINITY;   // unused slot: max(U - inf, 0) = 0
  }
  const bool is_qvar = variable_type == B200SV_Q_VAR;
  const double inv_ttm = 1.0 / ttm;
  double acc[2 * kStrikeChunk];
#pragma unroll
  for (int c = 0; c < 2 * kStrikeChunk; ++c) acc[c] = 0.0;
  auto accumulate = [&](double under) {
#pragma unroll
    for (int c = 0; c < kStrikeChunk; ++c) {
      const double d = fma(sg[c], under, nk[c]);
      const double pay = d > 0.0 ? d : 0.0;
      acc[2 * c] += pay;
      acc[2 * c + 1] = fma(pay, pay, acc[2 * c + 1]);
    }
  };
  const long long stride = (long long)nblocks * kThreads;
  long long i = (long long)block * kThreads + threadIdx.x;
  if (!is_qvar) {
    for (; i + (kPayoffUnroll - 1) * stride < n; i += kPayoffUnroll * stride) {
      double xs[kPayoffUnroll];
#pragma unroll
      for (int u = 0; u < kPayoffUnroll; ++u) xs[u] = (double)x[i + u * stride];
#pragma unroll
      for (int u = 0; u < kPayoffUnroll; ++u) accumulate(forward * exp(xs[u]) - corr);
    }
    for (; i < n; i += stride) accumulate(forward * exp((double)x[i]) - corr);
  } else {
    for (; i < n; i += stride) accumulate((double)q[i] * inv_ttm);
  }
  block_sum<2 * kStrikeChunk, kThreads>(acc, red);
  if (threadIdx.x == 0) {
    // count of paths this CTA visited (same for every strike)
    const long long first = (long long)block * kThreads;
    long long cnt = 0;
    if (first < n) {
      const long long full_rounds = (n - first) / stride, rem = (n - first) % stride;
      cnt = full_rounds * kThreads + (rem < kThreads ? rem : kThreads);
    }
#pragma unroll
    for (int c = 0; c < kStrikeChunk; ++c) {
      partials[(size_t)block * Kpad + 3 * (j0 + c) + 0] = acc[2 * c];
      partials[(size_t)block * Kpad + 3 * (j0 + c) + 1] = acc[2 * c + 1];
      partials[(size_t)block * Kpad + 3 * (j0 + c) + 2] = (double)cnt;
    }
  }
}

// correnction = np.nanmean(spots_t) - forward; multi-GPU: the GLOBAL (sum, count) is gathered from the peers' mailbox writes here
__device__ __forceinline__ double payoff_recentring(const double* __restrict__ moments, double forward, const P2pGather& gat) {
  __shared__ double sh_mom[2];
  if (threadIdx.x < 2) sh_mom[threadIdx.x] = gat.world ? p2p_gather(gat, threadIdx.x) : moments[threadIdx.x];
  __syncthreads();
  return sh_mom[0] / sh_mom[1] - forward;
}

template <typename Real>
__global__ void __launch_bounds__(kThreads) payoff_kernel(const Real* __restrict__ x, const Real* __restrict__ q, long long n,
                                                         double ttm, double forward, const double* __restrict__ strikes,
                                                         const int8_t* __restrict__ types, int J, int variable_type,
                                                         const double* __restrict__ moments, double* __restrict__ partials,
                                                         int Kpad /* = 3 * kStrikeChunk * gridDim.y */, P2pGather gat) {
  const double corr = payoff_recentring(moments, forward, gat);
  payoff_general_block<Real>(x, q, n, ttm, forward, strikes, types, J, variable_type, corr, partials, Kpad, blockIdx.y * kStrikeChunk, blockIdx.x, gridDim.x);
}

template <typename Real>
__global__ void __launch_bounds__(kThreads) payoff_vanilla_kernel(const Real* __restrict__ x, const Real* __restrict__ q, long long n,
                                                                 double ttm, double forward, const double* __restrict__ strikes,
                                                                 const int8_t* __restrict__ types, int J, int variable_type,
                                                                 const double* __restrict__ moments, double* __restrict__ partials,
                                                                 int Kpad, P2pGather gat) {
  const double corr = payoff_recentring(moments, forward, gat);
  payoff_vanilla_block<Real>(x, q, n, ttm, forward, strikes, types, J, variable_type, corr, partials, Kpad, blockIdx.y * kStrikeChunk, blockIdx.x, gridDim.x);
}

// optional fused Black-76 inversion of the prices just assembled (batched calibration objective): needs strikes/types/forward/ttm
struct IvolSpec {
  const double* strikes;
  const int8_t* types;
  double forward, ttm;
  double* ivols;       // nullptr: skip
};

__global__ void payoff_finalize_kernel(const double* __restrict__ sums, int J, double discfactor, double total_paths,
                                       double* __restrict__ prices, double* __restrict__ stderrs, P2pGather gat, IvolSpec iv = IvolSpec{}) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= J) return;
  const double s1 = gat.world ? p2p_gather(gat, 3 * j) : sums[3 * j];
  const double s2 = gat.world ? p2p_gather(gat, 3 * j + 1) : sums[3 * j + 1];
  const double cnt = gat.world ? p2p_gather(gat, 3 * j + 2) : sums[3 * j + 2];
  const double mean = s1 / cnt;
  double var = s2 / cnt - mean * mean;
  var = var > 0.0 ? var : 0.0;
  prices[j] = discfactor * mean;                               // discfactor*np.nanmean(payoff)
  stderrs[j] = discfactor * sqrt(var) / sqrt(total_paths);     // discfactor*np.nanstd(payoff) / sqrt(x0.shape[0])
  if (iv.ivols) iv.ivols[j] = black_implied_vol(iv.forward, iv.strikes[j], iv.ttm, discfactor, discfactor * mean, iv.types[j]);
}

// --------------------------------------------------------------------------------------------------------------------
// the whole chain in ONE persistent cooperative kernel (single GPU, fp64 state)
// --------------------------------------------------------------------------------------------------------------------
// north_star: "one persistent-thread kernel ... with a warp-shuffle block reduction of terminal payoffs into per-strike sums/sum-squares
// staged in shared memory".  The forward re-centring of utils/mc_payoffs.py:61-63 needs the mean over ALL paths before any payoff, so
// a chain is two grid-wide phases per maturity; here they are separated by grid.sync() instead of kernel boundaries:
//   for every maturity:  slice phase (Philox + stepper, state in registers, per-CTA moments)  -> grid.sync
//                        every CTA reduces the per-CTA moments in the same fixed order -> correction; payoff phase (per-CTA per-strike
//                        partial sums, the same block functions as the stand-alone payoff kernels)               -> grid.sync
//                        CTA j (j < J) reduces column j over the CTAs in fixed order and finalises price / std error / implied vol
// One launch instead of 5 per maturity: a 4-maturity chain at 1e4 paths drops from 0.24 ms to the latency of the dependent steps.
// The grid is one co-resident wave (cudaLaunchCooperativeKernel); buffers are reused across maturities -- the two syncs order every
// write after the last read of the previous use (a CTA cannot pass sync k+1 before every CTA has arrived, i.e. finished reading).
template <typename Consts>
struct CoopSliceSpec {
  Consts c;
  int nsteps, jo, J, kinds;
  double forward, ttm, discfactor;
};

struct CoopArgs {
  double *x, *v, *q;              // state SoA [n]
  long long n;
  double v_init;
  unsigned long long seed;
  int M, variable_type;
  const double* strikes;          // [Jtot]
  const int8_t* types;
  double* part_mom;               // [grid][2]
  double* part_pay;               // [grid][Kpad_max]
  int Kpad_max;
  double total_paths;
  double *prices, *stderrs, *ivols;   // [Jalloc] each; ivols may be nullptr
};

template <typename Path, typename Consts, int GAUSS>
__global__ void __launch_bounds__(kSliceThreads, B200SV_SLICE_MINBLOCKS) mc_chain_coop_kernel(CoopArgs a, const CoopSliceSpec<Consts>* __restrict__ specs) {
  static_assert(kSliceThreads == kThreads, "the payoff block functions and the slice phase share one CTA size");
  namespace cg = cooperative_groups;
  cg::grid_group grid = cg::this_grid();
  __shared__ double red[2 * kSliceThreads / 32];
  __shared__ double sh_corr;
  exp_table_init();
  if constexpr (GAUSS != kGaussF32) gauss64_table_init();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long stride = (long long)gridDim.x * kSliceThreads;
  for (int m = 0; m < a.M; ++m) {
    const CoopSliceSpec<Consts> sp = specs[m];
    // ---- slice phase ------------------------------------------------------------------------------------------------------------
    {
      double acc[2] = {0.0, 0.0};
      Path p(sp.c);
      for (long long i = (long long)blockIdx.x * kSliceThreads + threadIdx.x; i < a.n; i += stride) {
        double xi = 0.0, vi = a.v_init, qi = 0.0;
        if (m > 0) {
          xi = a.x[i];
          vi = a.v[i];
          qi = a.q[i];
        }
        p.load(xi, vi, qi);
        StepNormals<double, GAUSS> rng(a.seed, (unsigned long long)i, (unsigned int)m);
        run_slice_steps<false>(p, rng, sp.nsteps);
        if (p.overflowed()) {
          p.load(xi, vi, qi);
          run_slice_steps<true>(p, rng, sp.nsteps);
        }
        const double xT = p.x();
        a.x[i] = xT;
        a.v[i] = p.sigma();
        a.q[i] = p.q();
        const double spot = sp.forward * exp(xT);
        if (spot == spot) {
          acc[0] += spot;
          acc[1] += 1.0;
        }
      }
      block_sum<2, kSliceThreads>(acc, red);
      if (threadIdx.x == 0) {
        a.part_mom[2 * blockIdx.x + 0] = acc[0];
        a.part_mom[2 * blockIdx.x + 1] = acc[1];
      }
    }
    if (sp.J == 0) {           // nothing to price at this maturity: the state is stored, go on (uniform across the grid: no sync imbalance)
      grid.sync();
      continue;
    }
    grid.sync();
    // ---- global moments (same fixed order in every CTA: lanes stride over the CTAs, shuffle tree) -> correction ----------------------
    if (warp == 0) {
      double s0 = 0.0, s1 = 0.0;
      for (int b = lane; b < (int)gridDim.x; b += 32) {
        s0 += __ldcg(a.part_mom + 2 * b);
        s1 += __ldcg(a.part_mom + 2 * b + 1);
      }
      s0 = warp_sum(s0);
      s1 = warp_sum(s1);
      if (lane == 0) sh_corr = s0 / s1 - sp.forward;
    }
    __syncthreads();
    const double corr = sh_corr;
    // ---- payoff phase ---------------------------------------------------------------------------------------------------------------
    const int chunks = (sp.J + kStrikeChunk - 1) / kStrikeChunk;
    const int Kpad = 3 * kStrikeChunk * chunks;
    for (int ch = 0; ch < chunks; ++ch) {
      if (sp.kinds == 1)
        payoff_vanilla_block<double>(a.x, a.q, a.n, sp.ttm, sp.forward, a.strikes + sp.jo, a.types + sp.jo, sp.J, a.variable_type, corr, a.part_pay, Kpad,
                                     ch * kStrikeChunk, blockIdx.x, gridDim.x);
      else
        payoff_general_block<double>(a.x, a.q, a.n, sp.ttm, sp.forward, a.strikes + sp.jo, a.types + sp.jo, sp.J, a.variable_type, corr, a.part_pay, Kpad,
                                     ch * kStrikeChunk, blockIdx.x, gridDim.x);
    }
    grid.sync();
    // ---- finalise: strike j by CTA j % grid (warp 0), fixed-order sum over the CTAs ---------------------------------------------------
    for (int j = blockIdx.x; j < sp.J; j += gridDim.x) {
      if (warp == 0) {
        double s1 = 0.0, s2 = 0.0, cnt = 0.0;
        for (int b = lane; b < (int)gridDim.x; b += 32) {
          const double* row = a.part_pay + (size_t)b * Kpad + 3 * j;
          s1 += __ldcg(row);
          s2 += __ldcg(row + 1);
          cnt += __ldcg(row + 2);
        }
        s1 = warp_sum(s1);
        s2 = warp_sum(s2);
        cnt = warp_sum(cnt);
        if (lane == 0) {
          const double mean = s1 / cnt;
          double var = s2 / cnt - mean * mean;
          var = var > 0.0 ? var : 0.0;
          a.prices[sp.jo + j] = sp.discfactor * mean;
          a.stderrs[sp.jo + j] = sp.discfactor * sqrt(var) / sqrt(a.total_paths);
          if (a.ivols)
            a.ivols[sp.jo + j] = black_implied_vol(sp.forward, a.strikes[sp.jo + j], sp.ttm, sp.discfactor, sp.discfactor * mean, a.types[sp.jo + j]);
        }
      }
    }
    // the next maturity's slice phase overwrites part_mom only: every CTA has read it before arriving at the sync above
  }
}

// --------------------------------------------------------------------------------------------------------------------
// debug / parity export of the normals the fused kernel draws
// --------------------------------------------------------------------------------------------------------------------
template <int GAUSS>
__global__ void device_normals_kernel(unsigned long long seed, unsigned long long path0, long long n, unsigned int slice,
                                      int nsteps, double* __restrict__ z0, double* __restrict__ z1) {
  if constexpr (GAUSS != kGaussF32) gauss64_table_init();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  StepNormals<double, GAUSS> rng(seed, path0 + (unsigned long long)i, slice);
  if constexpr (GAUSS == kGaussF64) {
    for (int s = 0; s < nsteps; ++s) {
      double a, b;
      rng.get((uint32_t)s, a, b);
      z0[(size_t)s * n + i] = a;
      z1[(size_t)s * n + i] = b;
    }
  } else {
    for (int c = 0; 2 * c < nsteps; ++c) {
      double a0, a1, b0, b1;
      rng.get2((uint32_t)c, a0, a1, b0, b1);
      z0[(size_t)(2 * c) * n + i] = a0;
      z1[(size_t)(2 * c) * n + i] = a1;
      if (2 * c + 1 < nsteps) {
        z0[(size_t)(2 * c + 1) * n + i] = b0;
        z1[(size_t)(2 * c + 1) * n + i] = b1;
      }
    }
  }
}

// exp_pair self-test kernel (tests): out[2i] = exp(L), out[2i+1] = exp(-L)
__global__ void exp_pair_kernel(const double* __restrict__ L, long long n, double* __restrict__ out) {
  exp_table_init();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double a, b;
  exp_pair(L[i], a, b);
  out[2 * i] = a;
  out[2 * i + 1] = b;
}

// the stepper's variant on table units: out[2i] = exp(Ls ln2/256), out[2i+1] = exp(-Ls ln2/256), |Ls| clamped like the stepper does
__global__ void exp_pair_scaled_kernel(const double* __restrict__ Ls, long long n, double* __restrict__ out) {
  exp_table_init();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double a, b;
  exp_pair_scaled(clamp_log_scaled(Ls[i]), a, b);
  out[2 * i] = a;
  out[2 * i + 1] = b;
}

// --------------------------------------------------------------------------------------------------------------------
// host side
// --------------------------------------------------------------------------------------------------------------------
// host-side state of one rank's mailbox (p2p.cuh); created / connected through the b200sv_p2p_* entry points
struct P2pCtx {
  int world, rank, kmax;
  char* mail;                    // own mailbox (cudaMalloc, IPC-exported)
  char* peer[kMaxPeers];         // every rank's mailbox mapped into this process (peer[rank] == mail)
  size_t vals_bytes;             // 2 * world * kmax * 8; flags follow
  unsigned long long published;  // epoch of the last exchange this rank published
  unsigned long long consumed;   // epoch of the last exchange this rank gathered
  double* scratch;               // 1 double (tail of the own mailbox allocation): sink of the protocol-keeping gather below
  unsigned int* status;          // 1 word after scratch: timeout bits set by p2p_gather (p2p.cuh)
  unsigned int spin_limit;
};
static P2pGather make_gather(P2pCtx* c);
__global__ void p2p_gather_kernel(P2pGather g, int K, double* __restrict__ out);
// The double-buffer argument of p2p.cuh needs "publish e+1 only after gathering e" on every rank.  A caller that skips a gather (a
// maturity without strikes, a rank without paths) gets it inserted here: a 1-thread kernel that waits for epoch e's flags.
static P2pPublish make_publish(P2pCtx* c, cudaStream_t st) {
  P2pPublish p{};
  if (!c) return p;
  if (c->consumed < c->published) p2p_gather_kernel<<<1, 32, 0, st>>>(make_gather(c), 1, c->scratch);
  p.world = c->world;
  p.epoch = ++c->published;
  const int slot = (int)(p.epoch & 1ull);
  for (int s = 0; s < c->world; ++s) {
    p.peer_vals[s] = (double*)c->peer[s] + ((size_t)slot * c->world + c->rank) * c->kmax;
    p.peer_flags[s] = (unsigned long long*)(c->peer[s] + c->vals_bytes) + (size_t)slot * c->world + c->rank;
  }
  return p;
}
static P2pGather make_gather(P2pCtx* c) {
  P2pGather g{};
  if (!c) return g;
  g.world = c->world;
  g.kmax = c->kmax;
  g.epoch = c->consumed = c->published;
  g.spin_limit = c->spin_limit;
  g.status = c->status;
  const int slot = (int)(g.epoch & 1ull);
  g.vals = (const double*)c->mail + (size_t)slot * c->world * c->kmax;
  g.flags = (const unsigned long long*)(c->mail + c->vals_bytes) + (size_t)slot * c->world;
  return g;
}

// int(ttm * n) + 1 and dt = linspace(0, ttm, S+1)[1] - [0] (utils/funcs.py:44-47; numpy linspace: step = ttm / S, y[1] = 1*step)
static void time_grid(double ttm, int n_per_year, int* S, double* dt) {
  *S = (int)(ttm * (double)n_per_year) + 1;
  *dt = (*S == 1) ? ttm : ttm / (double)(*S);   // linspace sets the LAST point to `stop` exactly; with S == 1 y[1] is that point
}

// model -> (path, constants) of the slice and chain kernels: 0 LogSV, 1 Heston floor-Euler, 2 Heston QE
template <int MODEL>
struct ChainModel;
template <>
struct ChainModel<0> {
  template <typename Real>
  using Path = LogsvPath<Real>;
  using Consts = LogsvConsts;
};
template <>
struct ChainModel<1> {
  template <typename Real>
  using Path = HestonPath<Real, false>;
  using Consts = HestonConsts;
};
template <>
struct ChainModel<2> {
  template <typename Real>
  using Path = HestonPath<Real, true>;
  using Consts = HestonConsts;
};

template <int MODEL, typename Real, int G64>
static int launch_slice_t(void* x, void* v, void* q, long long n, long long path_offset, int init, double v_init, int nsteps,
                          int slice_index, double forward, uint64_t seed, const typename ChainModel<MODEL>::Consts& c,
                          double* moments_out, cudaStream_t st, P2pCtx* p2p) {
  const auto kernel = mc_slice_kernel<typename ChainModel<MODEL>::template Path<Real>, typename ChainModel<MODEL>::Consts, Real, G64>;
  SliceArgs<Real> a;
  a.x = (Real*)x;
  a.v = (Real*)v;
  a.q = (Real*)q;
  a.n = n;
  a.path_offset = (unsigned long long)path_offset;
  a.init = init;
  a.v_init = v_init;
  a.nsteps = nsteps;
  a.slice = (unsigned int)slice_index;
  a.seed = seed;
  a.forward = forward;
  Grid g = persistent_grid(kernel, kSliceThreads, n);
  size_t dyn_smem = 0;
#ifdef B200SV_TUNING   // occupancy sweep for profiles/: cap resident CTAs per SM with dynamic shared memory (tuning builds only)
  if (const char* e = getenv("B200SV_DEBUG_BLOCKS_PER_SM")) {
    const int bps = atoi(e);
    if (bps > 0) {
      dyn_smem = (size_t)(200 * 1024) / bps;
      if constexpr (MODEL == 0) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_smem);
      g.blocks = (int)std::min<long long>((long long)148 * bps, (n + kSliceThreads - 1) / kSliceThreads);
    }
  }
#endif
  DevBuf<double> partials(st);
  ensure_pool_threshold();      // device-level callers too: a pool that trims at every synchronisation stalls the whole node (DESIGN.md 5)
  B200SV_CUDA(partials.alloc(2 * (size_t)g.blocks));
  a.partials = partials.p;
  kernel<<<g.blocks, g.threads, dyn_smem, st>>>(a, c);
  if (int rc = launched("mc_slice_kernel")) return rc;
  reduce_partials_kernel<<<1, 64, 0, st>>>(partials.p, g.blocks, 2, 2, moments_out, make_publish(p2p, st));   // exchange #1 (producer)
  return launched("reduce_partials_kernel");
}

// B200SV_GAUSS_* bits -> GaussMode (philox.cuh); -1 = contradictory
static int gauss_mode(int flags) {
  const bool g64 = flags & B200SV_GAUSS_F64, paired = flags & B200SV_GAUSS_F64_PAIRED;
  if (g64 && paired) return -1;
  return paired ? kGaussF64Paired : (g64 ? kGaussF64 : kGaussF32);
}

// the state / Gaussian flag combinations the slice kernels are built for
static int check_slice_flags(int flags) {
  const int g = gauss_mode(flags);
  if (g < 0) return fail(-1, "invalid argument: B200SV_GAUSS_F64 and B200SV_GAUSS_F64_PAIRED are mutually exclusive");
  if ((flags & B200SV_STATE_F32) && g == kGaussF64Paired) return fail(-1, "invalid argument: the paired Gaussian check mode needs fp64 state");
  return 0;
}

// MODEL 0 = LogSV, 1 = Heston (the QE scheme, c.qe, runs model 2)
template <int MODEL>
static int launch_slice(void* x, void* v, void* q, long long n, long long path_offset, int init, double v_init, int nsteps,
                        int slice_index, double forward, uint64_t seed, int flags, const typename ChainModel<MODEL>::Consts& c,
                        double* moments_out, cudaStream_t st, P2pCtx* p2p = nullptr) {
  if constexpr (MODEL == 1)
    if (c.qe) return launch_slice<2>(x, v, q, n, path_offset, init, v_init, nsteps, slice_index, forward, seed, flags, c, moments_out, st, p2p);
  if (int rc = check_slice_flags(flags)) return rc;
  const bool f32 = flags & B200SV_STATE_F32;
  const int g = gauss_mode(flags);
#define B200SV_SLICE_CASE(REAL, G) \
  return launch_slice_t<MODEL, REAL, G>(x, v, q, n, path_offset, init, v_init, nsteps, slice_index, forward, seed, c, moments_out, st, p2p)
  if (!f32 && g == kGaussF32) B200SV_SLICE_CASE(double, kGaussF32);
  if (!f32 && g == kGaussF64) B200SV_SLICE_CASE(double, kGaussF64);
  if (!f32 && g == kGaussF64Paired) B200SV_SLICE_CASE(double, kGaussF64Paired);
  if (f32 && g == kGaussF32) B200SV_SLICE_CASE(float, kGaussF32);
  B200SV_SLICE_CASE(float, kGaussF64);
#undef B200SV_SLICE_CASE
}

// kinds: bit 0 = some 'C'/'P', bit 1 = some 'IC'/'IP' in this slice; 0 = unknown (device-level callers) -> general kernel
template <typename Real>
static int launch_payoff_t(const void* x, const void* q, long long n, double ttm, double forward, const double* strikes,
                           const int8_t* types, int J, int variable_type, int kinds, const double* moments, double* sums_out,
                           cudaStream_t st, P2pCtx* p2p = nullptr) {
  if (p2p && 3 * J > p2p->kmax) return fail(-1, "P2P mailbox too small for this slice (max_values < 3*J)");
  const P2pGather gat = make_gather(p2p);      // exchange #1 (consumer): the global re-centring moments
  const int chunks = (J + kStrikeChunk - 1) / kStrikeChunk;
  const int Kpad = 3 * kStrikeChunk * chunks;
  const bool vanilla = kinds == 1;
  Grid g = vanilla ? persistent_grid(payoff_vanilla_kernel<Real>, kThreads, n, kPayoffUnroll) : persistent_grid(payoff_kernel<Real>, kThreads, n);
  g.blocks = std::max(1, g.blocks / chunks);
  DevBuf<double> partials(st);
  ensure_pool_threshold();
  B200SV_CUDA(partials.alloc((size_t)Kpad * g.blocks));
  if (vanilla)
    payoff_vanilla_kernel<Real><<<dim3(g.blocks, chunks), g.threads, 0, st>>>((const Real*)x, (const Real*)q, n, ttm, forward, strikes,
                                                                                types, J, variable_type, moments, partials.p, Kpad, gat);
  else
    payoff_kernel<Real><<<dim3(g.blocks, chunks), g.threads, 0, st>>>((const Real*)x, (const Real*)q, n, ttm, forward, strikes,
                                                                        types, J, variable_type, moments, partials.p, Kpad, gat);
  if (int rc = launched("payoff_kernel")) return rc;
  reduce_partials_kernel<<<1, 256, 0, st>>>(partials.p, g.blocks, Kpad, 3 * J, sums_out, make_publish(p2p, st));   // exchange #2 (producer)
  return launched("reduce_partials_kernel");
}

static int payoff_kinds(const int8_t* types, int J) {
  int k = 0;
  for (int j = 0; j < J; ++j) k |= (types[j] >= 2) ? 2 : 1;
  return k;
}

static int validate_chain(int M, const double* ttms, const int* offsets, const int8_t* types, int variable_type) {
  B200SV_REQUIRE(M >= 1, "M must be >= 1");
  double t0 = 0.0;
  for (int m = 0; m < M; ++m) {
    B200SV_REQUIRE(ttms[m] > t0, "ttms must be positive and strictly increasing");   // data/option_chain.py:147-153
    B200SV_REQUIRE(offsets[m + 1] >= offsets[m], "offsets must be non-decreasing");
    t0 = ttms[m];
  }
  for (int j = offsets[0]; j < offsets[M]; ++j)
    if (types[j] < 0 || types[j] > 3) return fail(-3, "unknown option payoff code");      // utils/mc_payoffs.py:83-84
  if (variable_type != B200SV_LOG_RETURN && variable_type != B200SV_Q_VAR)
    return fail(-4, "variable_type not implemented");                                      // utils/mc_payoffs.py:69-70
  return 0;
}

// The payoff stage of the host-level MC chain drivers: the chain's strikes and types on the device, the moment and sum scratch, and B sets
// of outputs [prices | std errors | implied vols if asked for] of Jalloc values each, written per (set, maturity) and copied back once.
struct ChainPayoffs {
  const double *ttms, *forwards, *discfactors;
  const int* offsets;
  const int8_t* types;
  int variable_type, B, Jtot, Jalloc, nout;
  DevBuf<double> d_strikes, d_mom, d_sums, d_out;
  DevBuf<int8_t> d_types;

  ChainPayoffs(cudaStream_t st, int M, const double* ttms, const double* forwards, const double* discfactors, const int* offsets,
               const int8_t* types, int variable_type, int B, bool ivols)
      : ttms(ttms), forwards(forwards), discfactors(discfactors), offsets(offsets), types(types), variable_type(variable_type), B(B),
        Jtot(offsets[M] - offsets[0]), Jalloc(std::max(Jtot, 1)), nout(ivols ? 3 : 2), d_strikes(st), d_mom(st), d_sums(st), d_out(st),
        d_types(st) {}

  int alloc(const double* strikes) {
    B200SV_CUDA(d_strikes.upload(strikes + offsets[0], Jtot));
    B200SV_CUDA(d_types.upload(types + offsets[0], Jtot));
    B200SV_CUDA(d_out.alloc((size_t)nout * Jalloc * B));
    B200SV_CUDA(d_mom.alloc(2));
    B200SV_CUDA(d_sums.alloc(3 * (size_t)Jalloc));
    return 0;
  }

  // payoffs of set b at maturity m (none without strikes) over the state (x, q) of n paths, re-centred with the moments in d_mom
  int run(int b, int m, const void* x, const void* q, long long n, bool f32, double total_paths, cudaStream_t st) {
    const int J = offsets[m + 1] - offsets[m], jo = offsets[m] - offsets[0];
    if (J == 0) return 0;
    const int kinds = payoff_kinds(types + offsets[m], J);
    const int rc = f32 ? launch_payoff_t<float>(x, q, n, ttms[m], forwards[m], d_strikes.p + jo, d_types.p + jo, J, variable_type, kinds, d_mom.p, d_sums.p, st)
                       : launch_payoff_t<double>(x, q, n, ttms[m], forwards[m], d_strikes.p + jo, d_types.p + jo, J, variable_type, kinds, d_mom.p, d_sums.p, st);
    if (rc) return rc;
    double* out = d_out.p + (size_t)nout * Jalloc * b;
    const IvolSpec iv{d_strikes.p + jo, d_types.p + jo, forwards[m], ttms[m], nout == 3 ? out + 2 * Jalloc + jo : nullptr};
    payoff_finalize_kernel<<<(J + 127) / 128, 128, 0, st>>>(d_sums.p, J, discfactors[m], total_paths, out + jo, out + Jalloc + jo, P2pGather{}, iv);
    return launched("payoff_finalize_kernel");
  }

  // [B][Jtot] each; ivols only if the stage was made with them
  int copy_back(double* prices, double* stderrs, double* ivols, cudaStream_t st) {
    for (int b = 0; b < B && Jtot > 0; ++b) {
      const double* out = d_out.p + (size_t)nout * Jalloc * b;
      B200SV_CUDA(cudaMemcpyAsync(prices + (size_t)b * Jtot, out, sizeof(double) * Jtot, cudaMemcpyDeviceToHost, st));
      B200SV_CUDA(cudaMemcpyAsync(stderrs + (size_t)b * Jtot, out + Jalloc, sizeof(double) * Jtot, cudaMemcpyDeviceToHost, st));
      if (ivols) B200SV_CUDA(cudaMemcpyAsync(ivols + (size_t)b * Jtot, out + 2 * Jalloc, sizeof(double) * Jtot, cudaMemcpyDeviceToHost, st));
    }
    return 0;
  }
};

// the SoA state [3][n] of a host-level call: three host arrays to and from one device buffer
static int state_to_device(double* d, size_t n, const double* a, const double* b, const double* c, cudaStream_t st) {
  B200SV_CUDA(cudaMemcpyAsync(d, a, sizeof(double) * n, cudaMemcpyHostToDevice, st));
  B200SV_CUDA(cudaMemcpyAsync(d + n, b, sizeof(double) * n, cudaMemcpyHostToDevice, st));
  B200SV_CUDA(cudaMemcpyAsync(d + 2 * n, c, sizeof(double) * n, cudaMemcpyHostToDevice, st));
  return 0;
}
static int state_to_host(const double* d, size_t n, double* a, double* b, double* c, cudaStream_t st) {
  B200SV_CUDA(cudaMemcpyAsync(a, d, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
  B200SV_CUDA(cudaMemcpyAsync(b, d + n, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
  B200SV_CUDA(cudaMemcpyAsync(c, d + 2 * n, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
  return 0;
}

// the cooperative chain kernel of a model (fp64 state; kGaussF32 or kGaussF64 draws)
template <int MODEL>
static const void* coop_kernel(int gauss) {
  using CM = ChainModel<MODEL>;
  if (gauss == kGaussF64) return (const void*)mc_chain_coop_kernel<typename CM::template Path<double>, typename CM::Consts, kGaussF64>;
  return (const void*)mc_chain_coop_kernel<typename CM::template Path<double>, typename CM::Consts, kGaussF32>;
}

// Which chain driver?  The cooperative single-launch kernel wins where launch and host overhead matter (measured on B200, BTC chain,
// profiles/r02_coop_chain.txt: 1e4 paths 0.18 vs 0.24 ms, 1e6 paths 0.75 vs 0.76 ms) and loses 5-6 % at >= 1e7 paths, where its 128-register
// budget (slice + payoff phases in one kernel) costs more than 20 launches: it serves nb_path <= kCoopMaxPaths.
// B200SV_CHAIN_COOP=0 / 1 forces the multi-launch / cooperative driver (A/B measurements, tests).
constexpr long long kCoopMaxPaths = 4000000;        // LogSV
constexpr long long kCoopMaxPathsHeston = 500000;   // Heston's cheaper step leaves less to hide the fused kernel's register budget behind: 1e6 paths
                                                    // 0.926 (cooperative) vs 0.890 ms (20 launches)
static bool use_coop_chain(int flags, long long nb_path, bool heston = false) {
  if (flags & B200SV_STATE_F32) return false;
  const int g = gauss_mode(flags);
  if (g != kGaussF32 && g != kGaussF64) return false;
  static const int mode = [] {
    const char* e = getenv("B200SV_CHAIN_COOP");
    int dev = 0, coop = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
    if (!coop) return 0;
    return e ? (e[0] == '0' ? 0 : 2) : 1;      // 0 never, 1 by size, 2 always
  }();
  return mode == 2 || (mode == 1 && nb_path <= (heston ? kCoopMaxPathsHeston : kCoopMaxPaths));
}

// Small-chain fast path: ONE stream-ordered allocation, ONE host-to-device copy (strikes, types and the per-maturity specs of all B sets in
// one blob), ONE cooperative launch per parameter set, ONE device-to-host copy.
template <int MODEL>
static int mc_chain_host_coop(const b200sv_logsv_params* lp, const b200sv_heston_params* hp, int M, const double* ttms, const double* forwards,
                              const double* discfactors, const double* etas, const int* offsets, const double* strikes, const int8_t* types,
                              long long nb_path, int nb_steps_per_year, int is_spot, int variable_type, uint64_t seed, int flags,
                              double* prices_out, double* stderr_out, int scheme, int B, double* ivols_out) {
  using Spec = CoopSliceSpec<typename ChainModel<MODEL>::Consts>;
  const int Jtot = offsets[M] - offsets[0], Jalloc = std::max(Jtot, 1);
  const int gauss = gauss_mode(flags);
  const void* kernel = MODEL == 0 ? coop_kernel<0>(gauss) : (scheme == B200SV_HESTON_QE ? coop_kernel<2>(gauss) : coop_kernel<1>(gauss));
  const int blocks = persistent_grid(kernel, kSliceThreads, nb_path).blocks;
  int Jmax = 1;
  for (int m = 0; m < M; ++m) Jmax = std::max(Jmax, offsets[m + 1] - offsets[m]);
  const int Kpad_max = 3 * kStrikeChunk * ((Jmax + kStrikeChunk - 1) / kStrikeChunk);
  // device arena layout (8-byte units unless noted): [in: strikes Jalloc | specs B*M | types (bytes, padded)] [state 3n] [out B*3*Jalloc] [pm] [pp]
  const size_t spec_bytes = sizeof(Spec) * (size_t)M * B;
  const size_t in_bytes = sizeof(double) * Jalloc + spec_bytes + (((size_t)Jalloc + 7) & ~(size_t)7);
  const size_t out_doubles = (size_t)3 * Jalloc * B;
  const size_t total = in_bytes + sizeof(double) * (3 * (size_t)nb_path + out_doubles + 2 * (size_t)blocks + (size_t)Kpad_max * blocks);
  std::vector<char> h_in(in_bytes, 0);
  if (Jtot > 0) {
    memcpy(h_in.data(), strikes + offsets[0], sizeof(double) * Jtot);
    memcpy(h_in.data() + sizeof(double) * Jalloc + spec_bytes, types + offsets[0], Jtot);
  }
  Spec* h_specs = (Spec*)(h_in.data() + sizeof(double) * Jalloc);
  for (int b = 0; b < B; ++b) {
    double t0 = 0.0;
    for (int m = 0; m < M; ++m) {
      int S;
      double dt;
      time_grid(ttms[m] - t0, nb_steps_per_year, &S, &dt);
      t0 = ttms[m];
      const int J = offsets[m + 1] - offsets[m];
      Spec& sp = h_specs[(size_t)b * M + m];
      if constexpr (MODEL == 0)
        sp.c = make_logsv_consts(lp[b], etas ? etas[(size_t)b * M + m] : 1.0, is_spot != 0, dt);
      else
        sp.c = make_heston_consts(hp[b], dt, scheme);
      sp.nsteps = S;
      sp.jo = offsets[m] - offsets[0];
      sp.J = J;
      sp.kinds = J ? payoff_kinds(types + offsets[m], J) : 0;
      sp.forward = forwards[m];
      sp.ttm = ttms[m];
      sp.discfactor = discfactors[m];
    }
  }
  std::vector<double> h_out(out_doubles);
  const int rc = host_call([&](cudaStream_t st) {
    DevBuf<char> arena(st);
    B200SV_CUDA(arena.alloc(total));
    B200SV_CUDA(cudaMemcpyAsync(arena.p, h_in.data(), in_bytes, cudaMemcpyHostToDevice, st));      // pageable source: staged before the call returns
    double* d_strikes = (double*)arena.p;
    const Spec* d_specs = (const Spec*)(arena.p + sizeof(double) * Jalloc);
    const int8_t* d_types = (const int8_t*)(arena.p + sizeof(double) * Jalloc + spec_bytes);
    double* d_state = (double*)(arena.p + in_bytes);
    double* d_out = d_state + 3 * (size_t)nb_path;
    double* d_pm = d_out + out_doubles;
    double* d_pp = d_pm + 2 * (size_t)blocks;
    for (int b = 0; b < B; ++b) {
      double* out_b = d_out + (size_t)3 * Jalloc * b;
      CoopArgs a{};
      a.x = d_state;
      a.v = d_state + nb_path;
      a.q = d_state + 2 * nb_path;
      a.n = nb_path;
      a.v_init = MODEL == 0 ? lp[b].sigma0 : hp[b].v0;
      a.seed = seed;
      a.M = M;
      a.variable_type = variable_type;
      a.strikes = d_strikes;
      a.types = d_types;
      a.part_mom = d_pm;
      a.part_pay = d_pp;
      a.Kpad_max = Kpad_max;
      a.total_paths = (double)nb_path;
      a.prices = out_b;
      a.stderrs = out_b + Jalloc;
      a.ivols = ivols_out ? out_b + 2 * Jalloc : nullptr;
      const Spec* sp = d_specs + (size_t)b * M;
      void* kargs[] = {(void*)&a, (void*)&sp};
      if (int rc = launched("mc_chain_coop_kernel", cudaLaunchCooperativeKernel(kernel, dim3(blocks), dim3(kSliceThreads), kargs, 0, st))) return rc;
    }
    if (Jtot > 0) B200SV_CUDA(cudaMemcpyAsync(h_out.data(), d_out, sizeof(double) * out_doubles, cudaMemcpyDeviceToHost, st));
    return 0;
  });
  for (int b = 0; b < B && rc == 0 && Jtot > 0; ++b) {
    const double* o = h_out.data() + (size_t)3 * Jalloc * b;
    memcpy(prices_out + (size_t)b * Jtot, o, sizeof(double) * Jtot);
    memcpy(stderr_out + (size_t)b * Jtot, o + Jalloc, sizeof(double) * Jtot);
    if (ivols_out) memcpy(ivols_out + (size_t)b * Jtot, o + 2 * Jalloc, sizeof(double) * Jtot);
  }
  return rc;
}

// shared host-level chain driver
template <int MODEL>
static int mc_chain_host(const b200sv_logsv_params* lp, const b200sv_heston_params* hp, int M, const double* ttms,
                         const double* forwards, const double* discfactors, const double* etas, const int* offsets,
                         const double* strikes, const int8_t* types, long long nb_path, int nb_steps_per_year, int is_spot,
                         int variable_type, uint64_t seed, int flags, double* prices_out, double* stderr_out, int scheme = 0, int B = 1,
                         double* ivols_out = nullptr) {
  // B > 1: lp / hp point to B parameter sets, etas to [B][M], outputs to [B][Jtot]; the sets run back to back on one stream with the SAME
  // seed (common random numbers => a smooth objective in the parameters), no host synchronisation until the single copy back
  B200SV_REQUIRE(B >= 1, "B must be >= 1");
  B200SV_REQUIRE(nb_path >= 1, "nb_path must be >= 1");
  B200SV_REQUIRE(nb_steps_per_year >= 1, "nb_steps_per_year must be >= 1");
  if (int rc = validate_chain(M, ttms, offsets, types, variable_type)) return rc;
  if (use_coop_chain(flags, nb_path, MODEL == 1))
    return mc_chain_host_coop<MODEL>(lp, hp, M, ttms, forwards, discfactors, etas, offsets, strikes, types, nb_path, nb_steps_per_year, is_spot,
                                     variable_type, seed, flags, prices_out, stderr_out, scheme, B, ivols_out);
  if (int rc = check_slice_flags(flags)) return rc;
  const bool f32 = flags & B200SV_STATE_F32;
  const size_t esz = f32 ? 4 : 8;
  return host_call([&](cudaStream_t st) {
    DevBuf<char> x(st);
    ChainPayoffs pay(st, M, ttms, forwards, discfactors, offsets, types, variable_type, B, ivols_out != nullptr);
    B200SV_CUDA(x.alloc(3 * esz * (size_t)nb_path));
    if (int rc = pay.alloc(strikes)) return rc;
    char *v = x.p + esz * (size_t)nb_path, *q = x.p + 2 * esz * (size_t)nb_path;
    for (int b = 0; b < B; ++b) {
      double t0 = 0.0;
      for (int m = 0; m < M; ++m) {
        int S;
        double dt;
        time_grid(ttms[m] - t0, nb_steps_per_year, &S, &dt);
        t0 = ttms[m];
        int rc;
        if constexpr (MODEL == 0)
          rc = launch_slice<0>(x.p, v, q, nb_path, 0, m == 0, lp[b].sigma0, S, m, forwards[m], seed, flags,
                               make_logsv_consts(lp[b], etas ? etas[(size_t)b * M + m] : 1.0, is_spot != 0, dt), pay.d_mom.p, st);
        else
          rc = launch_slice<1>(x.p, v, q, nb_path, 0, m == 0, hp[b].v0, S, m, forwards[m], seed, flags, make_heston_consts(hp[b], dt, scheme),
                               pay.d_mom.p, st);
        if (rc == 0) rc = pay.run(b, m, x.p, q, nb_path, f32, (double)nb_path, st);
        if (rc) return rc;
      }
    }
    return pay.copy_back(prices_out, stderr_out, ivols_out, st);
  });
}

template <int MODEL>
static int terminal_host(const b200sv_logsv_params* lp, const b200sv_heston_params* hp, double ttm, long long nb_path,
                         int nb_steps_per_year, int is_spot, double eta, uint64_t seed, int flags, double* x, double* v, double* q, int scheme = 0) {
  B200SV_REQUIRE(nb_path >= 1 && ttm > 0.0 && nb_steps_per_year >= 1, "nb_path, ttm, nb_steps_per_year must be positive");
  B200SV_REQUIRE(!(flags & B200SV_STATE_F32), "terminal values are returned as float64: use B200SV_STATE_F64");
  if (int rc = check_slice_flags(flags)) return rc;
  int S;
  double dt;
  time_grid(ttm, nb_steps_per_year, &S, &dt);
  return host_call([&](cudaStream_t st) {
    DevBuf<double> d(st), d_mom(st);
    B200SV_CUDA(d.alloc(3 * (size_t)nb_path));
    B200SV_CUDA(d_mom.alloc(2));
    int rc;
    if constexpr (MODEL == 0)
      rc = launch_slice<0>(d.p, d.p + nb_path, d.p + 2 * nb_path, nb_path, 0, 1, lp->sigma0, S, 0, 1.0, seed, flags,
                           make_logsv_consts(*lp, eta, is_spot != 0, dt), d_mom.p, st);
    else
      rc = launch_slice<1>(d.p, d.p + nb_path, d.p + 2 * nb_path, nb_path, 0, 1, hp->v0, S, 0, 1.0, seed, flags, make_heston_consts(*hp, dt, scheme),
                           d_mom.p, st);
    return rc ? rc : state_to_host(d.p, nb_path, x, v, q, st);
  });
}

}  // namespace b200sv

#include "rough_kernels.cuh"
#include "hawkes_kernels.cuh"

using namespace b200sv;

extern "C" {

const char* b200sv_last_error(void) { return last_error().c_str(); }
int b200sv_version(void) { return B200SV_VERSION; }
// stream of the calling thread's host-level calls (like cublasSetStream; NULL = the legacy default stream)
int b200sv_set_stream(void* stream) {
  current_stream_ref() = (cudaStream_t)stream;
  return 0;
}
void* b200sv_get_stream(void) { return (void*)current_stream(); }
long long b200sv_launch_count(void) { return launch_count(); }
void b200sv_reset_launch_count(void) { launch_count() = 0; }

int b200sv_logsv_mc_chain(const b200sv_logsv_params* params, int M, const double* ttms, const double* forwards,
                          const double* discfactors, const double* etas, const int* offsets, const double* strikes,
                          const int8_t* types, long long nb_path, int nb_steps_per_year, int is_spot_measure, int variable_type,
                          uint64_t seed, int flags, double* prices_out, double* stderr_out) {
  B200SV_REQUIRE(params && ttms && forwards && discfactors && offsets && prices_out && stderr_out, "null pointer");
  return mc_chain_host<0>(params, nullptr, M, ttms, forwards, discfactors, etas, offsets, strikes, types, nb_path,
                          nb_steps_per_year, is_spot_measure, variable_type, seed, flags, prices_out, stderr_out);
}

int b200sv_heston_mc_chain(const b200sv_heston_params* params, int M, const double* ttms, const double* forwards,
                           const double* discfactors, const int* offsets, const double* strikes, const int8_t* types,
                           long long nb_path, int nb_steps_per_year, int variable_type, uint64_t seed, int flags, int scheme,
                           double* prices_out, double* stderr_out) {
  B200SV_REQUIRE(params && ttms && forwards && discfactors && offsets && prices_out && stderr_out, "null pointer");
  B200SV_REQUIRE(scheme == B200SV_HESTON_EULER_FLOOR || scheme == B200SV_HESTON_QE, "unknown Heston scheme");
  return mc_chain_host<1>(nullptr, params, M, ttms, forwards, discfactors, nullptr, offsets, strikes, types, nb_path,
                          nb_steps_per_year, 1, variable_type, seed, flags, prices_out, stderr_out, scheme);
}

int b200sv_logsv_mc_chain_batch(const b200sv_logsv_params* params, int B, int M, const double* ttms, const double* forwards,
                                const double* discfactors, const double* etas, const int* offsets, const double* strikes,
                                const int8_t* types, long long nb_path, int nb_steps_per_year, int is_spot_measure, uint64_t seed,
                                int flags, double* prices_out, double* stderr_out, double* ivols_out) {
  B200SV_REQUIRE(params && ttms && forwards && discfactors && offsets && prices_out && stderr_out, "null pointer");
  return mc_chain_host<0>(params, nullptr, M, ttms, forwards, discfactors, etas, offsets, strikes, types, nb_path, nb_steps_per_year,
                          is_spot_measure, B200SV_LOG_RETURN, seed, flags, prices_out, stderr_out, 0, B, ivols_out);
}

int b200sv_heston_mc_chain_batch(const b200sv_heston_params* params, int B, int M, const double* ttms, const double* forwards,
                                 const double* discfactors, const int* offsets, const double* strikes, const int8_t* types,
                                 long long nb_path, int nb_steps_per_year, uint64_t seed, int flags, int scheme, double* prices_out,
                                 double* stderr_out, double* ivols_out) {
  B200SV_REQUIRE(params && ttms && forwards && discfactors && offsets && prices_out && stderr_out, "null pointer");
  B200SV_REQUIRE(scheme == B200SV_HESTON_EULER_FLOOR || scheme == B200SV_HESTON_QE, "unknown Heston scheme");
  return mc_chain_host<1>(nullptr, params, M, ttms, forwards, discfactors, nullptr, offsets, strikes, types, nb_path, nb_steps_per_year, 1,
                          B200SV_LOG_RETURN, seed, flags, prices_out, stderr_out, scheme, B, ivols_out);
}

int b200sv_logsv_terminal(const b200sv_logsv_params* params, double ttm, long long nb_path, int nb_steps_per_year,
                          int is_spot_measure, double eta, uint64_t seed, int flags, double* x, double* sigma, double* qvar) {
  B200SV_REQUIRE(params && x && sigma && qvar, "null pointer");
  return terminal_host<0>(params, nullptr, ttm, nb_path, nb_steps_per_year, is_spot_measure, eta, seed, flags, x, sigma, qvar);
}

// simulate_logsv_x_vol_terminal with PER-PATH initial arrays and in-kernel draws (pricers/logsv_pricer.py:1007-1020 accepts length-N x0 / sigma0 /
// qvar0): the three arrays are uploaded, advanced by the fused kernel (init = 0) and copied back in place.  slice_index selects the Philox
// sub-stream (counter word 3), so that successive calls on the same seed continue with fresh normals like the chain pricer's slices.
int b200sv_logsv_terminal_from_state(const b200sv_logsv_params* params, double ttm, long long nb_path, int nb_steps_per_year, int is_spot_measure,
                                     double eta, uint64_t seed, int flags, int slice_index, double* x_inout, double* sigma_inout,
                                     double* qvar_inout) {
  B200SV_REQUIRE(params && x_inout && sigma_inout && qvar_inout, "null pointer");
  B200SV_REQUIRE(nb_path >= 1 && ttm > 0.0 && nb_steps_per_year >= 1 && slice_index >= 0, "nb_path, ttm, nb_steps_per_year must be positive");
  B200SV_REQUIRE(!(flags & B200SV_STATE_F32), "terminal values are returned as float64: use B200SV_STATE_F64");
  if (int rc = check_slice_flags(flags)) return rc;
  int S;
  double dt;
  time_grid(ttm, nb_steps_per_year, &S, &dt);
  const LogsvConsts c = make_logsv_consts(*params, eta, is_spot_measure != 0, dt);
  return host_call([&](cudaStream_t st) {
    DevBuf<double> d(st), d_mom(st);
    B200SV_CUDA(d.alloc(3 * (size_t)nb_path));
    B200SV_CUDA(d_mom.alloc(2));
    if (int rc = state_to_device(d.p, nb_path, x_inout, sigma_inout, qvar_inout, st)) return rc;
    if (int rc = launch_slice<0>(d.p, d.p + nb_path, d.p + 2 * nb_path, nb_path, 0, 0, params->sigma0, S, slice_index, 1.0, seed, flags, c, d_mom.p, st))
      return rc;
    return state_to_host(d.p, nb_path, x_inout, sigma_inout, qvar_inout, st);
  });
}

int b200sv_heston_terminal(const b200sv_heston_params* params, double ttm, long long nb_path, int nb_steps_per_year,
                           uint64_t seed, int flags, int scheme, double* x, double* var, double* qvar) {
  B200SV_REQUIRE(params && x && var && qvar, "null pointer");
  B200SV_REQUIRE(scheme == B200SV_HESTON_EULER_FLOOR || scheme == B200SV_HESTON_QE, "unknown Heston scheme");
  return terminal_host<1>(nullptr, params, ttm, nb_path, nb_steps_per_year, 1, 1.0, seed, flags, x, var, qvar, scheme);
}

// ---- device-level ---------------------------------------------------------------------------------------------------
int b200sv_dev_logsv_slice(void* x, void* sigma, void* qvar, long long n_local, long long path_offset, int init,
                           const b200sv_logsv_params* params, double eta, int is_spot_measure, int nsteps, double dt,
                           int slice_index, double forward, uint64_t seed, int flags, double* moments_out, void* p2p, void* stream) {
  B200SV_REQUIRE(x && sigma && qvar && params && moments_out, "null pointer");
  B200SV_REQUIRE(n_local >= 1 && nsteps >= 1 && dt > 0.0, "n_local, nsteps, dt must be positive");
  const LogsvConsts c = make_logsv_consts(*params, eta, is_spot_measure != 0, dt);
  return launch_slice<0>(x, sigma, qvar, n_local, path_offset, init, params->sigma0, nsteps, slice_index, forward, seed, flags, c,
                         moments_out, (cudaStream_t)stream, (P2pCtx*)p2p);
}

int b200sv_dev_heston_slice(void* x, void* var, void* qvar, long long n_local, long long path_offset, int init,
                            const b200sv_heston_params* params, int nsteps, double dt, int slice_index, double forward,
                            uint64_t seed, int flags, int scheme, double* moments_out, void* p2p, void* stream) {
  B200SV_REQUIRE(x && var && qvar && params && moments_out, "null pointer");
  B200SV_REQUIRE(n_local >= 1 && nsteps >= 1 && dt > 0.0, "n_local, nsteps, dt must be positive");
  B200SV_REQUIRE(scheme == B200SV_HESTON_EULER_FLOOR || scheme == B200SV_HESTON_QE, "unknown Heston scheme");
  const HestonConsts c = make_heston_consts(*params, dt, scheme);
  return launch_slice<1>(x, var, qvar, n_local, path_offset, init, params->v0, nsteps, slice_index, forward, seed, flags, c,
                         moments_out, (cudaStream_t)stream, (P2pCtx*)p2p);
}

int b200sv_dev_payoff_sums(const void* x, const void* qvar, long long n_local, int flags, double ttm, double forward,
                           const double* strikes, const int8_t* types, int J, int variable_type, int payoff_kinds_hint,
                           const double* moments, double* sums_out, void* p2p, void* stream) {
  B200SV_REQUIRE(x && strikes && types && moments && sums_out, "null pointer");
  B200SV_REQUIRE(J >= 1 && n_local >= 1, "J and n_local must be >= 1");
  if (variable_type != B200SV_LOG_RETURN && variable_type != B200SV_Q_VAR) return fail(-4, "variable_type not implemented");
  B200SV_REQUIRE(variable_type == B200SV_LOG_RETURN || qvar, "qvar required for Q_VAR");
  if (flags & B200SV_STATE_F32)
    return launch_payoff_t<float>(x, qvar ? qvar : x, n_local, ttm, forward, strikes, types, J, variable_type, payoff_kinds_hint, moments, sums_out, (cudaStream_t)stream, (P2pCtx*)p2p);
  return launch_payoff_t<double>(x, qvar ? qvar : x, n_local, ttm, forward, strikes, types, J, variable_type, payoff_kinds_hint, moments, sums_out, (cudaStream_t)stream, (P2pCtx*)p2p);
}

int b200sv_dev_payoff_finalize(const double* sums, int J, double discfactor, long long total_paths, double* prices_out,
                               double* stderr_out, void* p2p, void* stream) {
  B200SV_REQUIRE(sums && prices_out && stderr_out && J >= 1, "null pointer / J");
  // exchange #2 (consumer): with a P2P context the global sums are gathered from the mailbox, `sums` holds this rank's local ones
  payoff_finalize_kernel<<<(J + 127) / 128, 128, 0, (cudaStream_t)stream>>>(sums, J, discfactor, (double)total_paths, prices_out, stderr_out,
                                                                            make_gather((P2pCtx*)p2p));
  return launched("payoff_finalize_kernel");
}

int b200sv_dev_logsv_step_fixed(double* x, double* sigma, double* qvar, const double* W0, const double* W1, int S, long long N,
                                double dt, const b200sv_logsv_params* params, double eta, int is_spot_measure, int fast, void* stream) {
  B200SV_REQUIRE(x && sigma && qvar && W0 && W1 && params, "null pointer");
  B200SV_REQUIRE(S >= 0 && N >= 1 && dt > 0.0, "S, N, dt");
  if (fast) {
    const LogsvConsts c = make_logsv_consts(*params, eta, is_spot_measure != 0, dt);
    Grid g = persistent_grid(logsv_step_fixed_fast_kernel, kThreads, N);
    logsv_step_fixed_fast_kernel<<<g.blocks, g.threads, 0, (cudaStream_t)stream>>>(x, sigma, qvar, W0, W1, S, N, c);
    return launched("logsv_step_fixed_fast_kernel");
  }
  LogsvRaw r{params->theta, params->kappa1, params->kappa2, params->beta, params->volvol, eta,
             is_spot_measure ? -1.0 : 1.0, is_spot_measure ? 0.0 : params->beta * eta, dt};
  Grid g = persistent_grid(logsv_step_fixed_kernel, kThreads, N);
  logsv_step_fixed_kernel<<<g.blocks, g.threads, 0, (cudaStream_t)stream>>>(x, sigma, qvar, W0, W1, S, N, r);
  return launched("logsv_step_fixed_kernel");
}

int b200sv_dev_heston_step_fixed(double* x, double* var, double* qvar, const double* W0, const double* W1, int S, long long N,
                                 double dt, const b200sv_heston_params* params, void* stream) {
  B200SV_REQUIRE(x && var && qvar && W0 && W1 && params, "null pointer");
  B200SV_REQUIRE(S >= 0 && N >= 1 && dt > 0.0, "S, N, dt");
  Grid g = persistent_grid(heston_step_fixed_kernel, kThreads, N);
  heston_step_fixed_kernel<<<g.blocks, g.threads, 0, (cudaStream_t)stream>>>(x, var, qvar, W0, W1, S, N, *params, dt);
  return launched("heston_step_fixed_kernel");
}

static int spot_moments_impl(const double* x, long long n, double forward, double* moments_out, cudaStream_t st, P2pCtx* p2p) {
  Grid g = persistent_grid(spot_moments_kernel, kThreads, n);
  DevBuf<double> partials(st);
  ensure_pool_threshold();
  B200SV_CUDA(partials.alloc(2 * (size_t)g.blocks));
  spot_moments_kernel<<<g.blocks, g.threads, 0, st>>>(x, n, forward, partials.p);
  if (int rc = launched("spot_moments_kernel")) return rc;
  reduce_partials_kernel<<<1, 64, 0, st>>>(partials.p, g.blocks, 2, 2, moments_out, make_publish(p2p, st));
  return launched("reduce_partials_kernel");
}

int b200sv_dev_spot_moments(const double* x, long long n, double forward, double* moments_out, void* stream) {
  B200SV_REQUIRE(x && moments_out && n >= 1, "null pointer / n");
  return spot_moments_impl(x, n, forward, moments_out, (cudaStream_t)stream, nullptr);
}

// sharded rough-LogSV / Hawkes slices (multi_gpu.py): the steppers of rough_kernels.cuh / hawkes_kernels.cuh on a contiguous range of GLOBAL
// path ids, followed by this rank's re-centring moments (published to the peer-memory mailbox when `p2p` is given) -- the same two
// exchanges per maturity as the LogSV chain
int b200sv_dev_hawkesjd_slice(double* x, double* lambda_p, double* lambda_m, long long n_local, long long path_offset, int init,
                              const b200sv_hawkes_params* params, int nsteps, double dt, int slice_index, double forward, uint64_t seed,
                              int flags, double* moments_out, void* p2p, void* stream) {
  B200SV_REQUIRE(x && lambda_p && lambda_m && params && moments_out, "null pointer");
  B200SV_REQUIRE(n_local >= 1 && nsteps >= 1 && dt > 0.0 && slice_index >= 0, "n_local, nsteps, dt must be positive");
  B200SV_REQUIRE(!(flags & B200SV_STATE_F32), "the Hawkes route is float64 only");
  return launch_hawkes_slice(x, lambda_p, lambda_m, n_local, path_offset, init, *params, nsteps, dt, slice_index, forward, seed, flags,
                             moments_out, (cudaStream_t)stream, (P2pCtx*)p2p);
}

int b200sv_dev_rough_logsv_slice(double* log_spot, double* vol_factors, double* qvar, long long n_local, long long path_offset,
                                 const b200sv_logsv_params* params, int n_factors, const double* weights, const double* nodes, int nsteps,
                                 double h, double forward, uint64_t seed, int flags, double* moments_out, void* p2p, void* stream) {
  B200SV_REQUIRE(log_spot && qvar && params && weights && nodes && moments_out, "null pointer");
  B200SV_REQUIRE(n_local >= 1 && nsteps >= 1 && h > 0.0, "n_local, nsteps, h must be positive");
  B200SV_REQUIRE(n_factors >= 1 && n_factors <= kMaxRoughFactors, "1 <= n_factors <= 8");
  B200SV_REQUIRE(!(flags & B200SV_STATE_F32), "the rough-vol route is float64 only");
  const int g = gauss_mode(flags);
  B200SV_REQUIRE(g == kGaussF32 || g == kGaussF64, "gauss flags");
  const RoughConsts c = make_rough_consts(*params, n_factors, weights, nodes, h);
  if (int rc = launch_rough(n_factors, log_spot, vol_factors, qvar, nullptr, nullptr, nsteps, n_local, c, seed, path_offset, g, (cudaStream_t)stream))
    return rc;
  return spot_moments_impl(log_spot, n_local, forward, moments_out, (cudaStream_t)stream, (P2pCtx*)p2p);
}

// ---- host-level fixed-random steppers and payoffs ------------------------------------------------------------------------
static int step_fixed_host(int model, double* x, double* v, double* q, const double* W0, const double* W1, int S, long long N,
                           double dt, const b200sv_logsv_params* lp, double eta, int is_spot, const b200sv_heston_params* hp) {
  B200SV_REQUIRE(x && v && q && (S == 0 || (W0 && W1)), "null pointer");
  B200SV_REQUIRE(S >= 0 && N >= 1 && dt > 0.0, "S, N, dt");
  const size_t wn = (size_t)N * S;
  return host_call([&](cudaStream_t st) {
    DevBuf<double> d(st), w(st);
    B200SV_CUDA(d.alloc(3 * (size_t)N));
    B200SV_CUDA(w.alloc(2 * std::max<size_t>(wn, N)));
    if (int rc = state_to_device(d.p, N, x, v, q, st)) return rc;
    if (S > 0) {
      B200SV_CUDA(cudaMemcpyAsync(w.p, W0, sizeof(double) * wn, cudaMemcpyHostToDevice, st));
      B200SV_CUDA(cudaMemcpyAsync(w.p + wn, W1, sizeof(double) * wn, cudaMemcpyHostToDevice, st));
    }
    const int rc = model == 0 ? b200sv_dev_logsv_step_fixed(d.p, d.p + N, d.p + 2 * N, w.p, w.p + wn, S, N, dt, lp, eta, is_spot, 0, st)
                              : b200sv_dev_heston_step_fixed(d.p, d.p + N, d.p + 2 * N, w.p, w.p + wn, S, N, dt, hp, st);
    return rc ? rc : state_to_host(d.p, N, x, v, q, st);
  });
}

int b200sv_logsv_step_fixed(double* x, double* sigma, double* qvar, const double* W0, const double* W1, int S, long long N,
                            double dt, const b200sv_logsv_params* params, double eta, int is_spot_measure) {
  B200SV_REQUIRE(params, "null pointer");
  return step_fixed_host(0, x, sigma, qvar, W0, W1, S, N, dt, params, eta, is_spot_measure, nullptr);
}

int b200sv_heston_step_fixed(double* x, double* var, double* qvar, const double* W0, const double* W1, int S, long long N,
                             double dt, const b200sv_heston_params* params) {
  B200SV_REQUIRE(params, "null pointer");
  return step_fixed_host(1, x, var, qvar, W0, W1, S, N, dt, nullptr, 1.0, 1, params);
}

int b200sv_mc_payoffs(const double* x, const double* qvar, long long N, double ttm, double forward, const double* strikes,
                      const int8_t* types, int J, double discfactor, int variable_type, double* prices_out, double* stderr_out) {
  B200SV_REQUIRE(x && strikes && types && prices_out && stderr_out, "null pointer");
  B200SV_REQUIRE(N >= 1 && J >= 1, "N and J must be >= 1");
  for (int j = 0; j < J; ++j)
    if (types[j] < 0 || types[j] > 3) return fail(-3, "unknown option payoff code");
  if (variable_type != B200SV_LOG_RETURN && variable_type != B200SV_Q_VAR) return fail(-4, "variable_type not implemented");
  B200SV_REQUIRE(variable_type == B200SV_LOG_RETURN || qvar, "qvar required for Q_VAR");
  const int offsets[2] = {0, J};
  return host_call([&](cudaStream_t st) {
    DevBuf<double> d(st);
    ChainPayoffs pay(st, 1, &ttm, &forward, &discfactor, offsets, types, variable_type, 1, false);
    B200SV_CUDA(d.alloc(2 * (size_t)N));
    if (int rc = pay.alloc(strikes)) return rc;
    B200SV_CUDA(cudaMemcpyAsync(d.p, x, sizeof(double) * N, cudaMemcpyHostToDevice, st));
    if (qvar) B200SV_CUDA(cudaMemcpyAsync(d.p + N, qvar, sizeof(double) * N, cudaMemcpyHostToDevice, st));
    if (int rc = spot_moments_impl(d.p, N, forward, pay.d_mom.p, st, nullptr)) return rc;
    if (int rc = pay.run(0, 0, d.p, d.p + N, N, false, (double)N, st)) return rc;
    return pay.copy_back(prices_out, stderr_out, nullptr, st);
  });
}

int b200sv_device_normals(uint64_t seed, long long path0, long long n, int slice, int nsteps, int flags, double* z0, double* z1) {
  B200SV_REQUIRE(z0 && z1 && n >= 1 && nsteps >= 1, "null pointer / sizes");
  const int g = gauss_mode(flags);
  B200SV_REQUIRE(g >= 0, "B200SV_GAUSS_F64 and B200SV_GAUSS_F64_PAIRED are mutually exclusive");
  const size_t nz = (size_t)n * nsteps;
  return host_call([&](cudaStream_t st) {
    DevBuf<double> d(st);
    B200SV_CUDA(d.alloc(2 * nz));
    const int blocks = (int)((n + 127) / 128);
    if (g == kGaussF64)
      device_normals_kernel<kGaussF64><<<blocks, 128, 0, st>>>(seed, (unsigned long long)path0, n, (unsigned)slice, nsteps, d.p, d.p + nz);
    else if (g == kGaussF64Paired)
      device_normals_kernel<kGaussF64Paired><<<blocks, 128, 0, st>>>(seed, (unsigned long long)path0, n, (unsigned)slice, nsteps, d.p, d.p + nz);
    else
      device_normals_kernel<kGaussF32><<<blocks, 128, 0, st>>>(seed, (unsigned long long)path0, n, (unsigned)slice, nsteps, d.p, d.p + nz);
    if (int rc = launched("device_normals_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(z0, d.p, sizeof(double) * nz, cudaMemcpyDeviceToHost, st));
    B200SV_CUDA(cudaMemcpyAsync(z1, d.p + nz, sizeof(double) * nz, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

int b200sv_debug_exp_pair_scaled(const double* Ls, long long n, double* out /* 2n */) {
  B200SV_REQUIRE(Ls && out && n >= 1, "null pointer / n");
  return host_call([&](cudaStream_t st) {
    DevBuf<double> dl(st), dout(st);
    B200SV_CUDA(dl.upload(Ls, n));
    B200SV_CUDA(dout.alloc(2 * (size_t)n));
    exp_pair_scaled_kernel<<<(int)((n + 127) / 128), 128, 0, st>>>(dl.p, n, dout.p);
    if (int rc = launched("exp_pair_scaled_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(out, dout.p, sizeof(double) * 2 * n, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

int b200sv_debug_exp_pair(const double* L, long long n, double* out /* 2n */) {
  B200SV_REQUIRE(L && out && n >= 1, "null pointer / n");
  return host_call([&](cudaStream_t st) {
    DevBuf<double> dl(st), dout(st);
    B200SV_CUDA(dl.upload(L, n));
    B200SV_CUDA(dout.alloc(2 * (size_t)n));
    exp_pair_kernel<<<(int)((n + 127) / 128), 128, 0, st>>>(dl.p, n, dout.p);
    if (int rc = launched("exp_pair_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(out, dout.p, sizeof(double) * 2 * n, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

int b200sv_logsv_vol_paths(const b200sv_logsv_params* params, double ttm, long long nb_path, int nb_steps_per_year, int is_spot_measure,
                           uint64_t seed, const double* brownians, double* sigma_t_out) {
  B200SV_REQUIRE(params && sigma_t_out, "null pointer");
  B200SV_REQUIRE(nb_path >= 1 && ttm > 0.0 && nb_steps_per_year >= 1, "nb_path, ttm, nb_steps_per_year must be positive");
  int S;
  double dt;
  time_grid(ttm, nb_steps_per_year, &S, &dt);
  // adj = beta under the inverse measure, no eta (pricers/logsv_pricer.py:929-932)
  LogsvRaw r{params->theta, params->kappa1, params->kappa2, params->beta, params->volvol, 1.0, is_spot_measure ? -1.0 : 1.0,
             is_spot_measure ? 0.0 : params->beta, dt};
  const size_t ob = (size_t)(S + 1) * (size_t)nb_path;
  return host_call([&](cudaStream_t st) {
    DevBuf<double> d_out(st), d_w(st);
    B200SV_CUDA(d_out.alloc(ob));
    if (brownians) B200SV_CUDA(d_w.upload(brownians, (size_t)S * (size_t)nb_path));
    Grid g = persistent_grid(logsv_vol_paths_kernel, kThreads, nb_path);
    logsv_vol_paths_kernel<<<g.blocks, g.threads, 0, st>>>(d_out.p, d_w.p, S, nb_path, r, params->sigma0, seed, 0ull);
    if (int rc = launched("logsv_vol_paths_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(sigma_t_out, d_out.p, sizeof(double) * ob, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

// ---- rough-LogSV multi-factor MC (rough_kernels.cuh) ------------------------------------------------------------------------
int b200sv_rough_logsv_mc_chain(const b200sv_logsv_params* params, int B, int n_factors, const double* weights, const double* nodes, int M,
                                const double* ttms, const double* forwards, const double* discfactors, const int* offsets, const double* strikes,
                                const int8_t* types, long long nb_path, const int* nsteps, const double* hs, const double* Z0, const double* Z1,
                                long long z_rows, int variable_type, uint64_t seed, int flags, double* prices_out, double* stderr_out,
                                double* ivols_out, double* states_out) {
  B200SV_REQUIRE(params && weights && nodes && ttms && forwards && discfactors && offsets && nsteps && hs && prices_out && stderr_out, "null pointer");
  return rough_chain_host(params, B, n_factors, weights, nodes, M, ttms, forwards, discfactors, offsets, strikes, types, nb_path, nsteps, hs, Z0, Z1,
                          z_rows, variable_type, seed, flags, prices_out, stderr_out, ivols_out, states_out);
}

// ---- Hawkes jump-diffusion MC (hawkes_kernels.cuh) ---------------------------------------------------------------------------
int b200sv_hawkesjd_mc_chain(const b200sv_hawkes_params* params, int M, const double* ttms, const double* forwards, const double* discfactors,
                             const int* offsets, const double* strikes, const int8_t* types, long long nb_path, int variable_type, uint64_t seed,
                             int flags, double* prices_out, double* stderr_out) {
  B200SV_REQUIRE(params && ttms && forwards && discfactors && offsets && prices_out && stderr_out, "null pointer");
  return hawkes_chain_host(params, M, ttms, forwards, discfactors, offsets, strikes, types, nb_path, variable_type, seed, flags, prices_out,
                           stderr_out);
}

int b200sv_hawkesjd_terminal(const b200sv_hawkes_params* params, double ttm, long long nb_path, uint64_t seed, int flags, int slice_index,
                             int use_initial_arrays, double* x_inout, double* lambda_p_inout, double* lambda_m_inout) {
  B200SV_REQUIRE(params && x_inout && lambda_p_inout && lambda_m_inout, "null pointer");
  B200SV_REQUIRE(nb_path >= 1 && ttm > 0.0 && slice_index >= 0, "nb_path, ttm must be positive");
  if (int rc = check_hawkes_flags(flags)) return rc;
  int S;
  double dt;
  time_grid(ttm, kHawkesStepsPerYear, &S, &dt);
  return host_call([&](cudaStream_t st) {
    DevBuf<double> d(st), d_mom(st);
    B200SV_CUDA(d.alloc(3 * (size_t)nb_path));
    B200SV_CUDA(d_mom.alloc(2));
    if (use_initial_arrays)
      if (int rc = state_to_device(d.p, nb_path, x_inout, lambda_p_inout, lambda_m_inout, st)) return rc;
    if (int rc = launch_hawkes_slice(d.p, d.p + nb_path, d.p + 2 * nb_path, nb_path, 0, use_initial_arrays ? 0 : 1, *params, S, dt, slice_index, 1.0,
                                     seed, flags, d_mom.p, st))
      return rc;
    return state_to_host(d.p, nb_path, x_inout, lambda_p_inout, lambda_m_inout, st);
  });
}

int b200sv_hawkesjd_step_fixed(double* x, double* lambda_p, double* lambda_m, const double* W0, const double* U_P, const double* U_M,
                               const double* J_P, const double* J_M, int S, long long N, double dt, const b200sv_hawkes_params* params) {
  B200SV_REQUIRE(x && lambda_p && lambda_m && params && (S == 0 || (W0 && U_P && U_M && J_P && J_M)), "null pointer");
  B200SV_REQUIRE(S >= 0 && N >= 1 && dt > 0.0, "S, N, dt");
  const size_t wn = (size_t)N * (size_t)std::max(S, 1);
  return host_call([&](cudaStream_t st) {
    DevBuf<double> d(st), w(st);
    B200SV_CUDA(d.alloc(3 * (size_t)N));
    B200SV_CUDA(w.alloc(5 * wn));
    if (int rc = state_to_device(d.p, N, x, lambda_p, lambda_m, st)) return rc;
    const double* src[5] = {W0, U_P, U_M, J_P, J_M};
    if (S > 0)
      for (int k = 0; k < 5; ++k) B200SV_CUDA(cudaMemcpyAsync(w.p + k * wn, src[k], sizeof(double) * wn, cudaMemcpyHostToDevice, st));
    Grid g = persistent_grid(hawkes_step_fixed_kernel, kThreads, N);
    hawkes_step_fixed_kernel<<<g.blocks, g.threads, 0, st>>>(d.p, d.p + N, d.p + 2 * N, w.p, w.p + wn, w.p + 2 * wn, w.p + 3 * wn, w.p + 4 * wn, S, N,
                                                              make_hawkes_consts(*params, dt));
    if (int rc = launched("hawkes_step_fixed_kernel")) return rc;
    return state_to_host(d.p, N, x, lambda_p, lambda_m, st);
  });
}

int b200sv_hawkesjd_device_draws(uint64_t seed, long long path0, long long n, int slice, int S, double dt, const b200sv_hawkes_params* params,
                                 int flags, double* W0, double* U_P, double* U_M, double* J_P, double* J_M) {
  B200SV_REQUIRE(params && W0 && U_P && U_M && J_P && J_M && n >= 1 && S >= 1 && dt > 0.0, "null pointer / sizes");
  const int g = gauss_mode(flags);
  B200SV_REQUIRE(g == kGaussF32 || g == kGaussF64, "gauss flags");
  const size_t wn = (size_t)n * S;
  const HawkesConsts c = make_hawkes_consts(*params, dt);
  return host_call([&](cudaStream_t st) {
    DevBuf<double> d(st);
    B200SV_CUDA(d.alloc(5 * wn));
    const int blocks = (int)((n + 127) / 128);
    if (g == kGaussF64)
      hawkes_device_draws_kernel<kGaussF64><<<blocks, 128, 0, st>>>(seed, (unsigned long long)path0, n, (unsigned)slice, S, c, d.p, d.p + wn, d.p + 2 * wn,
                                                                    d.p + 3 * wn, d.p + 4 * wn);
    else
      hawkes_device_draws_kernel<kGaussF32><<<blocks, 128, 0, st>>>(seed, (unsigned long long)path0, n, (unsigned)slice, S, c, d.p, d.p + wn, d.p + 2 * wn,
                                                                    d.p + 3 * wn, d.p + 4 * wn);
    if (int rc = launched("hawkes_device_draws_kernel")) return rc;
    double* dst[5] = {W0, U_P, U_M, J_P, J_M};
    for (int k = 0; k < 5; ++k) B200SV_CUDA(cudaMemcpyAsync(dst[k], d.p + k * wn, sizeof(double) * wn, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}

// ---- P2P mailbox (p2p.cuh) -----------------------------------------------------------------------------------------------
int b200sv_p2p_create(int world, int rank, int max_values, void** ctx_out, unsigned char* handle_out /* 64 bytes */) {
  B200SV_REQUIRE(ctx_out && handle_out, "null pointer");
  B200SV_REQUIRE(world >= 1 && world <= kMaxPeers && rank >= 0 && rank < world && max_values >= 2, "world <= 8, 0 <= rank < world, max_values >= 2");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  P2pCtx* c = new P2pCtx();
  c->world = world;
  c->rank = rank;
  c->kmax = max_values;
  c->vals_bytes = sizeof(double) * 2 * (size_t)world * max_values;
  c->published = c->consumed = 0;
  const size_t flags_bytes = sizeof(unsigned long long) * 2 * (size_t)world;
  const size_t total = c->vals_bytes + flags_bytes + 2 * sizeof(double);
  cudaError_t e = cudaMalloc((void**)&c->mail, total);
  if (e == cudaSuccess) e = cudaMemset(c->mail, 0, total);
  cudaIpcMemHandle_t h;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, c->mail);
  if (e != cudaSuccess) {
    delete c;
    return fail(-2, std::string("b200sv_p2p_create: ") + cudaGetErrorString(e));
  }
  for (int s = 0; s < kMaxPeers; ++s) c->peer[s] = nullptr;
  c->peer[rank] = c->mail;
  c->scratch = (double*)(c->mail + c->vals_bytes + flags_bytes);
  c->status = (unsigned int*)(c->scratch + 1);
  c->spin_limit = kSpinLimit;
  memcpy(handle_out, &h, 64);
  *ctx_out = c;
  return 0;
}

int b200sv_p2p_connect(void* ctx, const unsigned char* handles /* world x 64 bytes, rank order */) {
  B200SV_REQUIRE(ctx && handles, "null pointer");
  P2pCtx* c = (P2pCtx*)ctx;
  for (int s = 0; s < c->world; ++s) {
    if (s == c->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + 64 * (size_t)s, 64);
    void* p = nullptr;
    B200SV_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    c->peer[s] = (char*)p;
  }
  return 0;
}

int b200sv_p2p_destroy(void* ctx) {
  if (!ctx) return 0;
  P2pCtx* c = (P2pCtx*)ctx;
  cudaDeviceSynchronize();
  for (int s = 0; s < c->world; ++s)
    if (s != c->rank && c->peer[s]) cudaIpcCloseMemHandle(c->peer[s]);
  cudaFree(c->mail);
  delete c;
  return 0;
}

int b200sv_p2p_set_spin_limit(void* ctx, unsigned int spins) {
  B200SV_REQUIRE(ctx && spins >= 1, "null pointer / spins");
  ((P2pCtx*)ctx)->spin_limit = spins;
  return 0;
}

// timeout bits of the exchanges since the last call (bit r: peer r did not publish within the spin limit); synchronises `stream` first
int b200sv_p2p_status(void* ctx, unsigned int* status_out, void* stream) {
  B200SV_REQUIRE(ctx && status_out, "null pointer");
  P2pCtx* c = (P2pCtx*)ctx;
  cudaStream_t st = (cudaStream_t)stream;
  B200SV_CUDA(cudaMemcpyAsync(status_out, c->status, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
  B200SV_CUDA(cudaStreamSynchronize(st));
  if (*status_out) B200SV_CUDA(cudaMemsetAsync(c->status, 0, sizeof(unsigned int), st));
  return 0;
}

// test hook: account for a publish that never happens (a peer that died / never arrived) -- the next gather on this context waits for an epoch
// nobody signals and must run into the spin limit: poisoned values + status bit, never a hang
int b200sv_debug_p2p_lose_publish(void* ctx) {
  B200SV_REQUIRE(ctx, "null pointer");
  ++((P2pCtx*)ctx)->published;
  return 0;
}

int b200sv_dev_p2p_publish(void* ctx, const double* vals, int K, void* stream) {
  B200SV_REQUIRE(ctx && K >= 1, "null pointer / K");
  P2pCtx* c = (P2pCtx*)ctx;
  B200SV_REQUIRE(K <= c->kmax, "K exceeds the mailbox size");
  p2p_publish_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(vals, K, make_publish(c, (cudaStream_t)stream));
  return launched("p2p_publish_kernel");
}

int b200sv_dev_p2p_gather(void* ctx, int K, double* out, void* stream) {
  B200SV_REQUIRE(ctx && out && K >= 1, "null pointer / K");
  P2pCtx* c = (P2pCtx*)ctx;
  B200SV_REQUIRE(K <= c->kmax, "K exceeds the mailbox size");
  p2p_gather_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(make_gather(c), K, out);
  return launched("p2p_gather_kernel");
}

}  // extern "C"
