// hawkes_kernels.cuh -- Hawkes jump-diffusion Monte Carlo (two mutually exciting jump intensities) for sm_100a.
// Included by mc_kernels.cu (same translation unit: it reuses the payoff / reduction launchers and the Philox generator).
//
// Replaces, behind the C ABI of include/b200sv.h (/root/reference/src/stochvolmodels/pricers/hawkes_jd_pricer.py):
//   simulate_hawkesjd_terminal   :718-779   1800 steps per year (:752); per step and path: one scaled normal w0, two exponential clocks
//                                           u = -ln(U)/dt compared with the intensities (a jump fires when lambda > u, :767-768), two
//                                           shifted-exponential jump sizes; explicit Euler on (x, lambda_p, lambda_m) (:765-776)
//   hawkesjd_mc_chain_pricer     :644-715   slices chained on the terminal state, payoffs = utils/mc_payoffs.py on x
//
// Two kernels.  hawkes_step_fixed_kernel: caller-supplied (W0, U_P, U_M, J_P, J_M) [S][N] in the reference's own form, reference
// evaluation order without FMA contraction (the reference is plain numpy: IEEE operations one by one) -- the parity entry, 40 B of inputs
// per path-step from HBM.  hawkes_slice_kernel: the same update with every draw made in-kernel (no HBM traffic but the state):
//   normals      the stepper's stream (philox.cuh, counter word 3 = slice): one Philox call feeds 4 steps (float draws) or 2 (fp64 draws)
//   jump clocks  a second stream (slice | 0x80000000), one call per TWO steps; a third (slice | 0x40000000) holds the jump sizes and is only
//   and sizes    evaluated when a clock fires (~lambda dt = 0.5 % of the steps).  u = (r + 1/2) 2^-32.
// b200sv_hawkesjd_device_draws exports the in-kernel draws in the reference's form so that the fused kernel is checked path by path
// against the oracle on ITS OWN inputs.
#pragma once

namespace b200sv {

struct HawkesConsts {
  double dt, sqrt_dt, inv_dt;
  double drift_dt;            // (mu - sigma^2 / 2) dt                               (:763)
  double comp_p, comp_m;      // dt (exp(shift) / (1 - mean) - 1)                    (:760-761)
  double sigma;
  double shift_p, mean_p, shift_m, mean_m;
  double theta_p, kappa_p, beta1_p, beta2_p, theta_m, kappa_m, beta1_m, beta2_m;
};

static HawkesConsts make_hawkes_consts(const b200sv_hawkes_params& p, double dt) {
  HawkesConsts c;
  c.dt = dt;
  c.sqrt_dt = std::sqrt(dt);
  c.inv_dt = 1.0 / dt;
  c.drift_dt = (p.mu - 0.5 * p.sigma * p.sigma) * dt;
  c.comp_p = dt * (std::exp(p.shift_p) / (1.0 - p.mean_p) - 1.0);
  c.comp_m = dt * (std::exp(p.shift_m) / (1.0 - p.mean_m) - 1.0);
  c.sigma = p.sigma;
  c.shift_p = p.shift_p;
  c.mean_p = p.mean_p;
  c.shift_m = p.shift_m;
  c.mean_m = p.mean_m;
  c.theta_p = p.theta_p;
  c.kappa_p = p.kappa_p;
  c.beta1_p = p.beta1_p;
  c.beta2_p = p.beta2_p;
  c.theta_m = p.theta_m;
  c.kappa_m = p.kappa_m;
  c.beta1_m = p.beta1_m;
  c.beta2_m = p.beta2_m;
  return c;
}

// one Euler step in the reference's evaluation order (:765-776), IEEE operations without contraction
__device__ __forceinline__ void hawkes_update(double& x, double& lp, double& lm, double w0, double jump_p, double jump_m, const HawkesConsts& c) {
  const double diffusion = __dadd_rn(__dadd_rn(__dadd_rn(c.drift_dt, -__dmul_rn(c.comp_p, lp)), -__dmul_rn(c.comp_m, lm)), __dmul_rn(c.sigma, w0));
  x = __dadd_rn(__dadd_rn(__dadd_rn(x, diffusion), jump_p), jump_m);
  const double load_p = __dadd_rn(__dmul_rn(c.beta1_p, jump_p), __dmul_rn(c.beta2_p, jump_m));
  const double load_m = __dadd_rn(__dmul_rn(c.beta1_m, jump_p), __dmul_rn(c.beta2_m, jump_m));
  lp = __dadd_rn(__dadd_rn(lp, __dmul_rn(__dmul_rn(c.kappa_p, __dadd_rn(c.theta_p, -lp)), c.dt)), load_p);
  lm = __dadd_rn(__dadd_rn(lm, __dmul_rn(__dmul_rn(c.kappa_m, __dadd_rn(c.theta_m, -lm)), c.dt)), load_m);
}

__global__ void __launch_bounds__(kThreads) hawkes_step_fixed_kernel(double* __restrict__ x, double* __restrict__ lam_p, double* __restrict__ lam_m,
                                                                    const double* __restrict__ W0, const double* __restrict__ U_P,
                                                                    const double* __restrict__ U_M, const double* __restrict__ J_P,
                                                                    const double* __restrict__ J_M, int S, long long N, HawkesConsts c) {
  const long long stride = (long long)gridDim.x * kThreads;
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < N; i += stride) {
    double xi = x[i], lp = lam_p[i], lm = lam_m[i];
    for (int s = 0; s < S; ++s) {
      const size_t o = (size_t)s * N + i;
      const double jp = lp > __ldg(U_P + o) ? __ldg(J_P + o) : 0.0;       // np.where(lambda_p0 > u_p, j_p, 0.0)
      const double jm = lm > __ldg(U_M + o) ? __ldg(J_M + o) : 0.0;
      hawkes_update(xi, lp, lm, __ldg(W0 + o), jp, jm, c);
    }
    x[i] = xi;
    lam_p[i] = lp;
    lam_m[i] = lm;
  }
}

// Jump streams of one path (counter word 3 = slice | flag; the stepper's normals use the plain slice):
//   clocks  flag 0x80000000, call k = step / 2:  words (x, y) = the (+, -) clocks of step 2k, (z, w) = those of step 2k + 1
//   sizes   flag 0x40000000, call = step:        words (x, y) = the (+, -) jump sizes -- evaluated only when a clock fires
// uniform in (0, 1) of a 32-bit word: (r + 1/2) 2^-32
__device__ __forceinline__ uint4 hawkes_clock_words(uint2 key, uint32_t plo, uint32_t phi, uint32_t pair, uint32_t slice) {
  return philox4x32_10(make_uint4(plo, phi, pair, slice | 0x80000000u), key);
}
__device__ __forceinline__ uint4 hawkes_size_words(uint2 key, uint32_t plo, uint32_t phi, uint32_t step, uint32_t slice) {
  return philox4x32_10(make_uint4(plo, phi, step, slice | 0x40000000u), key);
}
__device__ __forceinline__ double hawkes_uniform(uint32_t r) { return fma((double)r, 2.3283064365386963e-10, 1.1641532182693481e-10); }
// exponential clock -ln(U)/dt and shifted-exponential sizes exactly as b200sv_hawkesjd_device_draws exports them
__device__ __forceinline__ double hawkes_clock(double u, const HawkesConsts& c) { return __ddiv_rn(-log(u), c.dt); }
__device__ __forceinline__ double hawkes_size_p(double u, const HawkesConsts& c) { return __dadd_rn(c.shift_p, __dmul_rn(c.mean_p, -log(u))); }
__device__ __forceinline__ double hawkes_size_m(double u, const HawkesConsts& c) { return __dadd_rn(c.shift_m, -__dmul_rn(-c.mean_m, -log(u))); }

struct HawkesSliceArgs {
  double *x, *lam_p, *lam_m;
  long long n;
  unsigned long long path_offset;
  int init;                    // 1: start every path from (0, lambda_p0, lambda_m0)
  double lam_p0, lam_m0;
  int nsteps;
  unsigned int slice;
  unsigned long long seed;
  double forward;
  double* partials;            // [gridDim.x][2]: (sum F e^x over non-NaN, count) for the forward re-centring
};

// Throughput stepper.  Per step the common case (no jump, ~99.5 % of the steps at the reference's parameters) is 8 contracted fp64
// operations; whether a clock CAN fire is decided on the raw 32-bit word: -ln(u) >= 1 - u, so a jump needs 1 - u < lambda dt, i.e.
// r >= floor(2^32 (1 - lambda dt (1 + 1e-9))) - 1 (one DFMA + F2I + integer compare; the margins cover the rounding of the product and of
// the floor).  Only then are the logarithm, the exact comparison lambda > -ln(u)/dt of the reference (:767-768) and -- if it fires -- the
// size stream evaluated.  Same draws as b200sv_hawkesjd_device_draws exports; agreement with the strict kernel ~1e-15 (FMA contraction).
struct HawkesFast {
  double ssd;                // sigma sqrt(dt)
  double kdt_p, kdt_m;       // kappa dt
  double thr;                // dt (1 + 1e-9) 2^32
  double dt_lo;              // dt (1 - 1e-9)
};

// Does the clock with word r fire against intensity lam, i.e. is lam > -ln(u)/dt as the reference evaluates it (:767-768)?  With e = 1 - u
// (exact in fp64): -ln(u) <= e + e^2 for e <= 1/2, so e + e^2 < lam dt (1 - 1e-9) settles it without a logarithm; the band in between
// (relative width ~e, i.e. ~0.5 % of the candidates) takes the exact comparison, out of line.
__device__ __noinline__ bool hawkes_fires_exact(double lam, double u, double dt) { return lam > __ddiv_rn(-log(u), dt); }
__device__ __forceinline__ bool hawkes_fires(double lam, uint32_t r, double dt, double dt_lo) {
  const double u = hawkes_uniform(r), e = 1.0 - u;
  if (e <= 0.5 && fma(e, e, e) < lam * dt_lo) return true;
  return hawkes_fires_exact(lam, u, dt);
}
// both clocks firing in one step (~1e-5 of the steps): out of line
__device__ __noinline__ double2 hawkes_two_sizes(uint32_t wx, uint32_t wy, double shift_p, double mean_p, double shift_m, double mean_m) {
  return make_double2(__dadd_rn(shift_p, __dmul_rn(mean_p, -log(hawkes_uniform(wx)))), __dadd_rn(shift_m, -__dmul_rn(-mean_m, -log(hawkes_uniform(wy)))));
}

#ifndef B200SV_HAWKES_MINBLOCKS
#define B200SV_HAWKES_MINBLOCKS 2
#endif
template <int GAUSS>
__global__ void __launch_bounds__(kThreads, B200SV_HAWKES_MINBLOCKS) hawkes_slice_kernel(HawkesSliceArgs a, HawkesConsts c) {
  __shared__ double red[2 * kThreads / 32];
  if constexpr (GAUSS != kGaussF32) gauss64_table_init();
  double acc[2] = {0.0, 0.0};
  const uint2 key = make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32));
  const HawkesFast f{c.sigma * c.sqrt_dt, c.kappa_p * c.dt, c.kappa_m * c.dt, c.dt * (1.0 + 1e-9) * 4294967296.0, c.dt * (1.0 - 1e-9)};
  const long long stride = (long long)gridDim.x * kThreads;
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < a.n; i += stride) {
    double xi = 0.0, lp = a.lam_p0, lm = a.lam_m0;
    if (!a.init) {
      xi = a.x[i];
      lp = a.lam_p[i];
      lm = a.lam_m[i];
    }
    const unsigned long long path = a.path_offset + (unsigned long long)i;
    const uint32_t plo = (uint32_t)path, phi = (uint32_t)(path >> 32);
    StepNormals<double, GAUSS> rng(a.seed, path, a.slice);
    auto one_step = [&](double z, uint32_t rp, uint32_t rm, uint32_t step) {
      const uint32_t tp = __double2uint_rd(fma(-lp, f.thr, 4294967296.0)), tm = __double2uint_rd(fma(-lm, f.thr, 4294967296.0));
      const bool cand_p = rp >= max(tp, 1u) - 1u, cand_m = rm >= max(tm, 1u) - 1u;
      double jp = 0.0, jm = 0.0;
      if (cand_p || cand_m) {                                                     // ~1 % of the lane-steps: a clock may fire
        const bool fp_ = cand_p && hawkes_fires(lp, rp, c.dt, f.dt_lo), fm_ = cand_m && hawkes_fires(lm, rm, c.dt, f.dt_lo);
        if (fp_ || fm_) {
          const uint4 w = hawkes_size_words(key, plo, phi, step, a.slice);
          if (fp_ && fm_) {
            const double2 jj = hawkes_two_sizes(w.x, w.y, c.shift_p, c.mean_p, c.shift_m, c.mean_m);
            jp = jj.x;
            jm = jj.y;
          } else {                                                                // one logarithm serves whichever clock fired
            const double l = -log(hawkes_uniform(fp_ ? w.x : w.y));
            if (fp_) jp = __dadd_rn(c.shift_p, __dmul_rn(c.mean_p, l));            // = hawkes_size_p
            else jm = __dadd_rn(c.shift_m, -__dmul_rn(-c.mean_m, l));              // = hawkes_size_m
          }
        }
      }
      double d = fma(-c.comp_p, lp, c.drift_dt);
      d = fma(-c.comp_m, lm, d);
      d = fma(f.ssd, z, d);
      xi += d;
      lp = fma(f.kdt_p, c.theta_p - lp, lp);
      lm = fma(f.kdt_m, c.theta_m - lm, lm);
      if (jp != 0.0 || jm != 0.0) {
        xi += jp + jm;
        lp += fma(c.beta1_p, jp, c.beta2_p * jm);
        lm += fma(c.beta1_m, jp, c.beta2_m * jm);
      }
    };
    const int S = a.nsteps;
    for (int s = 0; s < S; s += 4) {                  // four steps: one (float) or two (fp64) calls of normals, two calls of clocks
      double z[4];
      if constexpr (GAUSS == kGaussF64) {
        rng.get((uint32_t)(s >> 1), z[0], z[1]);
        if (s + 2 < S) rng.get((uint32_t)(s >> 1) + 1u, z[2], z[3]);
      } else {
        rng.get2((uint32_t)(s >> 2), z[0], z[1], z[2], z[3]);
      }
      const uint4 c0 = hawkes_clock_words(key, plo, phi, (uint32_t)(s >> 1), a.slice);
      one_step(z[0], c0.x, c0.y, (uint32_t)s);
      if (s + 1 < S) one_step(z[1], c0.z, c0.w, (uint32_t)s + 1u);
      if (s + 2 < S) {
        const uint4 c1 = hawkes_clock_words(key, plo, phi, (uint32_t)(s >> 1) + 1u, a.slice);
        one_step(z[2], c1.x, c1.y, (uint32_t)s + 2u);
        if (s + 3 < S) one_step(z[3], c1.z, c1.w, (uint32_t)s + 3u);
      }
    }
    a.x[i] = xi;
    a.lam_p[i] = lp;
    a.lam_m[i] = lm;
    const double spot = a.forward * exp(xi);
    if (spot == spot) {
      acc[0] += spot;
      acc[1] += 1.0;
    }
  }
  block_sum<2, kThreads>(acc, red);
  if (threadIdx.x == 0) {
    a.partials[2 * blockIdx.x + 0] = acc[0];
    a.partials[2 * blockIdx.x + 1] = acc[1];
  }
}

// the in-kernel draws of the slice kernel in the reference's form: W0 = sqrt(dt) z, U = -ln(u)/dt, J = shift +- mean (-ln(u))   [S][n] each
template <int GAUSS>
__global__ void hawkes_device_draws_kernel(unsigned long long seed, unsigned long long path0, long long n, unsigned int slice, int S, HawkesConsts c,
                                           double* __restrict__ W0, double* __restrict__ U_P, double* __restrict__ U_M,
                                           double* __restrict__ J_P, double* __restrict__ J_M) {
  if constexpr (GAUSS != kGaussF32) gauss64_table_init();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long path = path0 + (unsigned long long)i;
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  StepNormals<double, GAUSS> rng(seed, path, slice);
  double z[4];
  for (int s = 0; s < S; ++s) {
    if constexpr (GAUSS == kGaussF64) {
      if ((s & 1) == 0) rng.get((uint32_t)(s >> 1), z[0], z[1]);
    } else {
      if ((s & 3) == 0) rng.get2((uint32_t)(s >> 2), z[0], z[1], z[2], z[3]);
    }
    const uint4 ck = hawkes_clock_words(key, (uint32_t)path, (uint32_t)(path >> 32), (uint32_t)(s >> 1), slice);
    const uint4 sz = hawkes_size_words(key, (uint32_t)path, (uint32_t)(path >> 32), (uint32_t)s, slice);
    const size_t o = (size_t)s * n + i;
    W0[o] = __dmul_rn(c.sqrt_dt, GAUSS == kGaussF64 ? z[s & 1] : z[s & 3]);
    U_P[o] = hawkes_clock(hawkes_uniform((s & 1) ? ck.z : ck.x), c);
    U_M[o] = hawkes_clock(hawkes_uniform((s & 1) ? ck.w : ck.y), c);
    J_P[o] = hawkes_size_p(hawkes_uniform(sz.x), c);
    J_M[o] = hawkes_size_m(hawkes_uniform(sz.y), c);
  }
}

static int check_hawkes_flags(int flags) {
  const int g = gauss_mode(flags);
  return g == kGaussF32 || g == kGaussF64 ? 0 : fail(-1, "invalid argument: gauss flags");
}

static int launch_hawkes_slice(double* x, double* lp, double* lm, long long n, long long path_offset, int init, const b200sv_hawkes_params& p,
                               int nsteps, double dt, int slice_index, double forward, uint64_t seed, int flags, double* moments_out,
                               cudaStream_t st, P2pCtx* p2p = nullptr) {
  if (int rc = check_hawkes_flags(flags)) return rc;
  HawkesSliceArgs a;
  a.x = x;
  a.lam_p = lp;
  a.lam_m = lm;
  a.n = n;
  a.path_offset = (unsigned long long)path_offset;
  a.init = init;
  a.lam_p0 = p.lambda_p;
  a.lam_m0 = p.lambda_m;
  a.nsteps = nsteps;
  a.slice = (unsigned int)slice_index;
  a.seed = seed;
  a.forward = forward;
  const HawkesConsts c = make_hawkes_consts(p, dt);
  Grid grid = persistent_grid(hawkes_slice_kernel<kGaussF32>, kThreads, n);
  DevBuf<double> partials(st);
  ensure_pool_threshold();
  B200SV_CUDA(partials.alloc(2 * (size_t)grid.blocks));
  a.partials = partials.p;
  if (gauss_mode(flags) == kGaussF64)
    hawkes_slice_kernel<kGaussF64><<<grid.blocks, grid.threads, 0, st>>>(a, c);
  else
    hawkes_slice_kernel<kGaussF32><<<grid.blocks, grid.threads, 0, st>>>(a, c);
  if (int rc = launched("hawkes_slice_kernel")) return rc;
  reduce_partials_kernel<<<1, 64, 0, st>>>(partials.p, grid.blocks, 2, 2, moments_out, make_publish(p2p, st));   // exchange #1 (producer)
  return launched("reduce_partials_kernel");
}

constexpr int kHawkesStepsPerYear = 5 * 360;     // hawkes_jd_pricer.py:752

static int hawkes_chain_host(const b200sv_hawkes_params* p, int M, const double* ttms, const double* forwards, const double* discfactors,
                             const int* offsets, const double* strikes, const int8_t* types, long long nb_path, int variable_type, uint64_t seed,
                             int flags, double* prices_out, double* stderr_out) {
  B200SV_REQUIRE(nb_path >= 1, "nb_path must be >= 1");
  B200SV_REQUIRE(!(flags & B200SV_STATE_F32), "the Hawkes route is float64 only");
  if (int rc = validate_chain(M, ttms, offsets, types, variable_type)) return rc;
  if (int rc = check_hawkes_flags(flags)) return rc;
  const size_t N = (size_t)nb_path;
  return host_call([&](cudaStream_t st) {
    DevBuf<double> d(st);
    ChainPayoffs pay(st, M, ttms, forwards, discfactors, offsets, types, variable_type, 1, false);
    B200SV_CUDA(d.alloc(3 * N));
    if (int rc = pay.alloc(strikes)) return rc;
    double t0 = 0.0;
    for (int m = 0; m < M; ++m) {
      int S;
      double dt;
      time_grid(ttms[m] - t0, kHawkesStepsPerYear, &S, &dt);
      t0 = ttms[m];
      if (int rc = launch_hawkes_slice(d.p, d.p + N, d.p + 2 * N, nb_path, 0, m == 0, *p, S, dt, m, forwards[m], seed, flags, pay.d_mom.p, st))
        return rc;
      // compute_mc_vars_payoff(x0=x0, sigma0=x0, qvar0=x0, ...) (:703): the log-return array stands in for every argument
      if (int rc = pay.run(0, m, d.p, d.p, nb_path, false, (double)nb_path, st)) return rc;
    }
    return pay.copy_back(prices_out, stderr_out, nullptr, st);
  });
}

}  // namespace b200sv
