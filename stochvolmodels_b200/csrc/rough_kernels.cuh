// rough_kernels.cuh -- rough-LogSV multi-factor Monte Carlo (Markovian lift of the rough kernel, n <= 8 factors) for sm_100a.
// Included by mc_kernels.cu (same translation unit: it reuses the payoff / reduction launchers and the Philox generator).
//
// Replaces, behind the C ABI of include/b200sv.h (paths under /root/reference/src/stochvolmodels/pricers):
//   log_spot_full_combined (f64 branch)            rough_logsv/split_simulation.py:340-361, 466-479
//     log_spot_full_solve2_f64                     :287-337      log-spot increment from the vol increment (c1 = c2 = 1/2)
//     drift_diffus_strand_f64                      :253-284      Strang splitting D(h/2) S(h) D(h/2)
//     drift_ode_solve2                             :76-124       classical RK4 on z_i' = -x_i (z_i - v0_i) + (k1 + k2 <w,z>)(theta - <w,z>)
//     diffus_sde_solve_f64                         :231-250      exact log-normal step of <w,z>, the same shift added to every factor
//   rough_logsv_mc_chain_pricer_fixed_randoms      logsv_pricer.py:1164-1232   (every maturity RESTARTS at t = 0 on its own grid and
//                                                  consumes the first S_m rows of Z0 / Z1)
//
// One thread = one path for the whole grid; the n factor values live in registers (template on n), the only HBM traffic is the two
// normals per step in the fixed-random mode (16 B / path-step, coalesced [S][P] rows) or nothing at all in the Philox mode, plus the
// terminal state.  ~160 fp64 instructions per step at n = 3 (8 RK4 slopes, one table exponential, one MUFU-seeded sqrt): fp64-pipe bound.
// The reference kernels are compiled fastmath=True, so its own evaluation order is not fixed; agreement with it is 1e-12.
#pragma once

namespace b200sv {

constexpr int kMaxRoughFactors = 8;

struct RoughConsts {
  double nodes[kMaxRoughFactors], weight[kMaxRoughFactors], wlam[kMaxRoughFactors];   // x_i, w_i, w_i x_i
  double v0;            // sigma0 / sum(w): initial value and mean-reversion anchor of EVERY factor (logsv_pricer.py:1194)
  double theta, kappa1, kappa2;
  double volvol, rho, rho_comp, inv_volvol;     // vartheta = sqrt(beta^2 + orthog_vol^2), rho = beta / vartheta (logsv_pricer.py:1197-1198)
  double wsum, w_inv, vv, w_lam_v0;             // sum w, 1 / sum w, vartheta * sum w, sum w_i x_i v0
  double h, half_h, sqrt_h, inv_h;
};

static RoughConsts make_rough_consts(const b200sv_logsv_params& p, int n, const double* weights, const double* nodes, double h) {
  RoughConsts c{};
  double wsum = 0.0;
  for (int i = 0; i < n; ++i) wsum += weights[i];
  c.v0 = p.sigma0 / wsum;
  c.w_lam_v0 = 0.0;
  for (int i = 0; i < n; ++i) {
    c.nodes[i] = nodes[i];
    c.weight[i] = weights[i];
    c.wlam[i] = weights[i] * nodes[i];
    c.w_lam_v0 += c.wlam[i] * c.v0;
  }
  c.theta = p.theta;
  c.kappa1 = p.kappa1;
  c.kappa2 = p.kappa2;
  c.volvol = std::sqrt(p.beta * p.beta + p.volvol * p.volvol);     // p.volvol carries the ORTHOGONAL vol-of-vol on this route
  c.rho = p.beta / c.volvol;
  c.rho_comp = std::sqrt(1.0 - c.rho * c.rho);
  c.inv_volvol = 1.0 / c.volvol;
  c.wsum = wsum;
  c.w_inv = 1.0 / wsum;
  c.vv = c.volvol * wsum;
  c.h = h;
  c.half_h = 0.5 * h;
  c.sqrt_h = std::sqrt(h);
  c.inv_h = 1.0 / h;
  return c;
}

template <int N>
struct RoughPath {
  double v[N];
  double ls, y;

  __device__ __forceinline__ static double wsum_of(const RoughConsts& c, const double (&z)[N]) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < N; ++i) s = fma(c.weight[i], z[i], s);
    return s;
  }
  // slope of the drift ODE at z (split_simulation.py:100-103)
  __device__ __forceinline__ static void slope(const RoughConsts& c, const double (&z)[N], double (&s)[N]) {
    const double zw = wsum_of(c, z);
    const double g = (c.kappa1 + c.kappa2 * zw) * (c.theta - zw);
#pragma unroll
    for (int i = 0; i < N; ++i) s[i] = fma(-c.nodes[i], z[i] - c.v0, g);
  }
  // classical RK4 over a step of size hh (drift_ode_solve2, :76-124)
  __device__ __forceinline__ static void drift(const RoughConsts& c, double (&z)[N], double hh) {
    double s1[N], s2[N], s3[N], s4[N], t[N];
    slope(c, z, s1);
#pragma unroll
    for (int i = 0; i < N; ++i) t[i] = fma(0.5 * hh, s1[i], z[i]);
    slope(c, t, s2);
#pragma unroll
    for (int i = 0; i < N; ++i) t[i] = fma(0.5 * hh, s2[i], z[i]);
    slope(c, t, s3);
#pragma unroll
    for (int i = 0; i < N; ++i) t[i] = fma(hh, s3[i], z[i]);
    slope(c, t, s4);
#pragma unroll
    for (int i = 0; i < N; ++i) z[i] = fma(hh / 6.0, (s1[i] + 2.0 * s2[i]) + (2.0 * s3[i] + s4[i]), z[i]);
  }
  __device__ __forceinline__ void init(const RoughConsts& c) {
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = c.v0;
    ls = 0.0;
    y = 0.0;
  }
  // one time step (log_spot_full_solve2_f64, :287-337): z0 drives the volatility, z1 the orthogonal part of the spot
  __device__ __forceinline__ void step(const RoughConsts& c, double z0, double z1) {
    const double vw = wsum_of(c, v);
    double w_lam_vol = 0.0;
#pragma unroll
    for (int i = 0; i < N; ++i) w_lam_vol = fma(c.wlam[i], v[i], w_lam_vol);
    // Strang splitting (:281-283)
    double u[N];
#pragma unroll
    for (int i = 0; i < N; ++i) u[i] = v[i];
    drift(c, u, c.half_h);
    const double yw = wsum_of(c, u);
    const double ex = clamp_log(fma(c.vv, z0 * c.sqrt_h, -0.5 * c.vv * c.vv * c.h));
    const double Yh = yw * exp_table(ex);                                               // diffus_sde_solve_f64 (:240-243)
    const double Q = c.w_inv * (Yh - yw);
#pragma unroll
    for (int i = 0; i < N; ++i) u[i] += Q;
    drift(c, u, c.half_h);
    double volw_h = wsum_of(c, u);
    if (!(volw_h > 0.0)) {          // NaN or <= 0: the reference resets every factor of that path to 1e-6 (:310-312)
#pragma unroll
      for (int i = 0; i < N; ++i) u[i] = 1e-6;
      volw_h = wsum_of(c, u);
    }
    double w_lam_vol_h = 0.0;
#pragma unroll
    for (int i = 0; i < N; ++i) w_lam_vol_h = fma(c.wlam[i], u[i], w_lam_vol_h);
    const double sq_vw = vw * vw, sq_vhw = volw_h * volw_h;
    const double term1 = c.inv_volvol *
                         (((volw_h - vw) * c.inv_h + 0.5 * w_lam_vol + 0.5 * w_lam_vol_h - c.w_lam_v0) * c.w_inv - c.kappa1 * c.theta +
                          (c.kappa1 - c.kappa2 * c.theta) * (0.5 * vw + 0.5 * volw_h) + c.kappa2 * (0.5 * sq_vw + 0.5 * sq_vhw)) *
                         c.h;
    const double term2 = 0.5 * c.h * sq_vw + 0.5 * c.h * sq_vhw;
    ls = ls - 0.5 * term2 + c.rho * term1 + c.rho_comp * (term2 > 0.0 ? fast_sqrt(term2) : sqrt(term2)) * z1;
    y = fma(0.5 * c.h, sq_vw + sq_vhw, y);
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = u[i];
  }
};

// Z0 / Z1 != nullptr: caller-supplied unit normals, row-major [S][P] (device); else in-kernel Philox draws (stream of philox.cuh with
// slice = 0 for EVERY maturity, so that maturity m consumes the first S_m steps of one fixed stream per path, as the reference does with
// the rows of Z0 / Z1).  vol_out: [N][P] factor values (may be nullptr), log_spot_out / qv_out: [P].
template <int N, int GAUSS>
__global__ void __launch_bounds__(kThreads) rough_logsv_kernel(double* __restrict__ log_spot_out, double* __restrict__ vol_out,
                                                              double* __restrict__ qv_out, const double* __restrict__ Z0,
                                                              const double* __restrict__ Z1, int S, long long P, RoughConsts c,
                                                              unsigned long long seed, unsigned long long path_offset) {
  exp_table_init();
  if constexpr (GAUSS != kGaussF32) gauss64_table_init();
  const long long stride = (long long)gridDim.x * kThreads;
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < P; i += stride) {
    RoughPath<N> p;
    p.init(c);
    if (Z0) {
      for (int s = 0; s < S; ++s) p.step(c, __ldg(Z0 + (size_t)s * P + i), __ldg(Z1 + (size_t)s * P + i));
    } else {
      StepNormals<double, GAUSS> rng(seed, path_offset + (unsigned long long)i, 0u);
      if constexpr (GAUSS == kGaussF64) {
        for (int s = 0; s < S; ++s) {
          double z0, z1;
          rng.get((uint32_t)s, z0, z1);
          p.step(c, z0, z1);
        }
      } else {
        for (int cidx = 0; 2 * cidx < S; ++cidx) {
          double a0, a1, b0, b1;
          rng.get2((uint32_t)cidx, a0, a1, b0, b1);
          p.step(c, a0, a1);
          if (2 * cidx + 1 < S) p.step(c, b0, b1);
        }
      }
    }
    log_spot_out[i] = p.ls;
    qv_out[i] = p.y;
    if (vol_out) {
#pragma unroll
      for (int k = 0; k < N; ++k) vol_out[(size_t)k * P + i] = p.v[k];
    }
  }
}

template <int N>
static int launch_rough_n(double* ls, double* vol, double* qv, const double* Z0, const double* Z1, int S, long long P, const RoughConsts& c,
                          uint64_t seed, long long path_offset, int gauss, cudaStream_t st) {
  Grid g = persistent_grid(rough_logsv_kernel<N, kGaussF32>, kThreads, P);
  if (gauss == kGaussF64)
    rough_logsv_kernel<N, kGaussF64><<<g.blocks, g.threads, 0, st>>>(ls, vol, qv, Z0, Z1, S, P, c, seed, (unsigned long long)path_offset);
  else
    rough_logsv_kernel<N, kGaussF32><<<g.blocks, g.threads, 0, st>>>(ls, vol, qv, Z0, Z1, S, P, c, seed, (unsigned long long)path_offset);
  return launched("rough_logsv_kernel");
}

static int launch_rough(int n, double* ls, double* vol, double* qv, const double* Z0, const double* Z1, int S, long long P, const RoughConsts& c,
                        uint64_t seed, long long path_offset, int gauss, cudaStream_t st) {
  switch (n) {
    case 1: return launch_rough_n<1>(ls, vol, qv, Z0, Z1, S, P, c, seed, path_offset, gauss, st);
    case 2: return launch_rough_n<2>(ls, vol, qv, Z0, Z1, S, P, c, seed, path_offset, gauss, st);
    case 3: return launch_rough_n<3>(ls, vol, qv, Z0, Z1, S, P, c, seed, path_offset, gauss, st);
    case 4: return launch_rough_n<4>(ls, vol, qv, Z0, Z1, S, P, c, seed, path_offset, gauss, st);
    case 5: return launch_rough_n<5>(ls, vol, qv, Z0, Z1, S, P, c, seed, path_offset, gauss, st);
    case 6: return launch_rough_n<6>(ls, vol, qv, Z0, Z1, S, P, c, seed, path_offset, gauss, st);
    case 7: return launch_rough_n<7>(ls, vol, qv, Z0, Z1, S, P, c, seed, path_offset, gauss, st);
    case 8: return launch_rough_n<8>(ls, vol, qv, Z0, Z1, S, P, c, seed, path_offset, gauss, st);
  }
  return fail(-1, "invalid argument: the rough-vol kernel supports 1..8 factors");
}

// host-level chain driver: B parameter sets x M maturities on ONE upload of the normals (or none at all with Philox draws)
static int rough_chain_host(const b200sv_logsv_params* params, int B, int n, const double* weights /*[B][n]*/, const double* nodes /*[B][n]*/, int M,
                            const double* ttms, const double* forwards, const double* discfactors, const int* offsets, const double* strikes,
                            const int8_t* types, long long nb_path, const int* nsteps /*[M]*/, const double* hs /*[M]*/, const double* Z0,
                            const double* Z1, long long z_rows, int variable_type, uint64_t seed, int flags, double* prices_out,
                            double* stderr_out, double* ivols_out, double* states_out /* B == 1: [M][(n+2)][P] log_spot, vol[n], qv */) {
  B200SV_REQUIRE(B >= 1 && n >= 1 && n <= kMaxRoughFactors, "B >= 1 and 1 <= n_factors <= 8");
  B200SV_REQUIRE(nb_path >= 1, "nb_path must be >= 1");
  B200SV_REQUIRE((Z0 == nullptr) == (Z1 == nullptr), "Z0 and Z1 must be supplied together");
  B200SV_REQUIRE(!states_out || B == 1, "terminal states are returned for a single parameter set");
  if (int rc = validate_chain(M, ttms, offsets, types, variable_type)) return rc;
  const int g = gauss_mode(flags);
  B200SV_REQUIRE(g == kGaussF32 || g == kGaussF64, "gauss flags");
  B200SV_REQUIRE(!(flags & B200SV_STATE_F32), "the rough-vol route is float64 only");
  int Smax = 0;
  for (int m = 0; m < M; ++m) {
    B200SV_REQUIRE(nsteps[m] >= 1 && hs[m] > 0.0, "nsteps / h must be positive");
    Smax = std::max(Smax, nsteps[m]);
  }
  B200SV_REQUIRE(!Z0 || z_rows >= Smax, "Z0 / Z1 have fewer rows than the longest grid");
  const size_t P = (size_t)nb_path;
  return host_call([&](cudaStream_t st) {
    DevBuf<double> d_state(st), d_z(st);
    ChainPayoffs pay(st, M, ttms, forwards, discfactors, offsets, types, variable_type, B, ivols_out != nullptr);
    B200SV_CUDA(d_state.alloc((size_t)(n + 2) * P));
    if (Z0) {
      B200SV_CUDA(d_z.alloc(2 * (size_t)Smax * P));
      B200SV_CUDA(cudaMemcpyAsync(d_z.p, Z0, sizeof(double) * (size_t)Smax * P, cudaMemcpyHostToDevice, st));
      B200SV_CUDA(cudaMemcpyAsync(d_z.p + (size_t)Smax * P, Z1, sizeof(double) * (size_t)Smax * P, cudaMemcpyHostToDevice, st));
    }
    if (int rc = pay.alloc(strikes)) return rc;
    double *d_ls = d_state.p, *d_vol = d_state.p + P, *d_qv = d_state.p + (size_t)(n + 1) * P;
    for (int b = 0; b < B; ++b)
      for (int m = 0; m < M; ++m) {
        const RoughConsts c = make_rough_consts(params[b], n, weights + (size_t)b * n, nodes + (size_t)b * n, hs[m]);
        if (int rc = launch_rough(n, d_ls, d_vol, d_qv, d_z.p, Z0 ? d_z.p + (size_t)Smax * P : nullptr, nsteps[m], nb_path, c, seed, 0, g, st))
          return rc;
        if (states_out)
          B200SV_CUDA(cudaMemcpyAsync(states_out + (size_t)m * (n + 2) * P, d_state.p, sizeof(double) * (size_t)(n + 2) * P, cudaMemcpyDeviceToHost, st));
        if (offsets[m + 1] == offsets[m]) continue;
        if (int rc = b200sv_dev_spot_moments(d_ls, nb_path, forwards[m], pay.d_mom.p, st)) return rc;
        // the reference hands (1, nb_path)-shaped arrays to compute_mc_vars_payoff, whose "/ sqrt(x0.shape[0])" is then "/ 1":
        // this route's std errors are discfactor * nanstd(payoff) (total_paths = 1)
        if (int rc = pay.run(b, m, d_ls, d_qv, nb_path, false, 1.0, st)) return rc;
      }
    return pay.copy_back(prices_out, stderr_out, ivols_out, st);
  });
}

}  // namespace b200sv
