// ivol_kernels.cu -- batched Black-76 implied-volatility inversion (SURVEY.md §8f "next" #1).
//
// In the reference this step is third-party (vanilla_option_pricers.infer_bsm_ivols_from_model_chain_prices, called from
// data/option_chain.py:327-346 right after every price_chain / model_mc_price_chain in compute_chain_prices_with_vols,
// model_pricer.py:109-120, and compute_mc_chain_implied_vols, :216-241).  That package is not in the reference tree, so bit-level
// parity with it is unpinned (DESIGN.md §2); what the reference pins -- the quickstart vols 0.999577 / 0.995757 and flat-vol
// round trips -- holds for any correct inversion; the reference's own assertions about the step (flat-vol recovery 1e-10, chain round trip
// 2e-10, single-option round trip 2e-12, slice / vanilla self-consistency 1e-12) are ported in tests/test_gpu_ivol_pins.py.  One thread per
// quote: safeguarded Newton in total-vol space (black.cuh), fp64 normcdf; the checker oracle/bsm.py is an independent 80-step bisection.
#include <cmath>
#include <vector>

#include "../../include/b200sv.h"
#include "common.cuh"
#include "black.cuh"

namespace b200sv {

struct QuoteSpec {
  double forward, strike, ttm, discfactor, price;
  int type;
};

__global__ void black_ivol_kernel(const QuoteSpec* __restrict__ q, int n, double* __restrict__ ivols) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const QuoteSpec s = q[i];
  ivols[i] = black_implied_vol(s.forward, s.strike, s.ttm, s.discfactor, s.price, s.type);
}

}  // namespace b200sv

using namespace b200sv;

extern "C" int b200sv_bsm_implied_vols(int M, const double* ttms, const double* forwards, const double* discfactors, const int* offsets,
                                       const double* strikes, const int8_t* types, const double* prices, double* ivols_out) {
  B200SV_REQUIRE(ttms && forwards && discfactors && offsets && strikes && types && prices && ivols_out, "null pointer");
  B200SV_REQUIRE(M >= 1, "M >= 1");
  const int n = offsets[M] - offsets[0];
  if (n <= 0) return 0;
  std::vector<QuoteSpec> q(n);
  for (int m = 0; m < M; ++m)
    for (int j = offsets[m]; j < offsets[m + 1]; ++j) {
      if (types[j] < 0 || types[j] > 3) return fail(-3, "unknown option payoff code");
      q[j - offsets[0]] = QuoteSpec{forwards[m], strikes[j], ttms[m], discfactors[m], prices[j - offsets[0]], (int)types[j]};
    }
  return host_call([&](cudaStream_t st) {
    DevBuf<QuoteSpec> dq(st);
    DevBuf<double> dv(st);
    B200SV_CUDA(dq.upload(q.data(), n));
    B200SV_CUDA(dv.alloc(n));
    black_ivol_kernel<<<(n + 63) / 64, 64, 0, st>>>(dq.p, n, dv.p);
    if (int rc = launched("black_ivol_kernel")) return rc;
    B200SV_CUDA(cudaMemcpyAsync(ivols_out, dv.p, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    return 0;
  });
}
