// TEST TOOL -- compiles the product's vertical-gradient fast path (unconfined_b200/csrc/fast.cuh:
// dz_terms_fast, dz_coef, eval_dz_split) for the HOST so that CPU tests can compare it with the
// oracle at single (a,p,z) points.  Not linked into libunconfined_b200.so.
#include <cmath>
#include <cstring>
#include "../../unconfined_b200/csrc/fast.cuh"

namespace {
double g_mn_vartheta = 0.0, g_mn_u0 = 1.0;

unc::DevParams params(int model, double kappa, double alphaD, double beta, double lD, double dD, double bD,
                      int moench_M) {
  unc::DevParams P;
  std::memset(&P, 0, sizeof P);
  P.mn_vartheta = g_mn_vartheta; P.mn_u0 = g_mn_u0;
  P.model = model; P.kappa = kappa; P.alphaD = alphaD; P.beta = beta;
  P.lD = lD; P.dD = dD; P.bD = bD; P.lD1 = 1.0 - lD; P.dD1 = 1.0 - dD; P.moench_M = moench_M;
  return P;
}

bool finite_c(unc::cplx c) { return std::isfinite(c.re) && std::isfinite(c.im); }
}  // namespace

extern "C" {

// run constants of model 6 (DevParams::mn_vartheta, mn_u0) for the next calls
void hc_set_mn(double vartheta, double u0) { g_mn_vartheta = vartheta; g_mn_u0 = u0; }

// df/dz at z of the formula of layer `lay` (1..3; 0 = the geometric layer of z, as
// lh_column_kernel<COL_DZ>), without the common factor, with fast_eta_max of a point at z.
// Returns 0 if the fast path declined.
int hc_fast_dz(int model, double kappa, double alphaD, double beta, double lD, double dD, double bD, int moench_M,
               double aux_re, double aux_im, double aux2_re, double aux2_im, double a, double p_re, double p_im,
               double z, int lay, double *out, double *eta_out) {
  const unc::DevParams P = params(model, kappa, alphaD, beta, lD, dD, bD, moench_M);
  if (lay <= 0) lay = (z < P.lD1) ? 1 : ((z < P.dD1) ? 2 : 3);
  unc::cplx eta, f;
  bool ok = unc::dz_terms_fast<-1>(P, unc::mk(p_re, p_im), unc::mk(aux_re, aux_im), unc::mk(aux2_re, aux2_im),
                                   a * a, 1.0, lay, unc::fast_eta_max(P, 1 << (lay - 1), z), z, &eta, &f);
  eta_out[0] = eta.re; eta_out[1] = eta.im;
  if (!ok) return 0;
  out[0] = f.re; out[1] = f.im;
  return 1;
}

// Overflow check of the derivative terms at the edge of the fast path: for the given eta
// (Re(eta)*m up to UNC_FAST_EXP_MAX, |Im eta| up to 2e5, w = 1, p = kappa eta^2 with a = 0),
// every layer's (k0, cp, cm), the water-table term, the derivative coefficients and both
// derivative forms (eval_dz_fast, eval_dz_split) at z in {0, 1-lD, 1-dD, 1} must be finite.
// Returns the number of non-finite intermediates (0 = ok), or -1 if the fast path declined.
int hc_dz_overflow_check(int model, double kappa, double alphaD, double beta, double lD, double dD, double bD,
                         int moench_M, double aux_re, double aux_im, double eta_re, double eta_im) {
  const unc::DevParams P = params(model, kappa, alphaD, beta, lD, dD, bD, moench_M);
  // p = kappa eta^2 (a = 0)
  const unc::cplx p = unc::mk(kappa * (eta_re * eta_re - eta_im * eta_im), kappa * 2.0 * eta_re * eta_im);
  unc::cplx eta;
  unc::Coef co[3];
  unc::cplx wt[2] = {unc::mk(0.0, 0.0), unc::mk(0.0, 0.0)};
  const unc::DzSink sink{co, wt};
  if (!unc::ap_terms_fast_s<-1>(P, p, unc::mk(aux_re, aux_im), unc::mk(1.0, 0.0), 0.0, 1.0, 7,
                                unc::fast_eta_max(P, 7, 1.0), &eta, sink))
    return -1;
  int bad = !finite_c(wt[0]) + !finite_c(wt[1]);
  const double zs[4] = {0.0, P.lD1, P.dD1, 1.0};
  for (int L = 0; L < 3; ++L) {
    const unc::Coef d = unc::dz_coef(eta, co[L]);
    bad += !finite_c(co[L].k0) + !finite_c(co[L].cp) + !finite_c(co[L].cm) + !finite_c(d.cp) + !finite_c(d.cm);
    for (double z : zs)
      bad += !finite_c(unc::eval_dz_fast(eta, co[L], z)) + !finite_c(unc::eval_dz_split(eta, co[L], wt[0], wt[1], z));
  }
  return bad;
}

}  // extern "C"
