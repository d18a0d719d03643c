// TEST TOOL -- compiles the product's screen fast path (unconfined_b200/csrc/fast.cuh: segment
// split, S(x) = sinh(x)/x, screen means) for the HOST so that CPU tests can compare it with the
// oracle at single (a,p) points.  Not linked into libunconfined_b200.so.
#include <cstring>
#include "../../unconfined_b200/csrc/fast.cuh"

extern "C" {

static double g_mn_vartheta = 0.0, g_mn_u0 = 1.0;
// run constants of model 6 (DevParams::mn_vartheta, mn_u0) for the next hc_fast_screen calls
void hc_set_mn(double vartheta, double u0) { g_mn_vartheta = vartheta; g_mn_u0 = u0; }

// the screen mean of fp over [zbot, ztop] (lh_screen_kernel's fast path: segments, per-(a,p)
// terms, one exp_pm + sincos + S(eta h) per segment), without the common factor.  Returns 0 if
// the fast path declined.
int hc_fast_screen(int model, double kappa, double alphaD, double beta, double lD, double dD, double bD,
                   int moench_M, double aux_re, double aux_im, double aux2_re, double aux2_im, double a,
                   double p_re, double p_im, double zbot, double ztop, double *out, double *eta_out) {
  unc::DevParams P;
  std::memset(&P, 0, sizeof P);
  P.mn_vartheta = g_mn_vartheta; P.mn_u0 = g_mn_u0;
  P.model = model; P.kappa = kappa; P.alphaD = alphaD; P.beta = beta;
  P.lD = lD; P.dD = dD; P.bD = bD; P.lD1 = 1.0 - lD; P.dD1 = 1.0 - dD; P.moench_M = moench_M;
  unc::ScreenSegs sg;
  unc::screen_segments(zbot, ztop, P.lD1, P.dD1, &sg);
  unc::cplx eta;
  unc::Coef co[3];
  bool ok = unc::ap_terms_fast(P, unc::mk(p_re, p_im), unc::mk(aux_re, aux_im), unc::mk(aux2_re, aux2_im), a * a,
                               1.0, sg.lay_mask, unc::fast_eta_max(P, sg.lay_mask, ztop), &eta, co);
  eta_out[0] = eta.re; eta_out[1] = eta.im;
  if (!ok) return 0;
  const unc::cplx f = model == 0 ? unc::screen_mean_fast<0>(eta, co, sg) : unc::screen_mean_fast<-1>(eta, co, sg);
  out[0] = f.re; out[1] = f.im;
  return 1;
}

// S(x) = sinh(x)/x of the fast path
void hc_sinhc(double re, double im, double *out) {
  const unc::cplx s = unc::sinhc_fast(unc::mk(re, im));
  out[0] = s.re; out[1] = s.im;
}

}  // extern "C"
