// TEST INFRASTRUCTURE ONLY -- C entry points of the screen oracle (oracle_screens.hpp),
// loaded through ctypes by oracle/screens.py for tests/ only; never by the product.  A library
// of its own next to liboracle.so (same flags); it carries its own libm-jitter state, set by
// orcs_set_jitter.
#include <cstdint>
#include <cstring>
#include <vector>
#include <cmath>
#ifdef _OPENMP
#include <omp.h>
#endif
#include "oracle_screens.hpp"

using namespace orc;

namespace {

template <class T>
int eval_screens_t(const params *prm, int64_t n, const double *tD, const int32_t *sv, const double *rD,
                   const double *zbot, const double *ztop, const double *ts_scale, int nthreads, double *s,
                   double *ds, int32_t *flags) {
  for (int64_t c = 0; c < n; ++c)
    if (!(zbot[c] >= 0.0 && ztop[c] <= 1.0 && zbot[c] < ztop[c])) return 1;
  tables<T> tb;
  tb.build(*prm);
#ifdef _OPENMP
  if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
#pragma omp parallel for schedule(dynamic, 1)
  for (int64_t c = 0; c < n; ++c) {
    const screen<T> sc = screen_segments<T>(zbot[c], ztop[c], *prm);
    T so, dso;
    int32_t fl;
    T scl = ts_scale ? T(ts_scale[c]) : T(prm->j0z[sv[c] - 1]) / T(rD[c]);
    eval_screen<T>(*prm, tb, T(tD[c]), sv[c], T(rD[c]), scl, sc, &so, &dso, &fl);
    s[c] = (double)so;
    ds[c] = (double)dso;
    if (flags) flags[c] = fl;
  }
  return 0;
}

template <class T>
void soln_screen_t(const params *prm, double a, double rD, double tD, double zbot, double ztop, double *out) {
  std::vector<cx<T>> p, lt, fp;
  dehoog_pvalues<T>(T(prm->tee_mult) * T(tD), *prm, p);
  lap_time<T>(*prm, p, lt);
  lap_hank_soln_screen<T>(T(a), T(rD), p, screen_segments<T>(zbot, ztop, *prm), *prm, lt, fp);
  for (size_t i = 0; i < fp.size(); ++i) { out[2 * i] = (double)fp[i].re; out[2 * i + 1] = (double)fp[i].im; }
}

}  // namespace

extern "C" {

// ulps = 0 disables; see oracle_math.hpp (jitter)
void orcs_set_jitter(double ulps, unsigned long long seed) {
  jitter().ulps = ulps;
  jitter().seed = seed;
}

// screened observation wells (unc_eval_screens' definition): one result per screen
// [zbot, ztop]; returns 1 if a screen is not a non-empty interval in [0, 1]
int orc_eval_screens(const params *prm, int64_t n, const double *tD, const int32_t *sv, const double *rD,
                     const double *zbot, const double *ztop, const double *ts_scale, int nthreads, double *s,
                     double *ds, int32_t *flags) {
  return eval_screens_t<double>(prm, n, tD, sv, rD, zbot, ztop, ts_scale, nthreads, s, ds, flags);
}

int orc_eval_screens_ld(const params *prm, int64_t n, const double *tD, const int32_t *sv, const double *rD,
                        const double *zbot, const double *ztop, const double *ts_scale, int nthreads, double *s,
                        double *ds, int32_t *flags) {
  return eval_screens_t<long double>(prm, n, tD, sv, rD, zbot, ztop, ts_scale, nthreads, s, ds, flags);
}

// the screen-averaged lap_hank_soln at one abscissa for the p-vector of time tD; out[p*2 + {0,1}]
void orc_soln_screen(const params *prm, double a, double rD, double tD, double zbot, double ztop, double *out) {
  soln_screen_t<double>(prm, a, rD, tD, zbot, ztop, out);
}

void orc_soln_screen_ld(const params *prm, double a, double rD, double tD, double zbot, double ztop, double *out) {
  soln_screen_t<long double>(prm, a, rD, tD, zbot, ztop, out);
}

}  // extern "C"
