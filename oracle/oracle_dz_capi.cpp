// TEST INFRASTRUCTURE ONLY -- C entry points of the vertical-gradient oracle (oracle_dz.hpp),
// loaded through ctypes by oracle/dz.py for tests/ only; never by the product.  A library of
// its own next to liboracle.so (same flags); it carries its own libm-jitter state, set by
// orcd_set_jitter.
#include <cstdint>
#include <cstring>
#include <vector>
#include <cmath>
#ifdef _OPENMP
#include <omp.h>
#endif
#include "oracle_dz.hpp"

using namespace orc;

namespace {

template <class T>
int eval_points_dz_t(const params *prm, int64_t n, const double *tD, const int32_t *sv, const double *rD,
                     const double *zD, const double *ts_scale, int nthreads, double *gz, double *dgz,
                     int32_t *flags) {
  for (int64_t c = 0; c < n; ++c)
    if (!(zD[c] >= 0.0 && zD[c] <= 1.0)) return 1;
  tables<T> tb;
  tb.build(*prm);
#ifdef _OPENMP
  if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
#pragma omp parallel for schedule(dynamic, 1)
  for (int64_t c = 0; c < n; ++c) {
    T go, dgo;
    int32_t fl;
    T scl = ts_scale ? T(ts_scale[c]) : T(prm->j0z[sv[c] - 1]) / T(rD[c]);
    eval_point_dz<T>(*prm, tb, T(tD[c]), sv[c], T(rD[c]), scl, T(zD[c]), dz_layer(zD[c], *prm), &go, &dgo, &fl);
    gz[c] = (double)go;
    dgz[c] = (double)dgo;
    if (flags) flags[c] = fl;
  }
  return 0;
}

template <class T>
void soln_dz_t(const params *prm, double a, double rD, double tD, double zD, int lay, double *out) {
  std::vector<cx<T>> p, lt, fp;
  dehoog_pvalues<T>(T(prm->tee_mult) * T(tD), *prm, p);
  lap_time<T>(*prm, p, lt);
  lap_hank_soln_dz<T>(T(a), T(rD), p, T(zD), lay > 0 ? lay : dz_layer(zD, *prm), *prm, lt, fp);
  for (size_t i = 0; i < fp.size(); ++i) { out[2 * i] = (double)fp[i].re; out[2 * i + 1] = (double)fp[i].im; }
}

// lap_hank_soln itself at one z of layer `lay`, in T (oracle.soln is double only)
template <class T>
void soln_value_t(const params *prm, double a, double rD, double tD, double zD, int lay, double *out) {
  std::vector<cx<T>> p, lt, fp;
  dehoog_pvalues<T>(T(prm->tee_mult) * T(tD), *prm, p);
  lap_time<T>(*prm, p, lt);
  soln_ws<T> ws;
  const T z = T(zD);
  lap_hank_soln<T>(T(a), T(rD), p, &z, &lay, 1, *prm, lt, ws, fp);
  for (size_t i = 0; i < fp.size(); ++i) { out[2 * i] = (double)fp[i].re; out[2 * i + 1] = (double)fp[i].im; }
}

}  // namespace

extern "C" {

// ulps = 0 disables; see oracle_math.hpp (jitter)
void orcd_set_jitter(double ulps, unsigned long long seed) {
  jitter().ulps = ulps;
  jitter().seed = seed;
}

// vertical gradient at points (unc_eval_points_dz's definition): gz, dgz per point, layers
// geometric; returns 1 if a zD is not in [0, 1]
int orc_eval_points_dz(const params *prm, int64_t n, const double *tD, const int32_t *sv, const double *rD,
                       const double *zD, const double *ts_scale, int nthreads, double *gz, double *dgz,
                       int32_t *flags) {
  return eval_points_dz_t<double>(prm, n, tD, sv, rD, zD, ts_scale, nthreads, gz, dgz, flags);
}

int orc_eval_points_dz_ld(const params *prm, int64_t n, const double *tD, const int32_t *sv, const double *rD,
                          const double *zD, const double *ts_scale, int nthreads, double *gz, double *dgz,
                          int32_t *flags) {
  return eval_points_dz_t<long double>(prm, n, tD, sv, rD, zD, ts_scale, nthreads, gz, dgz, flags);
}

// the z-derivative of lap_hank_soln at one abscissa for the p-vector of time tD; out[p*2 + {0,1}].
// lay = 1..3 selects the layer's formula; lay = 0 takes the geometric layer of zD.
void orc_soln_dz(const params *prm, double a, double rD, double tD, double zD, int lay, double *out) {
  soln_dz_t<double>(prm, a, rD, tD, zD, lay, out);
}

void orc_soln_dz_ld(const params *prm, double a, double rD, double tD, double zD, int lay, double *out) {
  soln_dz_t<long double>(prm, a, rD, tD, zD, lay, out);
}

// the point integrand lap_hank_soln at (zD, layer lay) in double or long double, so that the
// derivative can be checked against values of the same precision
void orc_soln_value(const params *prm, double a, double rD, double tD, double zD, int lay, double *out) {
  soln_value_t<double>(prm, a, rD, tD, zD, lay, out);
}

void orc_soln_value_ld(const params *prm, double a, double rD, double tD, double zD, int lay, double *out) {
  soln_value_t<long double>(prm, a, rD, tD, zD, lay, out);
}

}  // extern "C"
