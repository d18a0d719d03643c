// TEST INFRASTRUCTURE ONLY -- CPU oracle of the vertical drawdown gradient (the product's
// unc_eval_points_dz; PARITY UNPINNED as the rest of the oracle, see oracle_math.hpp).  Builds on
// the point restatement of oracle_core.hpp, which it leaves as it is.
#pragma once
#include "oracle_core.hpp"

namespace orc {

// ---------------------------------------------------------------------------
// Vertical gradient gz = d s_D / d z_D (the product's unc_eval_points_dz; no reference equivalent).
// The point algorithm with lap_hank_soln replaced by its z-derivative, in the operation order
// of the reference's expressions (laplace_hankel_solutions.f90:30-202):
//   cosh(eta z) -> eta sinh(eta z),  cosh(eta(c-z)) -> -eta sinh(eta(c-z)),
//   exp(eta(z-1)) -> eta exp(eta(z-1)),  constant terms -> 0.
// Layers are geometric: 1 if z < 1-lD, otherwise 2 if z < 1-dD, otherwise 3.
inline int dz_layer(double z, const params &prm) {
  if (z < 1.0 - prm.lD) return 1;
  if (z < 1.0 - prm.dD) return 2;
  return 3;
}

// d/dz of hantush's layer function of `lay` (:175-198), without theis/bD
template <class T>
cx<T> hantush_dz(cx<T> eta, T z, int lay, const params &prm) {
  const T dD1 = T(1) - T(prm.dD), lD1 = T(1) - T(prm.lD);
  cx<T> ff1 = csinh(eta * T(prm.dD));
  cx<T> ff2 = csinh(eta * lD1);
  cx<T> sh = csinh(eta);
  if (lay == 1) {
    cx<T> g3 = cexp((-eta) * lD1) - (ff1 + cexp(-eta) * ff2) / sh;
    return g3 * (eta * csinh(eta * z));
  }
  cx<T> g2 = (ff1 * (eta * csinh(eta * z)) + ff2 * ((-eta) * csinh(eta * (T(1) - z)))) / sh;
  if (lay == 2) return T(0) - g2;
  return (-eta) * csinh(eta * (dD1 - z)) - g2;
}

// z-derivative of lap_hank_soln for ONE z: fp[p] (common factor :118 included)
template <class T>
void lap_hank_soln_dz(T a, T rD, const std::vector<cx<T>> &p, T z, int lay, const params &prm,
                      const std::vector<cx<T>> &lt, std::vector<cx<T>> &fp) {
  const int np = (int)p.size();
  fp.resize(np);
  const int model = prm.model;
  for (int k = 0; k < np; ++k) {
    if (model == 0) {          // no z dependence
      fp[k] = cx<T>(0, 0);
      continue;
    }
    const cx<T> eta = csqrt((p[k] + a * a) / T(prm.kappa));
    cx<T> v;
    if (model == 1) {
      v = hantush_dz(eta, z, lay, prm) * theis(a, p[k]) / T(prm.bD);
    } else if (model == 2) {
      // uDf of hantushstorage (:253-266), double precision as the Amos routine
      const double PI = consts<double>::pi();
      const double CDw = prm.rDw * prm.rDw / (2.0 * (prm.l - prm.d) * prm.Ss);
      const double tDb = PI * prm.rDwobs * prm.rDwobs / (prm.sF * prm.Ss);
      const cx<double> pd((double)p[k].re, (double)p[k].im);
      const double ad = (double)a;
      cx<double> xi = prm.rDw * csqrt(pd);
      cx<double> K[2];
      int nzero;
      cbesk01(xi, K, &nzero);
      cx<double> A0 = 2.0 / (pd * CDw * K[0] + xi * K[1]);
      cx<double> uDf = A0 / ((pd + ad * ad) * (pd * tDb + 1.0));
      const cx<T> uDfT(T(uDf.re), T(uDf.im));
      v = (uDfT / T(prm.bD)) * hantush_dz(eta, z, lay, prm);
    } else if (model == 6) {
      const T beta0 = T(prm.mn_ak) * T(prm.mn_b);
      const T phiDa = T(prm.mn_psia) / T(prm.mn_b);
      const T phiDk = T(prm.mn_psik) / T(prm.mn_b);
      const T vartheta = beta0 * T(prm.mn_Sy) / (T(prm.Ss) * T(prm.mn_b)) * std::exp(-beta0 * (phiDa - phiDk));
      const T u0 = beta0 / T(2);
      cx<T> eta1 = csqrt((p[k] * vartheta + a * a) / T(prm.kappa));
      cx<T> q = eta1 / u0;
      cx<T> vv = csqrt(T(1) + q * q);
      cx<T> u = u0 * (T(1) - vv);
      cx<T> etasq = (p[k] + a * a) / T(prm.kappa);
      cx<T> Delta0 = eta * csinh(eta) - u * ccosh(eta);
      cx<T> pre = T(2) / (T(prm.kappa) * etasq);
      cx<T> ud = u / Delta0;
      v = pre * (T(0) + ud * (eta * csinh(eta * z)));
    } else {
      // models 3..5 (:64-93); top = udp at zD = 1 (layer 3) does not depend on z
      const T MAXEXP = consts<T>::maxexp();
      const cx<T> th = theis(a, p[k]);
      cx<T> udp, top;
      if (model == 4) {
        udp = cx<T>(0, 0);
        top = th;
      } else {
        udp = hantush_dz(eta, z, lay, prm) * th / T(prm.bD);
        const T one(1);
        const int three = 3;
        std::vector<cx<T>> ut;
        hantush(a, &one, &three, 1, std::vector<cx<T>>(1, p[k]), prm, ut);
        top = ut[0];
      }
      cx<T> xi = eta * T(prm.alphaD) / p[k];
      if (model == 3) {
        cx<T> s(0, 0);
        for (int mm = 0; mm < prm.moench_M; ++mm)
          s = s + T(1) / (T(1) + p[k] * (T(1) / T(prm.moench_gamma[mm])));
        xi = xi * T(prm.moench_M) / s;
      }
      if (eta.re < MAXEXP) {
        cx<T> den = (T(1) + T(prm.beta) * eta * xi) * ccosh(eta) + xi * csinh(eta);
        v = udp - top * (eta * csinh(eta * z)) / den;
      } else {
        cx<T> den = T(1) + T(prm.beta) * eta * xi + xi;
        v = udp - top * (eta * cexp(eta * (z - T(1)))) / den;
      }
    }
    fp[k] = v;
  }
  T aj = a * lm<T>::j0(a * rD);
  for (int k = 0; k < np; ++k) fp[k] = aj * fp[k] * lt[k];
}

// eval_column for ONE point with the z-derivative integrand (no carry between points: a stale
// infint is 0 and flagged)
template <class T>
void eval_point_dz(const params &prm, const tables<T> &tb, T tD, int sv, T rD, T ts_scale, T z, int lay,
                   T *gz_out, T *dgz_out, int32_t *flag) {
  const int np = tb.np, N = tb.N, R = tb.R, G = tb.G, nacc = tb.nacc;
  const T tee = T(prm.tee_mult) * tD;
  std::vector<cx<T>> p, lt;
  dehoog_pvalues<T>(tee, prm, p);
  lap_time<T>(prm, p, lt);
  std::vector<T> j0z(prm.n_j0z);
  for (int i = 0; i < prm.n_j0z; ++i) j0z[i] = T(prm.j0z[i]);
  const T arg = j0z[sv - 1] / rD;  // driver.f90:120
  std::vector<T> a;
  {
    std::vector<T> wtmp;
    tanh_sinh_setup<T>(prm.ts_k, ts_scale, wtmp, &a);
  }
  std::vector<cx<T>> fa((size_t)N * np), fp;
  for (int nn = 0; nn < N; ++nn) {
    lap_hank_soln_dz<T>(a[nn], rD, p, z, lay, prm, lt, fp);
    std::copy(fp.begin(), fp.end(), fa.begin() + (size_t)nn * np);
  }
  std::vector<cx<T>> finint(np), tmp(R);
  for (int k = 0; k < np; ++k) {
    for (int j = 1; j <= R; ++j) {
      const int step = 1 << (R - j);
      cx<T> sum(0, 0);
      for (int m = 1; m <= tb.Nv[j - 1]; ++m) sum = sum + tb.tsw[j - 1][m - 1] * fa[(size_t)(m * step - 1) * np + k];
      tmp[j - 1] = (arg / T(2)) * sum;
    }
    finint[k] = (R > 1) ? extraptozero<T>(tb.hv.data(), tmp.data(), R) : tmp[0];
  }
  std::vector<cx<T>> GLarea((size_t)nacc * np), GLz((size_t)G * np);
  for (int j = sv + 1; j <= sv + nacc; ++j) {
    const T lob = j0z[j - 2] / rD, hib = j0z[j - 1] / rD;
    const T width = hib - lob;
    for (int m = 0; m < G; ++m) {
      const T y = std::fma(width, tb.glx[m], hib + lob) / T(2);
      lap_hank_soln_dz<T>(y, rD, p, z, lay, prm, lt, fp);
      std::copy(fp.begin(), fp.end(), GLz.begin() + (size_t)m * np);
    }
    for (int k = 0; k < np; ++k) {
      cx<T> acc(0, 0);
      for (int m = 0; m < G; ++m) acc = acc + GLz[(size_t)m * np + k] * tb.glw[m];
      GLarea[(size_t)(j - sv - 1) * np + k] = (width / T(2)) * acc;
    }
  }
  std::vector<cx<T>> series(nacc), col(np);
  *flag = 0;
  for (int k = 0; k < np; ++k) {
    bool any = false;
    for (int j = 0; j < nacc; ++j) {
      series[j] = GLarea[(size_t)j * np + k];
      if (cabs(series[j]) > T(0)) any = true;
    }
    cx<T> infint(0, 0);
    if (any) infint = wynn_epsilon<T>(series.data(), nacc);
    else *flag |= 1;
    col[k] = finint[k] + infint;
  }
  *gz_out = dehoog_invlap<T>(tD, tee, col.data(), prm);
  for (int k = 0; k < np; ++k) col[k] = col[k] * p[k];
  *dgz_out = dehoog_invlap<T>(tD, tee, col.data(), prm) * tD;
}

}  // namespace orc
