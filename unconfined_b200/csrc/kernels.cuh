// sm_100a kernels for the Laplace-Hankel drawdown hot path (driver.f90:100-231 of the
// reference behind one launch).  FP64 CUDA-core work: no tensor cores (not a dense
// contraction), HBM traffic is ~40 B per point against ~1e7 FLOP, so the bound is the
// FP64 pipe.  See DESIGN.md for the layout; in short, per CTA = one (t,r) column and
// a tile of ZT z-values:
//   prologue  threads build the per-p tables (de Hoog p, lapTime, Moench / storage
//             factors) and the per-abscissa tables (a^2 and weight*a*J0(a rD)) in
//             shared memory;
//   phase A   one warp per p: lanes split the tanh-sinh nodes (Richardson folded into
//             one weight per node) and the Gauss-Lobatto nodes (contiguous blocks so a
//             lane touches at most two J0 intervals); partial sums are reduced with
//             warp shuffles;
//   phase B   one thread per (p,z): Wynn-epsilon on the interval areas;
//   phase C   one warp per (z, value|derivative): de Hoog q-d + continued fraction.
#pragma once
#include <cstdint>
#include "cmath.cuh"

#include "params.cuh"
#include "fast.cuh"
#include "wynn.cuh"
namespace unc {

// ---------------------------------------------------------------------------
// time.f90:34-124  lapTime(p) for one p (all behaviours; literal operation order)
__device__ __noinline__ cplx laptime_dev(const DevParams &P, cplx p) {
  const double *par = P.time_par;  // par[i-1] = timePar(i)
  const int tt = P.time_type;
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  if (tt == 1) return cexp_g((-par[0]) * p) / p;
  if (tt == 2) return cexp_g((-par[0]) * p) / p - cexp_g((-par[1]) * p) / p;
  if (tt == 3) return cexp_g((-par[0]) * p);
  if (tt == 4) return 1.0 / (p - p * cexp_g((-par[0]) * p)) * (1.0 - cexp_g((-par[1]) * p)) / p;
  if (tt == 5) return cexp_g((-par[1]) * p) / (p + p * cexp_g((-par[0]) * p));
  if (tt == 6) return cexp_g((-par[1]) * p) * p / (p * p + par[0] * par[0]);
  if (tt == 7) {
    // numerator is exp(x)-exp(x) as written in the reference (time.f90:72-74)
    cplx e1 = cexp_g(par[0] * p);
    return cexp_g((-par[1]) * p) / (p * p) * (e1 - e1) / (e1 + e1);
  }
  if (tt == 8) {
    cplx eh = cexp_g((-par[0]) * p / 2.0);
    return cexp_g((-par[1]) * p) * (1.0 - eh) / ((1.0 + eh) * p);
  }
  if (tt < 0 && tt >= -100) {
    const int n = -tt;
    const double tf = par[n];
    cplx s = mk(0.0, 0.0);
    double sq = 0.0, qprev = 0.0;
    for (int i = 1; i <= n; ++i) {
      double q = par[n + i];
      s = s + (q - qprev) * cexp_g((-par[i - 1]) * p);
      sq += q - qprev;
      qprev = q;
    }
    return (s - sq * cexp_g((-tf) * p)) / p;
  }
  if (tt <= -101) {
    const int n = -tt - 100;
    const double tf = par[n];
    cplx s = mk(0.0, 0.0);
    double sw = 0.0, wprev = 0.0;
    for (int i = 1; i <= n; ++i) {
      double ti = par[i - 1];
      double tnext = (i < n) ? par[i] : tf;
      double yi = par[n + i];
      double ynext = (i < n) ? par[n + i + 1] : 0.0;  // y(n+1) is out of bounds in the reference
      double W = (ynext - yi) / (tnext - ti);
      s = s + (W - wprev) * cexp_g((-ti) * p);
      sw += W - wprev;
      wprev = W;
    }
    return (s - sw * cexp_g((-tf) * p)) / (p * p);
  }
  return mk(nan, nan);
}

// ---------------------------------------------------------------------------
// cbessel.f90:877-1146 (cbesk) -> 5036-5495 (cbknu) for fnu=0, kode=1, n=2, Re z >= 0.
// K[0]=K0(z), K[1]=K1(z).  Out-of-range arguments give NaN (the reference prints ierr
// and carries on with whatever cy holds, laplace_hankel_solutions.f90:259-262).  Re z > alim
// takes the exp(-z) underflow branch (cbessel.f90:5215 -> 200 :5482, 190 :5458-5476, ckscl
// :5499-5611, cuchk :5895-5927): members that underflow come back as exact zeros.
__device__ __noinline__ void cbesk01_dev(cplx z, cplx *K) {
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  const double tol = 2.220446049250313e-16;
  const double r1m5 = 0.30102999566398120;  // log10(2)
  const double elim = 2.303 * (1021 * r1m5 - 3.0);
  const double alim = elim + fmax(-(r1m5 * 52) * 2.303, -41.45);
  const double pi = 3.141592653589793, hpi = 1.5707963267948966;
  const double rthpi = 1.2533141373155001;   // sqrt(8 atan 1)/2
  const double spi = 1.9098593171027440;     // 3/(2 atan 1)
  const double fpi = 1.89769999331517738, tth = 6.66666666666666666e-01;
  const double xx = z.re, yy = z.im;
  const double caz = hypot(xx, yy);
  K[0] = mk(nan, nan); K[1] = mk(nan, nan);
  if (!(caz <= fmin(0.5 / tol, 2147483647.0 * 0.5)) || !(caz >= DBL_MIN * 1.0e3) || !(xx >= 0.0)) return;
  const cplx rz = mk(2.0, 0.0) / z;
  cplx s1, s2;
  double csr = 1.0;
  bool iflag = false;
  if (caz <= 2.0) {
    // power series, cbessel.f90:5098-5200 with dnu=0: fc=1, t1=t2=1, g1=-cc(1), g2=1
    cplx smu = clog_g(rz);
    cplx f = mk(-5.77215664901532861e-01, 0.0) + smu;  // g1*cch + smu*g2, cch=(1,0)
    cplx p = mk(0.5, 0.0), q = mk(0.5, 0.0);
    s1 = f;
    s2 = p;
    double ak = 1.0, a1 = 1.0, bk = 1.0;
    cplx ck = mk(1.0, 0.0);
    if (caz >= tol) {
      cplx cz = z * z * 0.25;
      double t1 = 0.25 * caz * caz;
      do {
        f = (f * ak + p + q) / bk;
        p = p / ak;
        q = q / ak;
        double rk = 1.0 / ak;
        ck = ck * cz * rk;
        s1 = s1 + ck * f;
        s2 = s2 + ck * (p - f * ak);
        a1 = a1 * t1 * rk;
        bk = bk + ak + ak + 1.0;
        ak = ak + 1.0;
      } while (a1 > tol);
    }
    double css = 1.0;
    if (fabs(smu.re) > alim) { css = tol; csr = 1.0 / tol; }  // kflag=3
    cplx p2 = s2 * mk(css, 0.0);
    s2 = p2 * rz;
    s1 = s1 * mk(css, 0.0);
  } else {
    // Miller backward recurrence, cbessel.f90:5209-5327
    iflag = xx > alim;      // koded = 2: the values stay scaled by exp(z) until ckscl
    cplx coef = mk(rthpi, 0.0) / csqrt_g(z);
    if (!iflag) {
      double a1 = exp(-xx);
      cplx pt = a1 * mk(cos(yy), -sin(yy));
      coef = coef * pt;
    }
    double ak = 1.0;  // |cos(pi*dnu)|
    double fhs = 0.25;
    double t1 = 52 * r1m5 * 3.321928094;
    t1 = fmin(fmax(t1, 12.0), 60.0);
    double t2 = tth * t1 - 6.0;
    if (fabs(xx) * 2.0 < DBL_MIN) t1 = hpi;
    else t1 = fabs(atan(yy / xx));
    double fk;
    if (t2 <= caz) {
      double etest = ak / (pi * caz * tol);
      fk = 1.0;
      if (!(etest < 1.0)) {
        double fks = 2.0, rk = caz + caz + 2.0, a1 = 0.0, a2 = 1.0;
        bool found = false;
        for (int i = 1; i <= 30; ++i) {
          ak = fhs / fks;
          double bk = rk / (fk + 1.0);
          double tm = a2;
          a2 = bk * a2 - ak * a1;
          a1 = tm;
          rk = rk + 2.0;
          fks = fks + fk + fk + 2.0;
          fhs = fhs + fk + fk;
          fk = fk + 1.0;
          tm = fabs(a2) * fk;
          if (etest < tm) { found = true; break; }
        }
        if (!found) return;
        fk = fk + spi * t1 * sqrt(t2 / caz);
        fhs = 0.25;
      }
    } else {
      double a2 = sqrt(caz);
      ak = fpi * ak / (tol * sqrt(a2));
      double aa = 3.0 * t1 / (1.0 + caz);
      double bb = 14.7 * t1 / (28.0 + caz);
      ak = (log(ak) + caz * cos(aa) / (1.0 + 0.008 * caz)) / cos(bb);
      fk = 0.12125 * ak * ak / caz + 1.5;
    }
    int k = (int)fk;
    fk = k;
    double fks = fk * fk;
    cplx p1 = mk(0.0, 0.0), p2 = mk(tol, 0.0), cs = p2;
    for (int i = 1; i <= k; ++i) {
      double a1 = fks - fk;
      double a2 = (fks + fk) / (a1 + fhs);
      double rk = 2.0 / (fk + 1.0);
      double tt1 = (fk + xx) * rk;
      double tt2 = yy * rk;
      cplx pt = p2;
      p2 = (p2 * mk(tt1, tt2) - p1) * a2;
      p1 = pt;
      cs = cs + p2;
      fks = a1 - fk + 1.0;
      fk = fk - 1.0;
    }
    double tm = cabs_d(cs);
    cplx pt = mk(1.0 / tm, 0.0);
    s1 = pt * p2;
    cs = conj(cs) * pt;
    s1 = coef * s1 * cs;
    tm = cabs_d(p2);
    pt = mk(1.0 / tm, 0.0);
    p1 = pt * p1;
    p2 = conj(p2) * pt;
    pt = p1 * p2;
    s2 = s1 * (mk(1.0, 0.0) + (mk(0.5, 0.0) - pt) / z);
  }
  if (iflag) {
    // ckscl with zd = z, n = 2, ascle = bry(1) = 1e3*tiny/tol; survivors unscaled by csr(1) = tol
    const double ascle = 1.0e3 * DBL_MIN / tol;
    cplx y[2] = {s1, s2};
    int nz = 0, ic = 0;
#pragma unroll
    for (int i = 1; i <= 2; ++i) {
      const cplx sv = y[i - 1];
      const double as = cabs_d(sv);
      const double acs = -xx + log(as);
      nz += 1;
      y[i - 1] = mk(0.0, 0.0);
      if (acs >= -elim) {
        cplx cs = (-z) + clog_g(sv);
        const double aa2 = exp(cs.re) / tol;
        cs = aa2 * mk(cos(cs.im), sin(cs.im));
        int nw = 0;
        const double yr = fabs(cs.re), yi = fabs(cs.im);
        double st = fmin(yr, yi);
        if (!(st > ascle)) {
          const double ss = fmax(yr, yi);
          st = st / tol;
          if (ss < st) nw = 1;
        }
        if (nw == 0) { y[i - 1] = cs; nz -= 1; ic = i; }
      }
    }
    if (ic <= 1) { y[0] = mk(0.0, 0.0); nz = 2; }
    K[0] = mk(0.0, 0.0); K[1] = mk(0.0, 0.0);
    if (nz == 0) { K[0] = y[0] * mk(tol, 0.0); K[1] = y[1] * mk(tol, 0.0); }
    else if (nz == 1) K[1] = y[1] * mk(tol, 0.0);
    return;
  }
  K[0] = s1 * mk(csr, 0.0);
  K[1] = s2 * mk(csr, 0.0);
}

// ---------------------------------------------------------------------------
// Per-p shared tables
struct PTab {
  cplx *p;    // de Hoog abscissae (invlap.f90:166-170)
  cplx *lt;   // lapTime(p)
  cplx *aux;  // model 3: sum_m 1/(1+p/gamma_m); model 2: uDf numerator A0/(p*tDb+1) parts
  cplx *aux2; // model 2: (p*tDb + 1)
};

// laplace_hankel_solutions.f90:133-202 (hantush) for one (a,p) and a tile of z;
// also the layer-3 value at zD=1 when want_top (called from models 3/5, :81,162-170).
// Literal operation order; u[] excludes nothing: it is udp*theis/bD.
template <int ZT>
__device__ __forceinline__ void hantush_literal(const DevParams &P, double a2, cplx p, cplx eta,
                                                const double *z, const int *lay, int nzt,
                                                bool want_top, cplx *u, cplx *utop,
                                                bool storage_variant) {
  const cplx ff1 = csinh_g(eta * P.dD);
  const cplx ff2 = csinh_g(eta * P.lD1);
  const cplx sh = csinh_g(eta);
  bool any1 = false;
#pragma unroll
  for (int i = 0; i < ZT; ++i) if (i < nzt && lay[i] == 1) any1 = true;
  cplx g3 = mk(0.0, 0.0);
  if (any1) g3 = cexp_g((-eta) * P.lD1) - (ff1 + cexp_g(-eta) * ff2) / sh;
  const cplx th = 2.0 / (p + a2);
#pragma unroll
  for (int i = 0; i < ZT; ++i) {
    if (i < nzt) {
      cplx v;
      if (lay[i] == 1) {
        v = g3 * ccosh_g(eta * z[i]);
      } else {
        cplx g2 = (ff1 * ccosh_g(eta * z[i]) + ff2 * ccosh_g(eta * (1.0 - z[i]))) / sh;
        if (lay[i] == 2) v = 1.0 - g2;
        else v = ccosh_g(eta * (P.dD1 - z[i])) - g2;
      }
      u[i] = storage_variant ? v : v * th / P.bD;
    }
  }
  if (want_top) {
    cplx g1 = ccosh_g(eta * (P.dD1 - 1.0));
    cplx g2 = (ff1 * ccosh_g(eta * 1.0) + ff2 * ccosh_g(eta * (1.0 - 1.0))) / sh;
    *utop = (g1 - g2) * th / P.bD;
  }
}

// laplace_hankel_solutions.f90:30-116: fp(p, z-tile) at one abscissa, WITHOUT the common
// factor a*J0(a rD)*lapTime(p) of :118 (folded into the quadrature weight / applied per p).
template <int ZT>
__device__ __forceinline__ void soln_literal(const DevParams &P, const PTab &T, int pi, double a2,
                                             const double *z, const int *lay, int nzt, cplx *f) {
  const cplx p = T.p[pi];
  const int model = P.model;
  if (model == 0) {
    cplx th = 2.0 / (p + a2);
#pragma unroll
    for (int i = 0; i < ZT; ++i) f[i] = th;
    return;
  }
  const cplx eta = csqrt_g((p + a2) / P.kappa);
  if (model == 6) {
    // laplace_hankel_solutions.f90:404-442  mishraNeumanMalama (MNtype 1)
    const cplx eta1 = csqrt_g((p * P.mn_vartheta + a2) / P.kappa);
    const cplx q = eta1 / P.mn_u0;
    const cplx v = csqrt_g(1.0 + q * q);
    const cplx u = P.mn_u0 * (1.0 - v);
    const cplx etasq = (p + a2) / P.kappa;
    const cplx Delta0 = eta * csinh_g(eta) - u * ccosh_g(eta);
    const cplx pre = 2.0 / (P.kappa * etasq);
    const cplx ud = u / Delta0;
#pragma unroll
    for (int i = 0; i < ZT; ++i)
      if (i < nzt) f[i] = pre * (1.0 + ud * ccosh_g(eta * z[i]));
    return;
  }
  if (model == 1) {
    cplx dummy;
    hantush_literal<ZT>(P, a2, p, eta, z, lay, nzt, false, f, &dummy, false);
    return;
  }
  if (model == 2) {
    // :204-301  u = (uDf/bD)*uDp,  uDf = A0/((p+a^2)*(p*tDb+1))
    cplx dummy, uDp[ZT];
    hantush_literal<ZT>(P, a2, p, eta, z, lay, nzt, false, uDp, &dummy, true);
    cplx uDf = T.aux[pi] / ((p + a2) * T.aux2[pi]);
    cplx pre = uDf / P.bD;
#pragma unroll
    for (int i = 0; i < ZT; ++i) if (i < nzt) f[i] = pre * uDp[i];
    return;
  }
  // models 3,4,5  (:64-93)
  cplx xi = eta * P.alphaD / p;
  if (model == 3) xi = xi * (double)P.moench_M / T.aux[pi];
  cplx udp[ZT], top;
  if (model == 4) {
    cplx th = 2.0 / (p + a2);
#pragma unroll
    for (int i = 0; i < ZT; ++i) udp[i] = th;
    top = th;
  } else {
    hantush_literal<ZT>(P, a2, p, eta, z, lay, nzt, true, udp, &top, false);
  }
  const double MAXEXP = 12.014551129705717;  // -log(epsilon(1d0))/3  (constants.f90:66)
  if (eta.re < MAXEXP) {
    cplx den = (1.0 + P.beta * eta * xi) * ccosh_g(eta) + xi * csinh_g(eta);
#pragma unroll
    for (int i = 0; i < ZT; ++i)
      if (i < nzt) f[i] = udp[i] - top * ccosh_g(eta * z[i]) / den;
  } else {
    cplx den = 1.0 + P.beta * eta * xi + xi;
#pragma unroll
    for (int i = 0; i < ZT; ++i)
      if (i < nzt) f[i] = udp[i] - top * cexp_g(eta * (z[i] - 1.0)) / den;
  }
}

// Far beyond the overflow threshold the literal formulas need not be executed to know their
// value.  hantush (laplace_hankel_solutions.f90:176-198) divides by sinh(eta) in every layer
// (g2 :179-180, g3 :183-184).  For Re(eta) >= 800 glibc's csinh returns (+-Inf, +-Inf): its
// components are e^709/2 * e^(Re eta - 709) * {cos, sin}(Im eta), which overflow unless
// |cos| or |sin| < 1.3e-39, impossible for a non-zero double |Im eta| < 2e5 other than a
// denormal-small one; between 718 and 800 the same is established from the actual sine and
// cosine (below).  GCC's Fortran-rules (Smith) division by a divisor whose two
// components are infinite forms ratio = Inf/Inf = NaN and returns (NaN, NaN) whatever the
// numerator is, and NaN survives every later product and sum of models 1, 2, 3 and 5
// (:200, :299, :84-92).  Re(eta) in (fast-path bound, 718) still takes the literal path, and so
// does the real Laplace parameter p_0 (Im eta = 0: sinh(eta) = (Inf, 0) there).
__device__ __forceinline__ bool literal_is_nan(const DevParams &P, cplx eta) {
  const int m = P.model;
  if (!((m == 1 || m == 2 || m == 3 || m == 5) && eta.re >= 718.0 && fabs(eta.im) < 2.0e5)) return false;
  if (eta.re >= 800.0) return fabs(eta.im) > 1e-30;
  // closer to the threshold the overflow of BOTH components is checked on the actual phase:
  // |component| = e^709.78 * e^(Re eta - 709.78)/2 * |cos or sin|, so Re eta >= 718 (e^8.2/2 = 1.8e3)
  // overflows whenever |cos|, |sin| > 1e-3; Re eta >= 745 (e^35/2 = 8e14) whenever they exceed 1e-10
  double sn, cs;
  sincos_q(eta.im, &sn, &cs);
  const double mn = fmin(fabs(sn), fabs(cs));
  return mn > 1e-3 || (eta.re >= 745.0 && mn > 1e-10);
}

// Literal evaluation for ONE z (slow path of the fast kernels: Re(eta) beyond the
// fast-path bound, where the reference's overflow behaviour is part of the contract).
__device__ __noinline__ cplx soln_literal_one(const DevParams &P, const PTab &T, int pi, double a2,
                                              double z, int lay) {
  cplx f[1];
  soln_literal<1>(P, T, pi, a2, &z, &lay, 1, f);
  return f[0];
}

// ---------------------------------------------------------------------------
// Literal screen means (slow path of lh_screen_kernel).  The operation sequence of
// hantush_literal / soln_literal for ONE z, evaluated at the segment midpoint m with every
// z-dependent factor (cosh(eta z), cosh(eta(1-z)), cosh(eta(dD1-z)), exp(eta(z-1))) multiplied
// by S = csinh(eta h)/(eta h); constant terms unchanged.  Every Hantush-type layer function
// still divides by sinh(eta), so literal_is_nan applies unchanged.
__device__ __forceinline__ cplx sinhc_lit(cplx x) {
  if (x.re == 0.0 && x.im == 0.0) return mk(1.0, 0.0);
  return csinh_g(x) / x;
}

__device__ __forceinline__ cplx hantush_literal_mean(const DevParams &P, double a2, cplx p, cplx eta, double m,
                                                     cplx S, int lay, bool storage_variant) {
  const cplx ff1 = csinh_g(eta * P.dD);
  const cplx ff2 = csinh_g(eta * P.lD1);
  const cplx sh = csinh_g(eta);
  const cplx th = 2.0 / (p + a2);
  cplx v;
  if (lay == 1) {
    const cplx g3 = cexp_g((-eta) * P.lD1) - (ff1 + cexp_g(-eta) * ff2) / sh;
    v = g3 * (ccosh_g(eta * m) * S);
  } else {
    const cplx g2 = (ff1 * (ccosh_g(eta * m) * S) + ff2 * (ccosh_g(eta * (1.0 - m)) * S)) / sh;
    if (lay == 2) v = 1.0 - g2;
    else v = ccosh_g(eta * (P.dD1 - m)) * S - g2;
  }
  return storage_variant ? v : v * th / P.bD;
}

// mean over the segment [m-h, m+h] of layer `lay` of fp(p) at one abscissa, without the common
// factor a*J0(a rD)*lapTime(p) (as soln_literal)
__device__ __noinline__ cplx soln_literal_mean(const DevParams &P, const PTab &T, int pi, double a2, double m,
                                               double h, int lay) {
  const cplx p = T.p[pi];
  const int model = P.model;
  if (model == 0) return 2.0 / (p + a2);
  const cplx eta = csqrt_g((p + a2) / P.kappa);
  const cplx S = sinhc_lit(eta * h);
  if (model == 6) {
    const cplx eta1 = csqrt_g((p * P.mn_vartheta + a2) / P.kappa);
    const cplx q = eta1 / P.mn_u0;
    const cplx v = csqrt_g(1.0 + q * q);
    const cplx u = P.mn_u0 * (1.0 - v);
    const cplx etasq = (p + a2) / P.kappa;
    const cplx Delta0 = eta * csinh_g(eta) - u * ccosh_g(eta);
    const cplx pre = 2.0 / (P.kappa * etasq);
    const cplx ud = u / Delta0;
    return pre * (1.0 + ud * (ccosh_g(eta * m) * S));
  }
  if (model == 1) return hantush_literal_mean(P, a2, p, eta, m, S, lay, false);
  if (model == 2) {
    const cplx uDp = hantush_literal_mean(P, a2, p, eta, m, S, lay, true);
    const cplx uDf = T.aux[pi] / ((p + a2) * T.aux2[pi]);
    return uDf / P.bD * uDp;
  }
  // models 3,4,5: the water-table term's factor at zD = 1 (top) is a constant of the segment
  cplx xi = eta * P.alphaD / p;
  if (model == 3) xi = xi * (double)P.moench_M / T.aux[pi];
  cplx udp, top;
  if (model == 4) {
    udp = 2.0 / (p + a2);
    top = udp;
  } else {
    udp = hantush_literal_mean(P, a2, p, eta, m, S, lay, false);
    cplx unused;
    hantush_literal<1>(P, a2, p, eta, &m, &lay, 0, true, &unused, &top, false);
  }
  const double MAXEXP = 12.014551129705717;  // -log(epsilon(1d0))/3  (constants.f90:66)
  if (eta.re < MAXEXP) {
    const cplx den = (1.0 + P.beta * eta * xi) * ccosh_g(eta) + xi * csinh_g(eta);
    return udp - top * (ccosh_g(eta * m) * S) / den;
  }
  const cplx den = 1.0 + P.beta * eta * xi + xi;
  return udp - top * (cexp_g(eta * (m - 1.0)) * S) / den;
}

// screen mean = sum_i w_i mean_i (weights applied componentwise: no real->complex promotion,
// so an infinite segment mean stays (Inf, x) as the point path's value would)
__device__ __noinline__ cplx screen_literal(const DevParams &P, const PTab &T, int pi, double a2,
                                            const ScreenSegs *sg) {
  cplx f = mk(0.0, 0.0);
  for (int i = 0; i < sg->n; ++i) {
    const cplx v = soln_literal_mean(P, T, pi, a2, sg->m[i], sg->h[i], sg->L[i] + 1);
    const cplx wv = mk(sg->w[i] * v.re, sg->w[i] * v.im);
    f = (i == 0) ? wv : f + wv;
  }
  return f;
}

// ---------------------------------------------------------------------------
// Literal vertical gradient (slow path of lh_dz_kernel): the z-derivative of hantush_literal /
// soln_literal for ONE z in their operation order.  cosh(eta z) -> eta sinh(eta z),
// cosh(eta(c-z)) -> -eta sinh(eta(c-z)), exp(eta(z-1)) -> eta exp(eta(z-1)); constant terms
// (the 1 of layer 2, udp of model 4, the 1 of model 6) become 0.  Every Hantush-type layer
// function still divides by sinh(eta), so literal_is_nan applies unchanged.
__device__ __forceinline__ cplx hantush_literal_dz(const DevParams &P, double a2, cplx p, cplx eta, double z,
                                                   int lay, bool storage_variant) {
  const cplx ff1 = csinh_g(eta * P.dD);
  const cplx ff2 = csinh_g(eta * P.lD1);
  const cplx sh = csinh_g(eta);
  const cplx th = 2.0 / (p + a2);
  cplx v;
  if (lay == 1) {
    const cplx g3 = cexp_g((-eta) * P.lD1) - (ff1 + cexp_g(-eta) * ff2) / sh;
    v = g3 * (eta * csinh_g(eta * z));
  } else {
    const cplx g2 = (ff1 * (eta * csinh_g(eta * z)) + ff2 * ((-eta) * csinh_g(eta * (1.0 - z)))) / sh;
    if (lay == 2) v = 0.0 - g2;
    else v = (-eta) * csinh_g(eta * (P.dD1 - z)) - g2;
  }
  return storage_variant ? v : v * th / P.bD;
}

// d/dz of fp(p) at one abscissa for layer `lay`, without the common factor a*J0(a rD)*lapTime(p)
__device__ __noinline__ cplx soln_literal_dz(const DevParams &P, const PTab &T, int pi, double a2, double z,
                                             int lay) {
  const cplx p = T.p[pi];
  const int model = P.model;
  if (model == 0) return mk(0.0, 0.0);
  const cplx eta = csqrt_g((p + a2) / P.kappa);
  if (model == 6) {
    const cplx eta1 = csqrt_g((p * P.mn_vartheta + a2) / P.kappa);
    const cplx q = eta1 / P.mn_u0;
    const cplx v = csqrt_g(1.0 + q * q);
    const cplx u = P.mn_u0 * (1.0 - v);
    const cplx etasq = (p + a2) / P.kappa;
    const cplx Delta0 = eta * csinh_g(eta) - u * ccosh_g(eta);
    const cplx pre = 2.0 / (P.kappa * etasq);
    const cplx ud = u / Delta0;
    return pre * (0.0 + ud * (eta * csinh_g(eta * z)));
  }
  if (model == 1) return hantush_literal_dz(P, a2, p, eta, z, lay, false);
  if (model == 2) {
    const cplx uDp = hantush_literal_dz(P, a2, p, eta, z, lay, true);
    const cplx uDf = T.aux[pi] / ((p + a2) * T.aux2[pi]);
    return uDf / P.bD * uDp;
  }
  // models 3,4,5: the water-table term's factor at zD = 1 (top) does not depend on z
  cplx xi = eta * P.alphaD / p;
  if (model == 3) xi = xi * (double)P.moench_M / T.aux[pi];
  cplx udp, top;
  if (model == 4) {
    udp = mk(0.0, 0.0);
    top = 2.0 / (p + a2);
  } else {
    udp = hantush_literal_dz(P, a2, p, eta, z, lay, false);
    cplx unused;
    hantush_literal<1>(P, a2, p, eta, &z, &lay, 0, true, &unused, &top, false);
  }
  const double MAXEXP = 12.014551129705717;  // -log(epsilon(1d0))/3  (constants.f90:66)
  if (eta.re < MAXEXP) {
    const cplx den = (1.0 + P.beta * eta * xi) * ccosh_g(eta) + xi * csinh_g(eta);
    return udp - top * (eta * csinh_g(eta * z)) / den;
  }
  const cplx den = 1.0 + P.beta * eta * xi + xi;
  return udp - top * (eta * cexp_g(eta * (z - 1.0))) / den;
}

// ---------------------------------------------------------------------------
// invlap.f90:46-141  de Hoog, Knight & Stokes for one time, executed by one warp.
// f: np=2M+1 transform values (shared, stride fstride); if pmul != NULL each value is
// multiplied by p first (driver.f90:228).  q,e,d: per-warp scratch of np complex each.
__device__ __noinline__ double dehoog_warp(const DevParams &P, const cplx *f, int fstride,
                                           const cplx *pmul, double t, double tee, cplx *q,
                                           cplx *e, cplx *d, int lane) {
  const int M = P.M, n2 = 2 * M;
  const unsigned full = 0xffffffffu;
  double mx = -1.0;
  bool anynum = false;
  for (int i = lane; i <= n2; i += 32) {
    cplx v = f[i * fstride];
    if (pmul) v = v * pmul[i];
    double a = hypot(v.re, v.im);
    if (!isnan(a)) { anynum = true; mx = fmax(mx, a); }
    if (isnan(v.re) || isnan(v.im)) v = mk(0.0, 0.0);
    d[i] = v;              // f for now
    e[i] = mk(0.0, 0.0);   // e(:,0) = 0
  }
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(full, mx, o));
  anynum = __any_sync(full, anynum);
  __syncwarp();
  if (!anynum || !(mx > DBL_MIN)) return 0.0;
  // q(:,1)
  for (int i = lane; i <= n2 - 1; i += 32) {
    if (i == 0) q[0] = d[1] / (d[0] / 2.0);
    else q[i] = d[i + 1] / d[i];
  }
  __syncwarp();
  if (lane == 0) d[0] = d[0] / 2.0;
  for (int r = 1; r <= M; ++r) {
    int mxi = 2 * (M - r);
    cplx t0 = mk(0, 0), t1 = mk(0, 0);
    if (lane <= mxi) t0 = q[lane + 1] - q[lane] + e[lane + 1];
    if (lane + 32 <= mxi) t1 = q[lane + 33] - q[lane + 32] + e[lane + 33];
    __syncwarp();
    if (lane <= mxi) e[lane] = t0;
    if (lane + 32 <= mxi) e[lane + 32] = t1;
    if (lane == 0) d[2 * r - 1] = -q[0];
    __syncwarp();
    if (lane == 0) d[2 * r] = -e[0];
    if (r != M) {
      mxi = 2 * (M - (r + 1)) + 1;
      if (lane <= mxi) t0 = q[lane + 1] * e[lane + 1] / e[lane];
      if (lane + 32 <= mxi) t1 = q[lane + 33] * e[lane + 33] / e[lane + 32];
      __syncwarp();
      if (lane <= mxi) q[lane] = t0;
      if (lane + 32 <= mxi) q[lane + 32] = t1;
      __syncwarp();
    }
  }
  __syncwarp();
  // z = exp(i*pi*t/tee)   (invlap.f90:110)
  const double PI = 3.141592653589793;
  double sn, cs;
  sincos_g((PI * t) / tee, &sn, &cs);
  const cplx zz = mk(cs, sn);
  cplx Am2 = mk(0.0, 0.0), Am1 = d[0], Bm2 = mk(1.0, 0.0), Bm1 = mk(1.0, 0.0);
  for (int n = 1; n <= n2 - 1; ++n) {
    cplx dn = d[n];
    cplx An = Am1 + dn * Am2 * zz;
    cplx Bn = Bm1 + dn * Bm2 * zz;
    Am2 = Am1; Am1 = An; Bm2 = Bm1; Bm1 = Bn;
  }
  cplx brem = (1.0 + (d[n2 - 1] - d[n2]) * zz) / 2.0;
  cplx rem = (-brem) * (1.0 - csqrt_g(1.0 + d[n2] * zz / (brem * brem)));
  cplx A2M = Am1 + rem * Am2;
  cplx B2M = Bm1 + rem * Bm2;
  const double gamma = P.alpha - P.log_tol / (2.0 * tee);
  return exp(gamma * t) / tee * (A2M / B2M).re;
}

// Complex quotient for the q-d table: a * conj(b)/|b|^2 with the hardware reciprocal + two
// Newton steps (<= ~2 ulp) while |b| is far from the over/underflow of |b|^2; otherwise the
// reference's own Smith division, so zero/huge/tiny divisors keep their Inf/NaN flow.
__device__ __noinline__ cplx cdiv_smith(cplx a, cplx b) { return a / b; }   // rare: kept out of line
__device__ __forceinline__ cplx cdiv_q(cplx a, cplx b) {
  const double m = fmax(fabs(b.re), fabs(b.im));
  if (m > 1e-140 && m < 1e140) {
    const double inv = rcp_fast(fma(b.re, b.re, b.im * b.im));
    return cmulf(a, mk(b.re * inv, -(b.im * inv)));
  }
  return cdiv_smith(a, b);
}

// The same inversion done by ONE thread (lane-parallel over inversions): the warp version
// above keeps 32 lanes on a <=53-entry row and pays ~7000 warp instructions per inversion;
// with one inversion per lane the q-d table is two thread-local columns updated in place
// (e(i,r) and q(i,r+1) only read entries at i and i+1 of the previous column).
// deriv: invert fp*p (driver.f90:228) with p regenerated as in deHoog_pvalues.
// EXACT: the q-d table with the reference's Smith division throughout (see dehoog_lane).
template <int MT, bool EXACT>
__device__ __noinline__ double dehoog_lane_t(const DevParams &P, const cplx *f, int fstride,
                                             bool deriv, double t, double tee) {
  auto cdiv_q = [](cplx a, cplx b) { return EXACT ? cdiv_smith(a, b) : ::unc::cdiv_q(a, b); };
  const int M = (MT > 0) ? MT : P.M, n2 = 2 * M;   // MT > 0: loop bounds known at compile time
  const double PI = 3.141592653589793;
  cplx q[2 * 31 + 2], e[2 * 31 + 2], d[2 * 31 + 2];
  double mx = -1.0;
  bool anynum = false;
  const double sigma = P.alpha - P.log_tol / (2.0 * tee);   // invlap.f90:166-170
  for (int i = 0; i <= n2; ++i) {
    cplx v = f[(size_t)i * fstride];
    if (deriv) v = v * mk(sigma, PI * (double)i / tee);
    // maxval(abs(fp)) > tiny (invlap.f90:69): abs = hypot, which is NaN iff a component is NaN
    // and none is Inf; the largest |component| decides except in the band [tiny/2, tiny]
    const bool nn = isnan(v.re) || isnan(v.im);
    const bool inf = isinf(v.re) || isinf(v.im);
    if (!(nn && !inf)) { anynum = true; mx = fmax(mx, fmax(fabs(v.re), fabs(v.im))); }
    if (nn) v = mk(0.0, 0.0);
    d[i] = v;
    e[i] = mk(0.0, 0.0);
  }
  if (!anynum) return 0.0;
  if (!(mx > DBL_MIN)) {
    if (!(mx > 0.5 * DBL_MIN)) return 0.0;
    double mh = 0.0;
    for (int i = 0; i <= n2; ++i) mh = fmax(mh, hypot(d[i].re, d[i].im));
    if (!(mh > DBL_MIN)) return 0.0;
  }
  q[0] = cdiv_q(d[1], mk(0.5 * d[0].re, 0.5 * d[0].im));
  for (int i = 1; i <= n2 - 1; ++i) q[i] = cdiv_q(d[i + 1], d[i]);
  d[0] = mk(0.5 * d[0].re, 0.5 * d[0].im);
#ifdef UNC_DEHOOG_ROWWISE
  // rows are processed in register blocks of UB entries so that the thread-local loads of a
  // block are all in flight together (the table lives in L2-backed local memory)
  constexpr int UB = 6;
  for (int r = 1; r <= M; ++r) {
    int mxi = 2 * (M - r);
    cplx qi = q[0];
    d[2 * r - 1] = -qi;
    for (int i0 = 0; i0 <= mxi; i0 += UB) {
      cplx qn[UB], en[UB];
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        const int i = min(i0 + u, mxi);          // clamped loads stay inside the row
        qn[u] = q[i + 1];
        en[u] = e[i + 1];
      }
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        if (i0 + u <= mxi) {
          e[i0 + u] = qn[u] - qi + en[u];
          qi = qn[u];
        }
      }
    }
    d[2 * r] = -e[0];
    if (r != M) {
      mxi = 2 * (M - (r + 1)) + 1;
      cplx ei = e[0];
      for (int i0 = 0; i0 <= mxi; i0 += UB) {
        cplx qn[UB], en[UB];
#pragma unroll
        for (int u = 0; u < UB; ++u) {
          const int i = min(i0 + u, mxi);
          qn[u] = q[i + 1];
          en[u] = e[i + 1];
        }
#pragma unroll
        for (int u = 0; u < UB; ++u) {
          if (i0 + u <= mxi) {
            q[i0 + u] = cdiv_q(qn[u] * en[u], ei);
            ei = en[u];
          }
        }
      }
    }
  }
#else
  // q-d rhombus, R = 2 columns per sweep.  Column r (invlap.f90:80-95) needs of column r-1 only
  // the entries i and i+1, so a sweep over i can carry R consecutive columns as a software
  // pipeline in registers: stage s turns the stream (q(i,r), e(i,r-1)) into (q(i,r+1), e(i,r))
  // with a lag of two entries, reads come from the thread-local arrays once per sweep and
  // the last stage writes behind the read position.  One load pair and one store pair per
  // entry and SWEEP instead of three of each per entry and COLUMN: the table lives in
  // L2-backed local memory and those round trips were what the inversion cost.  Stage s+1
  // consumes what stage s produced on the previous step (pipeline registers), so the R
  // stage updates of a step are independent instruction streams.
  {
#ifndef UNC_DEHOOG_R
#define UNC_DEHOOG_R 2   // measured on C5a (ms/step): column-wise 114.9, R=2 112.5, R=3 114.4, R=4 117.9 (spills)
#endif
    constexpr int R = UNC_DEHOOG_R;
    for (int r0 = 1; r0 <= M; r0 += R) {
      const int ns = min(R, M - r0 + 1);
      const int Lq0 = 2 * (M - r0) + 1;          // last q index of column r0
      cplx qprev[R], eprev[R], inq[R], ine[R];
#pragma unroll
      for (int s2 = 0; s2 < R; ++s2) { qprev[s2] = eprev[s2] = inq[s2] = ine[s2] = mk(0.0, 0.0); }
      const int tend = Lq0 + 3 * (ns - 1);
      for (int tk = 0; tk <= tend; ++tk) {
        cplx outq[R], oute[R];
        if (tk <= Lq0) { inq[0] = q[tk]; ine[0] = e[tk]; }
#pragma unroll
        for (int s2 = 0; s2 < R; ++s2) {
          outq[s2] = oute[s2] = mk(0.0, 0.0);
          const int j = tk - 3 * s2;
          if (s2 < ns && j >= 0 && j <= Lq0 - 2 * s2) {
            const int r = r0 + s2;
            const cplx qi = inq[s2], ei = ine[s2];
            if (j == 0) d[2 * r - 1] = -qi;
            if (j >= 1) {
              const cplx eo = qi - qprev[s2] + ei;        // e(j-1, r)
              if (j == 1) d[2 * r] = -eo;
              if (j >= 2) {
                const cplx qo = cdiv_q(qprev[s2] * eo, eprev[s2]);   // q(j-2, r+1)
                if (s2 == ns - 1) { q[j - 2] = qo; e[j - 2] = eprev[s2]; }
                else { outq[s2] = qo; oute[s2] = eprev[s2]; }
              }
              eprev[s2] = eo;
            }
            qprev[s2] = qi;
          }
        }
#pragma unroll
        for (int s2 = 0; s2 + 1 < R; ++s2) { inq[s2 + 1] = outq[s2]; ine[s2 + 1] = oute[s2]; }
      }
    }
  }
#endif
  double sn, cs;
  sincos_g((PI * t) / tee, &sn, &cs);
  const cplx zz = mk(cs, sn);
  cplx Am2 = mk(0.0, 0.0), Am1 = d[0], Bm2 = mk(1.0, 0.0), Bm1 = mk(1.0, 0.0);
  for (int n = 1; n <= n2 - 1; ++n) {
    const cplx dn = d[n];
    cplx An = Am1 + dn * Am2 * zz;
    cplx Bn = Bm1 + dn * Bm2 * zz;
    Am2 = Am1; Am1 = An; Bm2 = Bm1; Bm1 = Bn;
  }
  cplx brem = (1.0 + (d[n2 - 1] - d[n2]) * zz) / 2.0;
  cplx rem = (-brem) * (1.0 - csqrt_g(1.0 + d[n2] * zz / (brem * brem)));
  cplx A2M = Am1 + rem * Am2;
  cplx B2M = Bm1 + rem * Bm2;
  const double gamma = P.alpha - P.log_tol / (2.0 * tee);
  return exp(gamma * t) / tee * (A2M / B2M).re;
}

template <bool EXACT>
__device__ __forceinline__ double dehoog_lane_m(const DevParams &P, const cplx *f, int fstride,
                                                bool deriv, double t, double tee) {
#ifndef UNC_DEHOOG_RUNTIME_M
  if (P.M == 26) return dehoog_lane_t<26, EXACT>(P, f, fstride, deriv, t, tee);   // the decks' values
  if (P.M == 10) return dehoog_lane_t<10, EXACT>(P, f, fstride, deriv, t, tee);
#endif
  return dehoog_lane_t<0, EXACT>(P, f, fstride, deriv, t, tee);
}

// The reciprocal-based quotient rounds differently from Smith's division, and where the q-d
// rhombus is ill-conditioned (tiny early-time drawdowns: C5a t = 1, r = 330..500 m, z ~ 3 m)
// that alone can break it down to Inf - Inf although the reference's division does not.  Such
// a result is recomputed with the reference's division (the warp version's arithmetic); finite
// results are unchanged.
__device__ __forceinline__ double dehoog_lane(const DevParams &P, const cplx *f, int fstride,
                                              bool deriv, double t, double tee) {
  const double v = dehoog_lane_m<false>(P, f, fstride, deriv, t, tee);
  if (isfinite(v)) return v;
  return dehoog_lane_m<true>(P, f, fstride, deriv, t, tee);
}

// Wynn-epsilon for the grid kernel.  Measured alternatives (C5a, ms per step, same build
// otherwise): blocked column order without the in-column early exit (wynn_blk) 123.4; plain
// column order (wynn_dev) 125.6; epsilon table in registers in anti-diagonal order
// (wynn_reg<12>: no local memory but one serial dependency chain) ~+15%; four series in
// lockstep over local memory +6%.  UNC_WYNN_REG / UNC_WYNN_PLAIN select the others.  The grid8
// kernel keeps the table of nacc <= 14 terms in the warp's idle shared-memory stage instead
// (wynn_loz via finish8): +1.6% when first tried, -3.9% (94.7 -> 91.0 ms) once the kernel body
// had been slimmed down -- the same change, a different register allocation around it.
__device__ __noinline__ cplx wynn_grid(const cplx *series, int nacc) {
#ifdef UNC_WYNN_REG
  if (nacc <= 12) return wynn_reg<12>(series, nacc);
#endif
#ifdef UNC_WYNN_PLAIN
  return wynn_dev(series, nacc);
#else
  return wynn_blk(series, nacc);
#endif
}

// ---------------------------------------------------------------------------
__device__ __forceinline__ double shfl_down_d(double v, int d) { return __shfl_down_sync(0xffffffffu, v, d); }
__device__ __forceinline__ double shfl_xor_d(double v, int d) { return __shfl_xor_sync(0xffffffffu, v, d); }

// Fast-path evaluation of one abscissa for the ZT z-values of a point-kernel tile, as a
// separate function (own register allocation; the kernel around it holds the accumulators).
template <int ZT, int MODEL, int LMASK>
__device__ __noinline__ bool point_eval_t(const DevParams &P, cplx pp, cplx aux, cplx aux2, double a2v, double w,
                                          int lay_mask_rt, double eta_max, const double *zt, const int *lt_, int nzt,
                                          cplx *f) {
  cplx eta;
  Coef co[3];
  const int lay_mask = (LMASK > 0) ? LMASK : lay_mask_rt;   // a single z: its layer is a compile-time constant too
  if (!ap_terms_fast_t<MODEL>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, &eta, co)) return false;
#pragma unroll
  for (int k = 0; k < ZT; ++k)
    if (k < nzt) {
      const int L = lt_[k] - 1;
      const Coef &c = (L == 0) ? co[0] : ((L == 1) ? co[1] : co[2]);
      f[k] = eval_z_fast(eta, c, zt[k]);
    } else f[k] = mk(0.0, 0.0);
  return true;
}

// model (and, for a single z, the layer) known at compile time inside the call (see
// ap_terms_fast_t); the switches are warp-uniform
template <int ZT, int MODEL>
__device__ __forceinline__ bool point_eval_m(const DevParams &P, cplx pp, cplx aux, cplx aux2, double a2v, double w,
                                             int lay_mask, double eta_max, const double *zt, const int *lt_, int nzt,
                                             cplx *f) {
  if (ZT == 1) {
    if (lay_mask == 1) return point_eval_t<ZT, MODEL, 1>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, zt, lt_, nzt, f);
    if (lay_mask == 2) return point_eval_t<ZT, MODEL, 2>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, zt, lt_, nzt, f);
    if (lay_mask == 4) return point_eval_t<ZT, MODEL, 4>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, zt, lt_, nzt, f);
  }
  return point_eval_t<ZT, MODEL, 0>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, zt, lt_, nzt, f);
}
template <int ZT>
__device__ __forceinline__ bool point_eval(const DevParams &P, cplx pp, cplx aux, cplx aux2, double a2v, double w,
                                           int lay_mask, double eta_max, const double *zt, const int *lt_, int nzt,
                                           cplx *f) {
  switch (P.model) {
    case 0: return point_eval_m<ZT, 0>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, zt, lt_, nzt, f);
    case 1: return point_eval_m<ZT, 1>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, zt, lt_, nzt, f);
    case 2: return point_eval_m<ZT, 2>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, zt, lt_, nzt, f);
    case 3: return point_eval_m<ZT, 3>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, zt, lt_, nzt, f);
    case 4: return point_eval_m<ZT, 4>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, zt, lt_, nzt, f);
    case 5: return point_eval_m<ZT, 5>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, zt, lt_, nzt, f);
    default: return point_eval_m<ZT, 6>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, zt, lt_, nzt, f);
  }
}

// Fast-path screen mean at one abscissa (lh_screen_kernel): the per-(a,p) terms of the layers
// the screen touches, then one exp_pm + sincos and one S(eta h) per segment.
template <int MODEL>
__device__ __noinline__ bool screen_eval_t(const DevParams &P, cplx pp, cplx aux, cplx aux2, double a2v, double w,
                                           int lay_mask, double eta_max, const ScreenSegs *sg, cplx *f) {
  cplx eta;
  Coef co[3];
  if (!ap_terms_fast_t<MODEL>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, &eta, co)) return false;
  *f = screen_mean_fast<MODEL>(eta, co, *sg);
  return true;
}
__device__ __forceinline__ bool screen_eval(const DevParams &P, cplx pp, cplx aux, cplx aux2, double a2v, double w,
                                            int lay_mask, double eta_max, const ScreenSegs *sg, cplx *f) {
  switch (P.model) {
    case 0: return screen_eval_t<0>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, sg, f);
    case 1: return screen_eval_t<1>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, sg, f);
    case 2: return screen_eval_t<2>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, sg, f);
    case 3: return screen_eval_t<3>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, sg, f);
    case 4: return screen_eval_t<4>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, sg, f);
    case 5: return screen_eval_t<5>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, sg, f);
    default: return screen_eval_t<6>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, sg, f);
  }
}

// Fast-path vertical gradient at one abscissa (lh_dz_kernel): dz_terms_fast for the point's layer
// (a compile-time constant, as for a single z in point_eval_m).
template <int MODEL, int LMASK>
__device__ __noinline__ bool dz_eval_t(const DevParams &P, cplx pp, cplx aux, cplx aux2, double a2v, double w,
                                       double eta_max, double z, cplx *f) {
  cplx eta;
  return dz_terms_fast<MODEL>(P, pp, aux, aux2, a2v, w, (LMASK == 1) ? 1 : ((LMASK == 2) ? 2 : 3), eta_max, z,
                              &eta, f);
}
template <int MODEL>
__device__ __forceinline__ bool dz_eval_m(const DevParams &P, cplx pp, cplx aux, cplx aux2, double a2v, double w,
                                          int lay_mask, double eta_max, double z, cplx *f) {
  if (lay_mask == 1) return dz_eval_t<MODEL, 1>(P, pp, aux, aux2, a2v, w, eta_max, z, f);
  if (lay_mask == 2) return dz_eval_t<MODEL, 2>(P, pp, aux, aux2, a2v, w, eta_max, z, f);
  return dz_eval_t<MODEL, 4>(P, pp, aux, aux2, a2v, w, eta_max, z, f);
}
__device__ __forceinline__ bool dz_eval(const DevParams &P, cplx pp, cplx aux, cplx aux2, double a2v, double w,
                                        int lay_mask, double eta_max, double z, cplx *f) {
  switch (P.model) {
    case 0: return dz_eval_m<0>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, z, f);
    case 1: return dz_eval_m<1>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, z, f);
    case 2: return dz_eval_m<2>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, z, f);
    case 3: return dz_eval_m<3>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, z, f);
    case 4: return dz_eval_m<4>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, z, f);
    case 5: return dz_eval_m<5>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, z, f);
    default: return dz_eval_m<6>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, z, f);
  }
}

#ifndef UNC_PWARPS
#define UNC_PWARPS 8       // warps per CTA of the point kernel
#endif
#define UNC_PTHREADS (UNC_PWARPS * 32)
#ifndef UNC_POINT_MINB
#define UNC_POINT_MINB (16 / UNC_PWARPS)   // 128 registers, 16 warps per SM: C5b 481 ms vs 595 ms at 226 registers and 8 warps
#endif
// Work unit = one (t,r) column and a tile of ZT z-values; a CTA takes PT units (PT > 1 only with
// ZT = 1: scattered points and time series, where the Wynn phase has np and the de Hoog phase
// two jobs per unit -- a quarter of the threads and of the warps of a CTA; with four units per
// CTA both phases are full).
struct PointUnit {
  long long col;
  double tD, tee;
  double eta_max;
  int z0, nzt, lay_mask, valid;
};

__host__ __device__ inline size_t point_unit_bytes(int np, int nacc, int na, int ZT) {
  size_t b = 0;
  b += (size_t)4 * np * sizeof(cplx);                 // p, lt, aux, aux2
  b += (size_t)2 * na * sizeof(double);               // a2, wj
  b += (size_t)np * ZT * sizeof(cplx);                // finint -> totlap
  b += (size_t)ZT * (2 * sizeof(double) + 2 * sizeof(int));  // z, stale masks (64 bit), lay (padded)
  return (b + 15) & ~(size_t)15;
}

__host__ __device__ inline size_t point_smem_bytes(int np, int nacc, int na, int ZT, int PT) {
  size_t areas = (size_t)PT * np * ZT * nacc * sizeof(cplx);
  size_t scratch = (size_t)UNC_PWARPS * 3 * np * sizeof(cplx);  // de Hoog q,e,d per warp (aliases the areas)
  size_t b = (areas > scratch ? areas : scratch) + (size_t)PT * point_unit_bytes(np, nacc, na, ZT);
  b += (size_t)PT * sizeof(PointUnit);
  b = (b + 15) & ~(size_t)15;
#ifdef UNC_BUDGET_SEQSUM
  b += (size_t)UNC_PWARPS * na * sizeof(cplx);           // every abscissa's value, per warp
#endif
  return b;
}

template <int ZT, int PT>
__global__ void __launch_bounds__(UNC_PTHREADS, UNC_POINT_MINB)
lh_point_kernel(const __grid_constant__ DevParams P, const __grid_constant__ Job J) {
  static_assert(ZT == 1 || PT == 1, "several units per CTA only for one z per unit");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int np = P.np, nacc = P.nacc, G = P.G;
  const int na = P.nts_pad + P.gl_rounds * 32;
  const int ntiles = (J.nz + ZT - 1) / ZT;
  // carry post-pass (ZT == 1 only): the units come from a list instead of the launch grid
  const int fix_mode = (ZT == 1) ? J.fix_mode : 0;
  const long long nunits = fix_mode ? J.fix_n : J.ncol * (long long)ntiles;
  const long long unit0 = (long long)blockIdx.x * PT;

  // carve shared memory: areas of all units | per-unit tables | unit descriptors
  unsigned char *sp = smem_raw;
  cplx *s_area_all = (cplx *)sp;
  {
    size_t areas = (size_t)PT * np * ZT * nacc * sizeof(cplx);
    size_t scratch = (size_t)UNC_PWARPS * 3 * np * sizeof(cplx);
    sp += areas > scratch ? areas : scratch;
  }
  unsigned char *unit_base = sp;
  const size_t ub = point_unit_bytes(np, nacc, na, ZT);
  sp += (size_t)PT * ub;
  PointUnit *s_unit = (PointUnit *)sp;
#ifdef UNC_BUDGET_SEQSUM
  cplx *s_seq = (cplx *)(smem_raw + point_smem_bytes(np, nacc, na, ZT, PT)) - (size_t)UNC_PWARPS * na + (size_t)warp * na;
#endif
  struct UnitMem {
    PTab T;
    double *a2, *wj;
    cplx *fin;
    double *z;
    unsigned long long *mask;
    int *lay;
  };
  auto unit_mem = [&](int u) {
    UnitMem m;
    unsigned char *q = unit_base + (size_t)u * ub;
    m.T.p = (cplx *)q; q += np * sizeof(cplx);
    m.T.lt = (cplx *)q; q += np * sizeof(cplx);
    m.T.aux = (cplx *)q; q += np * sizeof(cplx);
    m.T.aux2 = (cplx *)q; q += np * sizeof(cplx);
    m.a2 = (double *)q; q += na * sizeof(double);
    m.wj = (double *)q; q += na * sizeof(double);
    m.fin = (cplx *)q; q += (size_t)np * ZT * sizeof(cplx);
    m.z = (double *)q; q += ZT * sizeof(double);
    m.mask = (unsigned long long *)q; q += ZT * sizeof(unsigned long long);
    m.lay = (int *)q;
    return m;
  };

  // ---- prologue -------------------------------------------------------------
  if (tid < PT) {
    const int u = tid;
    const long long U = unit0 + u;
    PointUnit d;
    d.valid = U < nunits ? 1 : 0;
    const long long pt = d.valid ? (fix_mode ? (long long)J.fix_list[U] : U) : 0;
    d.col = fix_mode ? pt / J.nz : pt / ntiles;
    d.z0 = (fix_mode ? (int)(pt % J.nz) : (int)(pt % ntiles)) * ZT;
    d.nzt = d.valid ? min(ZT, J.nz - d.z0) : 0;
    const long long tcol = d.col + J.col0;
    d.tD = J.tD[tcol / J.tdiv];
    d.tee = P.tee_mult * d.tD;
    UnitMem m = unit_mem(u);
    const double *zsrc = J.zD + (J.zstride ? d.col * (long long)J.nz : 0) + d.z0;
    const int *lsrc = J.zLay + (J.zstride ? d.col * (long long)J.nz : 0) + d.z0;
    int lay_mask = 0;
    double zabs = 0.0;
    for (int i = 0; i < ZT; ++i) {
      const double zv = (i < d.nzt) ? zsrc[i] : 0.0;
      const int lv = (i < d.nzt) ? lsrc[i] : 2;
      m.z[i] = zv; m.lay[i] = lv; m.mask[i] = 0ull;
      if (i < d.nzt) { lay_mask |= 1 << (lv - 1); zabs = fmax(zabs, fabs(zv)); }
    }
    d.lay_mask = lay_mask;
    d.eta_max = fast_eta_max(P, lay_mask, zabs);
    s_unit[u] = d;
  }
  __syncthreads();
  for (int k = tid; k < PT * np; k += UNC_PTHREADS) {
    const int u = k / np, i = k - u * np;
    if (!s_unit[u].valid) continue;
    UnitMem m = unit_mem(u);
    const double tee = s_unit[u].tee;
    // invlap.f90:166-170
    const double PI = 3.141592653589793;
    double sigma = P.alpha - P.log_tol / (2.0 * tee);
    cplx p = mk(sigma, PI * (double)i / tee);
    m.T.p[i] = p;
    m.T.lt[i] = laptime_dev(P, p);
    cplx aux = mk(0.0, 0.0), aux2 = mk(0.0, 0.0);
    if (P.model == 3) {
      // sum(1/(1 + p .X. 1/gamma), dim=2)   laplace_hankel_solutions.f90:74
      for (int mm = 0; mm < P.moench_M; ++mm) aux = aux + 1.0 / (1.0 + p * (1.0 / P.moench_gamma[mm]));
    } else if (P.model == 2) {
      // :253-266  xi = rDw*sqrt(p); A0 = 2/(p*CDw*K0 + xi*K1)
      cplx xi = P.rDw * csqrt_g(p);
      cplx K[2];
      cbesk01_dev(xi, K);
      aux = 2.0 / (p * P.CDw * K[0] + xi * K[1]);
      aux2 = p * P.tDb + 1.0;
    }
    m.T.aux[i] = aux;
    m.T.aux2[i] = aux2;
  }
  for (int k = tid; k < PT * na; k += UNC_PTHREADS) {
    const int u = k / na, idx = k - u * na;
    if (!s_unit[u].valid) continue;
    UnitMem m = unit_mem(u);
    const long long col = s_unit[u].col, tcol = col + J.col0;
    const int sv = J.sv[tcol / J.tdiv];
    const double rD = J.rD[tcol % J.rmod];
    const double arg = P.j0z[sv - 1] / rD;                      // driver.f90:120
    const double tscale = J.ts_scale ? J.ts_scale[col] : arg;  // driver.f90:121-126
    double a = 0.0, w = 0.0;
    if (idx < P.nts_pad) {
      if (idx < P.N) {
        a = (P.ts_T[idx] * tscale) / 2.0;  // integration.f90:62
        w = P.ts_wc[idx] * (arg / 2.0);    // driver.f90:135,154 + Richardson (linear in tmp)
#ifdef UNC_BUDGET_NEVILLE
        w = arg / 2.0;                     // level weights applied in the sequential sums below
#endif
      }
    } else {
      const int node = idx - P.nts_pad;   // a round of phase A = 32 consecutive nodes
      if (node < nacc * G) {
        const int j = node / G, mm = node - j * G;
        const double lob = P.j0z[sv + j - 1] / rD;  // driver.f90:188-193
        const double hib = P.j0z[sv + j] / rD;
        const double width = hib - lob;
        a = fma(width, P.gl_x[mm], hib + lob) / 2.0;
        w = P.gl_w[mm] * (width / 2.0);
      }
    }
    m.a2[idx] = a * a;
    m.wj[idx] = (w != 0.0) ? w * (a * j0_dev(a * rD)) : 0.0;  // laplace_hankel_solutions.f90:118
  }
  __syncthreads();

  // ---- phase A: Hankel quadrature sums, one warp per (unit, p) ------------------
  // A round = 32 CONSECUTIVE abscissae, one per lane, tanh-sinh rounds first, then the
  // Gauss-Lobatto nodes in interval order.  The abscissae beyond the fast-path bound (literal
  // path, ~15x the cost) are the largest ones of a point: with consecutive nodes per round they
  // fill a few whole rounds instead of costing two lanes of EVERY round (the former blocked
  // mapping, lane <-> 18 consecutive nodes, ran the literal path divergently in all rounds).
  const int rounds = P.gl_rounds;
  const int ngl = nacc * G;
  for (int job = warp; job < PT * np; job += UNC_PWARPS) {
    const int u = job / np, pi = job - u * np;
    const PointUnit un = s_unit[u];
    if (!un.valid) continue;
    const UnitMem m = unit_mem(u);
    const unsigned long long pmask = (fix_mode == 1) ? J.fix_need[J.fix_list[unit0 + u]] : ~0ull;   // p to evaluate
    if (!((pmask >> pi) & 1ull)) continue;
    const int nzt = un.nzt, lay_mask = un.lay_mask;
    const double eta_max = un.eta_max;
    double zt[ZT];
    int lt_[ZT];
#pragma unroll
    for (int i = 0; i < ZT; ++i) { zt[i] = m.z[i]; lt_[i] = m.lay[i]; }
    cplx accT[ZT], run[ZT];
#pragma unroll
    for (int i = 0; i < ZT; ++i) { accT[i] = mk(0, 0); run[i] = mk(0, 0); }
    const cplx pp = m.T.p[pi], aux = m.T.aux[pi], aux2 = m.T.aux2[pi];
    const int nts_rounds = P.nts_pad / 32;
    cplx *area_p = s_area_all + ((size_t)u * np + pi) * ZT * nacc;
    int jrun = 0;   // interval whose area the lanes are accumulating in run[] (uniform over the warp)
    int jlo_next = 0;   // first interval of the current round
    // (a source of the carry post-pass only needs the Gauss-Lobatto part)
    for (int i = (fix_mode == 1) ? nts_rounds : 0; i < nts_rounds + rounds; ++i) {
      const bool ts = i < nts_rounds;
      const int node = (i - nts_rounds) * 32 + lane;
      const int idx = ts ? i * 32 + lane : P.nts_pad + node;
      const bool valid = ts ? (idx < P.N) : (node < ngl);
      cplx f[ZT];
#pragma unroll
      for (int k = 0; k < ZT; ++k) f[k] = mk(0.0, 0.0);
      if (valid) {
        const double w = m.wj[idx], a2v = m.a2[idx];
        // per-abscissa evaluation as a call: 2% faster than inlined (own register allocation)
        if (!point_eval<ZT>(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, zt, lt_, nzt, f)) {
          const cplx eta_l = csqrt_pos(cscalef(mk(pp.re + a2v, pp.im), 1.0 / P.kappa));
          const bool sure_nan = literal_is_nan(P, eta_l);
          const double nanv = __longlong_as_double(0x7ff8000000000000LL);
#pragma unroll
          for (int k = 0; k < ZT; ++k)
            if (k < nzt) {
              if (sure_nan) f[k] = mk(nanv, nanv);
              else {
                cplx v = soln_literal_one(P, m.T, pi, a2v, zt[k], lt_[k]);
                f[k] = mk(w * v.re, w * v.im);
              }
            } else f[k] = mk(0.0, 0.0);
        }
#ifdef UNC_BUDGET_SEQSUM
        if (ZT == 1) s_seq[ts ? idx : P.N + node] = f[0];
#endif
      }
      if (ts) {
#pragma unroll
        for (int k = 0; k < ZT; ++k) accT[k] = caddf(accT[k], f[k]);
      } else {
        // the (at most two, for G >= 32) intervals this round touches, in order
        // (no integer divisions here: the first interval of a round follows from the previous round's)
        const int base = (i - nts_rounds) * 32, last = min(base + 31, ngl - 1);
        while (base >= (jlo_next + 1) * G) jlo_next += 1;
        const int j_lo = jlo_next;
        int j_hi = j_lo, myj = -1;
        while (last >= (j_hi + 1) * G) j_hi += 1;
        if (valid) { myj = j_lo; while (node >= (myj + 1) * G) myj += 1; }
        for (int j = j_lo; j <= j_hi; ++j) {
          if (j != jrun) {
            // interval jrun is complete: per-lane partial sums -> its area (once per interval)
#pragma unroll
            for (int k = 0; k < ZT; ++k) {
              double vr = run[k].re, vi = run[k].im;
              for (int o = 16; o > 0; o >>= 1) { vr += shfl_xor_d(vr, o); vi += shfl_xor_d(vi, o); }
              if (lane == 0) area_p[k * nacc + jrun] = mk(vr, vi);
              run[k] = mk(0.0, 0.0);
            }
            jrun = j;
          }
          if (myj == j) {
#pragma unroll
            for (int k = 0; k < ZT; ++k) run[k] = caddf(run[k], f[k]);
          }
        }
      }
    }
#pragma unroll
    for (int k = 0; k < ZT; ++k) {
      double vr = run[k].re, vi = run[k].im;
      for (int o = 16; o > 0; o >>= 1) { vr += shfl_xor_d(vr, o); vi += shfl_xor_d(vi, o); }
      if (lane == 0) area_p[k * nacc + jrun] = mk(vr, vi);
    }
#pragma unroll
    for (int k = 0; k < ZT; ++k) {
      double tr = accT[k].re, ti = accT[k].im;
      for (int o = 16; o > 0; o >>= 1) { tr += shfl_xor_d(tr, o); ti += shfl_xor_d(ti, o); }
      if (lane == 0) m.fin[pi * ZT + k] = mk(tr, ti);
    }
#ifdef UNC_BUDGET_SEQSUM
    // error-budget build: redo the sums sequentially in the reference's order (driver.f90:135-157,
    // 201-202) from the stored per-abscissa values, one lane per p
    __syncwarp();
    if (ZT == 1 && lane == 0) {
#ifdef UNC_BUDGET_NEVILLE
      // R level sums with their own weights, then extraptozero (integration.f90:192-237)
      cplx c_[12], d_[12];
      double x_[12];
      const int R = P.R;
      const double *lw = P.ts_lw;
      for (int j = 1; j <= R; ++j) {
        const int kv = P.ts_k - R + j, Nv = (1 << kv) - 1, step = 1 << (R - j);
        cplx sum = mk(0.0, 0.0);
        for (int mm = 1; mm <= Nv; ++mm) sum = caddf(sum, cscalef(s_seq[mm * step - 1], lw[mm - 1]));
        lw += Nv;
        c_[j - 1] = d_[j - 1] = sum;
        x_[j - 1] = 4.0 / (double)(1 << kv);
      }
      int ns = R;                    // hv decreasing: the smallest x is the last
      cplx y = c_[ns - 1];
      ns -= 1;
      for (int mm = 1; mm <= R - 1; ++mm) {
        for (int i = 1; i <= R - mm; ++i) {
          const double dx = x_[i - 1] - x_[i + mm - 1];
          const cplx den = mk((c_[i].re - d_[i - 1].re) / dx, (c_[i].im - d_[i - 1].im) / dx);
          d_[i - 1] = cscalef(den, x_[i + mm - 1]);
          c_[i - 1] = cscalef(den, x_[i - 1]);
        }
        cplx dy;
        if (2 * ns < R - mm) dy = c_[ns];
        else { dy = d_[ns - 1]; ns -= 1; }
        y = caddf(y, dy);
      }
      m.fin[pi * ZT] = (R > 1) ? y : c_[0];
#else
      cplx sum = mk(0.0, 0.0);
      for (int mm = 0; mm < P.N; ++mm) sum = caddf(sum, s_seq[mm]);
      m.fin[pi * ZT] = sum;
#endif
      for (int j = 0; j < nacc; ++j) {
        cplx a_ = mk(0.0, 0.0);
        for (int mm = 0; mm < G; ++mm) a_ = caddf(a_, s_seq[P.N + j * G + mm]);
        area_p[j] = a_;
      }
    }
    __syncwarp();
#endif
  }
  __syncthreads();

  // ---- phase B: Wynn-epsilon per (unit,p,z), totlap = finint + infint -----------
  for (int k = tid; k < PT * np * ZT; k += UNC_PTHREADS) {
    const int u = k / (np * ZT), kk = k - u * (np * ZT);
    const int pi = kk / ZT, zi = kk - pi * ZT;
    if (!s_unit[u].valid) continue;
    const UnitMem m = unit_mem(u);
    const unsigned long long pmask = (fix_mode == 1) ? J.fix_need[J.fix_list[unit0 + u]] : ~0ull;
    if (zi < s_unit[u].nzt && ((pmask >> pi) & 1ull)) {
      const double nan = __longlong_as_double(0x7ff8000000000000LL);
      const cplx lt = m.T.lt[pi];
      cplx series[UNC_MAX_NACC];
      bool any = false;
      for (int j = 0; j < nacc; ++j) {
        cplx a = s_area_all[(((size_t)u * np + pi) * ZT + zi) * nacc + j];
        a = is_finite_c(a) ? a * lt : mk(nan, nan);
        series[j] = a;
        if (cabs_d(a) > 0.0) any = true;   // driver.f90:209
      }
      cplx infint = mk(0.0, 0.0);
      if (any) infint = wynn_any(series, nacc);
      else {
        atomicOr(&m.mask[zi], 1ull << pi);
        if (fix_mode == 2) {
          // driver.f90:209-211: infint(p,z) keeps the value of the last (t,r) that set it
          const int src = J.fix_src[(size_t)(unit0 + u) * np + pi];
          if (src >= 0) {
            const double *v = J.fix_val + ((size_t)src * np + pi) * 2;
            infint = mk(v[0], v[1]);
          }
        }
      }
      if (fix_mode == 1) {
        double *v = J.fix_val + ((size_t)(unit0 + u) * np + pi) * 2;
        v[0] = infint.re; v[1] = infint.im;
      }
      cplx fin = m.fin[kk];
      fin = is_finite_c(fin) ? fin * lt : mk(nan, nan);
      m.fin[kk] = fin + infint;  // totlap, driver.f90:216
    }
  }
  __syncthreads();
  if (fix_mode == 1) return;

  // ---- phase C: de Hoog inversion of value and log-time derivative ------------
  cplx *scr = s_area_all + (size_t)warp * 3 * np;
  for (int job = warp; job < PT * 2 * ZT; job += UNC_PWARPS) {
    const int u = job / (2 * ZT), jj = job - u * (2 * ZT);
    const int zi = jj >> 1, deriv = jj & 1;
    const PointUnit un = s_unit[u];
    if (!un.valid || zi >= un.nzt) continue;
    const UnitMem m = unit_mem(u);
    double v = dehoog_warp(P, m.fin + zi, ZT, deriv ? m.T.p : nullptr, un.tD, un.tee, scr, scr + np,
                           scr + 2 * np, lane);
    if (lane == 0) {
      const long long o = un.col * (long long)J.nz + un.z0 + zi;
      const long long U = unit0 + u;
      if (fix_mode == 2) {
        if (deriv) { J.fix_ds[U] = v * un.tD; if (J.ds) J.ds[o] = v * un.tD; }
        else { J.fix_s[U] = v; if (J.s) J.s[o] = v; }
      } else if (deriv) J.ds[o] = v * un.tD;  // driver.f90:228
      else {
        J.s[o] = v;
        if (J.flags) J.flags[o] = m.mask[zi] != 0ull ? 1 : 0;
        if (J.smask) J.smask[o] = m.mask[zi];
        if (J.nstale && m.mask[zi] != 0ull) atomicAdd(J.nstale, 1u);
      }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------
// Screened observation wells (unc_eval_screens): lh_point_kernel<1,1> with one screen per CTA.
// The screen's up to three segments take the place of the unit's z-tile and the integrand is
// their weighted mean (screen_eval / screen_literal); the prologue tables, the phase-A sums, the
// Wynn and de Hoog phases are the point kernel's, step for step.  Job::zD holds the bottoms,
// `ztop` the tops; fix_mode is 0 or 3 (cost-ordered list), there is no carry between screens.
__host__ __device__ inline size_t screen_smem_bytes(int np, int nacc, int na) {
  size_t b = (size_t)np * nacc * sizeof(cplx);                       // areas
  const size_t scratch = (size_t)UNC_PWARPS * 3 * np * sizeof(cplx);  // de Hoog q,e,d per warp (aliases the areas)
  if (scratch > b) b = scratch;
  b += (size_t)4 * np * sizeof(cplx);                                 // p, lt, aux, aux2
  b += (size_t)2 * na * sizeof(double);                               // a2, wj
  b += (size_t)np * sizeof(cplx);                                     // finint -> totlap
  b += sizeof(ScreenSegs) + 16;                                       // segments, stale mask
  return (b + 15) & ~(size_t)15;
}

__global__ void __launch_bounds__(UNC_PTHREADS, UNC_POINT_MINB)
lh_screen_kernel(const __grid_constant__ DevParams P, const __grid_constant__ Job J, const double *__restrict__ ztop) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int np = P.np, nacc = P.nacc, G = P.G;
  const int na = P.nts_pad + P.gl_rounds * 32;
  if ((long long)blockIdx.x >= J.ncol) return;
  const long long col = (J.fix_mode == 3) ? (long long)J.fix_list[blockIdx.x] : (long long)blockIdx.x;

  unsigned char *sp = smem_raw;
  cplx *s_area = (cplx *)sp;
  {
    const size_t areas = (size_t)np * nacc * sizeof(cplx);
    const size_t scratch = (size_t)UNC_PWARPS * 3 * np * sizeof(cplx);
    sp += areas > scratch ? areas : scratch;
  }
  PTab T;
  T.p = (cplx *)sp; sp += np * sizeof(cplx);
  T.lt = (cplx *)sp; sp += np * sizeof(cplx);
  T.aux = (cplx *)sp; sp += np * sizeof(cplx);
  T.aux2 = (cplx *)sp; sp += np * sizeof(cplx);
  double *s_a2 = (double *)sp; sp += na * sizeof(double);
  double *s_wj = (double *)sp; sp += na * sizeof(double);
  cplx *s_fin = (cplx *)sp; sp += np * sizeof(cplx);
  ScreenSegs *s_seg = (ScreenSegs *)sp; sp += sizeof(ScreenSegs);
  unsigned long long *s_mask = (unsigned long long *)(((size_t)sp + 7) & ~(size_t)7);

  const double tD = J.tD[col], tee = P.tee_mult * tD;
  // ---- prologue -------------------------------------------------------------
  if (tid == 0) {
    ScreenSegs sg;
    screen_segments(J.zD[col], ztop[col], P.lD1, P.dD1, &sg);
    *s_seg = sg;
    *s_mask = 0ull;
  }
  for (int i = tid; i < np; i += UNC_PTHREADS) {
    // invlap.f90:166-170
    const double PI = 3.141592653589793;
    double sigma = P.alpha - P.log_tol / (2.0 * tee);
    cplx p = mk(sigma, PI * (double)i / tee);
    T.p[i] = p;
    T.lt[i] = laptime_dev(P, p);
    cplx aux = mk(0.0, 0.0), aux2 = mk(0.0, 0.0);
    if (P.model == 3) {
      for (int mm = 0; mm < P.moench_M; ++mm) aux = aux + 1.0 / (1.0 + p * (1.0 / P.moench_gamma[mm]));
    } else if (P.model == 2) {
      cplx xi = P.rDw * csqrt_g(p);
      cplx K[2];
      cbesk01_dev(xi, K);
      aux = 2.0 / (p * P.CDw * K[0] + xi * K[1]);
      aux2 = p * P.tDb + 1.0;
    }
    T.aux[i] = aux;
    T.aux2[i] = aux2;
  }
  {
    const int sv = J.sv[col];
    const double rD = J.rD[col];
    const double arg = P.j0z[sv - 1] / rD;                      // driver.f90:120
    const double tscale = J.ts_scale ? J.ts_scale[col] : arg;  // driver.f90:121-126
    for (int idx = tid; idx < na; idx += UNC_PTHREADS) {
      double a = 0.0, w = 0.0;
      if (idx < P.nts_pad) {
        if (idx < P.N) {
          a = (P.ts_T[idx] * tscale) / 2.0;  // integration.f90:62
          w = P.ts_wc[idx] * (arg / 2.0);    // driver.f90:135,154 + Richardson (linear in tmp)
        }
      } else {
        const int node = idx - P.nts_pad;
        if (node < nacc * G) {
          const int j = node / G, mm = node - j * G;
          const double lob = P.j0z[sv + j - 1] / rD;  // driver.f90:188-193
          const double hib = P.j0z[sv + j] / rD;
          const double width = hib - lob;
          a = fma(width, P.gl_x[mm], hib + lob) / 2.0;
          w = P.gl_w[mm] * (width / 2.0);
        }
      }
      s_a2[idx] = a * a;
      s_wj[idx] = (w != 0.0) ? w * (a * j0_dev(a * rD)) : 0.0;  // laplace_hankel_solutions.f90:118
    }
  }
  __syncthreads();
  const int lay_mask = s_seg->lay_mask;
  const double eta_max = fast_eta_max(P, lay_mask, ztop[col]);   // zabs = ztop

  // ---- phase A: Hankel quadrature sums, one warp per p (as lh_point_kernel) ------------
  const int rounds = P.gl_rounds;
  const int ngl = nacc * G;
  const int nts_rounds = P.nts_pad / 32;
  for (int pi = warp; pi < np; pi += UNC_PWARPS) {
    cplx accT = mk(0, 0), run = mk(0, 0);
    const cplx pp = T.p[pi], aux = T.aux[pi], aux2 = T.aux2[pi];
    cplx *area_p = s_area + (size_t)pi * nacc;
    int jrun = 0, jlo_next = 0;
    for (int i = 0; i < nts_rounds + rounds; ++i) {
      const bool ts = i < nts_rounds;
      const int node = (i - nts_rounds) * 32 + lane;
      const int idx = ts ? i * 32 + lane : P.nts_pad + node;
      const bool valid = ts ? (idx < P.N) : (node < ngl);
      cplx f = mk(0.0, 0.0);
      if (valid) {
        const double w = s_wj[idx], a2v = s_a2[idx];
        if (!screen_eval(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, s_seg, &f)) {
          const cplx eta_l = csqrt_pos(cscalef(mk(pp.re + a2v, pp.im), 1.0 / P.kappa));
          if (literal_is_nan(P, eta_l)) {
            const double nanv = __longlong_as_double(0x7ff8000000000000LL);
            f = mk(nanv, nanv);
          } else {
            const cplx v = screen_literal(P, T, pi, a2v, s_seg);
            f = mk(w * v.re, w * v.im);
          }
        }
      }
      if (ts) {
        accT = caddf(accT, f);
      } else {
        const int base = (i - nts_rounds) * 32, last = min(base + 31, ngl - 1);
        while (base >= (jlo_next + 1) * G) jlo_next += 1;
        const int j_lo = jlo_next;
        int j_hi = j_lo, myj = -1;
        while (last >= (j_hi + 1) * G) j_hi += 1;
        if (valid) { myj = j_lo; while (node >= (myj + 1) * G) myj += 1; }
        for (int j = j_lo; j <= j_hi; ++j) {
          if (j != jrun) {
            double vr = run.re, vi = run.im;
            for (int o = 16; o > 0; o >>= 1) { vr += shfl_xor_d(vr, o); vi += shfl_xor_d(vi, o); }
            if (lane == 0) area_p[jrun] = mk(vr, vi);
            run = mk(0.0, 0.0);
            jrun = j;
          }
          if (myj == j) run = caddf(run, f);
        }
      }
    }
    {
      double vr = run.re, vi = run.im;
      for (int o = 16; o > 0; o >>= 1) { vr += shfl_xor_d(vr, o); vi += shfl_xor_d(vi, o); }
      if (lane == 0) area_p[jrun] = mk(vr, vi);
      double tr = accT.re, ti = accT.im;
      for (int o = 16; o > 0; o >>= 1) { tr += shfl_xor_d(tr, o); ti += shfl_xor_d(ti, o); }
      if (lane == 0) s_fin[pi] = mk(tr, ti);
    }
  }
  __syncthreads();

  // ---- phase B: Wynn-epsilon per p, totlap = finint + infint -------------------------
  for (int pi = tid; pi < np; pi += UNC_PTHREADS) {
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    const cplx lt = T.lt[pi];
    cplx series[UNC_MAX_NACC];
    bool any = false;
    for (int j = 0; j < nacc; ++j) {
      cplx a = s_area[(size_t)pi * nacc + j];
      a = is_finite_c(a) ? a * lt : mk(nan, nan);
      series[j] = a;
      if (cabs_d(a) > 0.0) any = true;   // driver.f90:209
    }
    cplx infint = mk(0.0, 0.0);
    if (any) infint = wynn_any(series, nacc);
    else atomicOr(s_mask, 1ull << pi);   // stale: infint = 0, flagged
    cplx fin = s_fin[pi];
    fin = is_finite_c(fin) ? fin * lt : mk(nan, nan);
    s_fin[pi] = fin + infint;  // totlap, driver.f90:216
  }
  __syncthreads();

  // ---- phase C: de Hoog inversion of value (warp 0) and log-time derivative (warp 1) --------
  if (warp < 2) {
    const int deriv = warp;
    cplx *scr = s_area + (size_t)warp * 3 * np;
    const double v = dehoog_warp(P, s_fin, 1, deriv ? T.p : nullptr, tD, tee, scr, scr + np, scr + 2 * np, lane);
    if (lane == 0) {
      if (deriv) J.ds[col] = v * tD;  // driver.f90:228
      else {
        J.s[col] = v;
        if (J.flags) J.flags[col] = *s_mask != 0ull ? 1 : 0;
      }
    }
  }
}

// ---------------------------------------------------------------------------
// Vertical gradient at points (unc_eval_points_dz): lh_point_kernel<1,1> with one point per CTA
// and the integrand replaced by its z-derivative (dz_eval / soln_literal_dz); the prologue
// tables, the phase-A sums, the Wynn and de Hoog phases are the point kernel's, step for step.
// The layer is geometric (1 below 1-lD, 2 below 1-dD, else 3), not read from zLay.  fix_mode is
// 0 or 3 (cost-ordered list); there is no carry between points.  A body of its own, as
// lh_screen_kernel: routing the point kernel through a shared body changes its code.
__host__ __device__ inline size_t dz_smem_bytes(int np, int nacc, int na) {
  size_t b = (size_t)np * nacc * sizeof(cplx);                       // areas
  const size_t scratch = (size_t)UNC_PWARPS * 3 * np * sizeof(cplx);  // de Hoog q,e,d per warp (aliases the areas)
  if (scratch > b) b = scratch;
  b += (size_t)4 * np * sizeof(cplx);                                 // p, lt, aux, aux2
  b += (size_t)2 * na * sizeof(double);                               // a2, wj
  b += (size_t)np * sizeof(cplx);                                     // finint -> totlap
  b += 16;                                                            // stale mask
  return (b + 15) & ~(size_t)15;
}

__global__ void __launch_bounds__(UNC_PTHREADS, UNC_POINT_MINB)
lh_dz_kernel(const __grid_constant__ DevParams P, const __grid_constant__ Job J) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int np = P.np, nacc = P.nacc, G = P.G;
  const int na = P.nts_pad + P.gl_rounds * 32;
  if ((long long)blockIdx.x >= J.ncol) return;
  const long long col = (J.fix_mode == 3) ? (long long)J.fix_list[blockIdx.x] : (long long)blockIdx.x;

  unsigned char *sp = smem_raw;
  cplx *s_area = (cplx *)sp;
  {
    const size_t areas = (size_t)np * nacc * sizeof(cplx);
    const size_t scratch = (size_t)UNC_PWARPS * 3 * np * sizeof(cplx);
    sp += areas > scratch ? areas : scratch;
  }
  PTab T;
  T.p = (cplx *)sp; sp += np * sizeof(cplx);
  T.lt = (cplx *)sp; sp += np * sizeof(cplx);
  T.aux = (cplx *)sp; sp += np * sizeof(cplx);
  T.aux2 = (cplx *)sp; sp += np * sizeof(cplx);
  double *s_a2 = (double *)sp; sp += na * sizeof(double);
  double *s_wj = (double *)sp; sp += na * sizeof(double);
  cplx *s_fin = (cplx *)sp; sp += np * sizeof(cplx);
  unsigned long long *s_mask = (unsigned long long *)(((size_t)sp + 7) & ~(size_t)7);

  const double tD = J.tD[col], tee = P.tee_mult * tD;
  const double z = J.zD[col];
  const int lay = (z < P.lD1) ? 1 : ((z < P.dD1) ? 2 : 3);
  // ---- prologue -------------------------------------------------------------
  if (tid == 0) *s_mask = 0ull;
  for (int i = tid; i < np; i += UNC_PTHREADS) {
    // invlap.f90:166-170
    const double PI = 3.141592653589793;
    double sigma = P.alpha - P.log_tol / (2.0 * tee);
    cplx p = mk(sigma, PI * (double)i / tee);
    T.p[i] = p;
    T.lt[i] = laptime_dev(P, p);
    cplx aux = mk(0.0, 0.0), aux2 = mk(0.0, 0.0);
    if (P.model == 3) {
      for (int mm = 0; mm < P.moench_M; ++mm) aux = aux + 1.0 / (1.0 + p * (1.0 / P.moench_gamma[mm]));
    } else if (P.model == 2) {
      cplx xi = P.rDw * csqrt_g(p);
      cplx K[2];
      cbesk01_dev(xi, K);
      aux = 2.0 / (p * P.CDw * K[0] + xi * K[1]);
      aux2 = p * P.tDb + 1.0;
    }
    T.aux[i] = aux;
    T.aux2[i] = aux2;
  }
  {
    const int sv = J.sv[col];
    const double rD = J.rD[col];
    const double arg = P.j0z[sv - 1] / rD;                      // driver.f90:120
    const double tscale = J.ts_scale ? J.ts_scale[col] : arg;  // driver.f90:121-126
    for (int idx = tid; idx < na; idx += UNC_PTHREADS) {
      double a = 0.0, w = 0.0;
      if (idx < P.nts_pad) {
        if (idx < P.N) {
          a = (P.ts_T[idx] * tscale) / 2.0;  // integration.f90:62
          w = P.ts_wc[idx] * (arg / 2.0);    // driver.f90:135,154 + Richardson (linear in tmp)
        }
      } else {
        const int node = idx - P.nts_pad;
        if (node < nacc * G) {
          const int j = node / G, mm = node - j * G;
          const double lob = P.j0z[sv + j - 1] / rD;  // driver.f90:188-193
          const double hib = P.j0z[sv + j] / rD;
          const double width = hib - lob;
          a = fma(width, P.gl_x[mm], hib + lob) / 2.0;
          w = P.gl_w[mm] * (width / 2.0);
        }
      }
      s_a2[idx] = a * a;
      s_wj[idx] = (w != 0.0) ? w * (a * j0_dev(a * rD)) : 0.0;  // laplace_hankel_solutions.f90:118
    }
  }
  __syncthreads();
  const int lay_mask = 1 << (lay - 1);
  const double eta_max = fast_eta_max(P, lay_mask, z);   // as for a point (0 <= z <= 1)

  // ---- phase A: Hankel quadrature sums, one warp per p (as lh_point_kernel) ------------
  const int rounds = P.gl_rounds;
  const int ngl = nacc * G;
  const int nts_rounds = P.nts_pad / 32;
  for (int pi = warp; pi < np; pi += UNC_PWARPS) {
    cplx accT = mk(0, 0), run = mk(0, 0);
    const cplx pp = T.p[pi], aux = T.aux[pi], aux2 = T.aux2[pi];
    cplx *area_p = s_area + (size_t)pi * nacc;
    int jrun = 0, jlo_next = 0;
    for (int i = 0; i < nts_rounds + rounds; ++i) {
      const bool ts = i < nts_rounds;
      const int node = (i - nts_rounds) * 32 + lane;
      const int idx = ts ? i * 32 + lane : P.nts_pad + node;
      const bool valid = ts ? (idx < P.N) : (node < ngl);
      cplx f = mk(0.0, 0.0);
      if (valid) {
        const double w = s_wj[idx], a2v = s_a2[idx];
        if (!dz_eval(P, pp, aux, aux2, a2v, w, lay_mask, eta_max, z, &f)) {
          const cplx eta_l = csqrt_pos(cscalef(mk(pp.re + a2v, pp.im), 1.0 / P.kappa));
          if (literal_is_nan(P, eta_l)) {
            const double nanv = __longlong_as_double(0x7ff8000000000000LL);
            f = mk(nanv, nanv);
          } else {
            const cplx v = soln_literal_dz(P, T, pi, a2v, z, lay);
            f = mk(w * v.re, w * v.im);
          }
        }
      }
      if (ts) {
        accT = caddf(accT, f);
      } else {
        const int base = (i - nts_rounds) * 32, last = min(base + 31, ngl - 1);
        while (base >= (jlo_next + 1) * G) jlo_next += 1;
        const int j_lo = jlo_next;
        int j_hi = j_lo, myj = -1;
        while (last >= (j_hi + 1) * G) j_hi += 1;
        if (valid) { myj = j_lo; while (node >= (myj + 1) * G) myj += 1; }
        for (int j = j_lo; j <= j_hi; ++j) {
          if (j != jrun) {
            double vr = run.re, vi = run.im;
            for (int o = 16; o > 0; o >>= 1) { vr += shfl_xor_d(vr, o); vi += shfl_xor_d(vi, o); }
            if (lane == 0) area_p[jrun] = mk(vr, vi);
            run = mk(0.0, 0.0);
            jrun = j;
          }
          if (myj == j) run = caddf(run, f);
        }
      }
    }
    {
      double vr = run.re, vi = run.im;
      for (int o = 16; o > 0; o >>= 1) { vr += shfl_xor_d(vr, o); vi += shfl_xor_d(vi, o); }
      if (lane == 0) area_p[jrun] = mk(vr, vi);
      double tr = accT.re, ti = accT.im;
      for (int o = 16; o > 0; o >>= 1) { tr += shfl_xor_d(tr, o); ti += shfl_xor_d(ti, o); }
      if (lane == 0) s_fin[pi] = mk(tr, ti);
    }
  }
  __syncthreads();

  // ---- phase B: Wynn-epsilon per p, totlap = finint + infint -------------------------
  for (int pi = tid; pi < np; pi += UNC_PTHREADS) {
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    const cplx lt = T.lt[pi];
    cplx series[UNC_MAX_NACC];
    bool any = false;
    for (int j = 0; j < nacc; ++j) {
      cplx a = s_area[(size_t)pi * nacc + j];
      a = is_finite_c(a) ? a * lt : mk(nan, nan);
      series[j] = a;
      if (cabs_d(a) > 0.0) any = true;   // driver.f90:209
    }
    cplx infint = mk(0.0, 0.0);
    if (any) infint = wynn_any(series, nacc);
    else atomicOr(s_mask, 1ull << pi);   // stale: infint = 0, flagged
    cplx fin = s_fin[pi];
    fin = is_finite_c(fin) ? fin * lt : mk(nan, nan);
    s_fin[pi] = fin + infint;  // totlap, driver.f90:216
  }
  __syncthreads();

  // ---- phase C: de Hoog inversion of gz (warp 0) and of its log-time derivative (warp 1) ----
  if (warp < 2) {
    const int deriv = warp;
    cplx *scr = s_area + (size_t)warp * 3 * np;
    const double v = dehoog_warp(P, s_fin, 1, deriv ? T.p : nullptr, tD, tee, scr, scr + np, scr + 2 * np, lane);
    if (lane == 0) {
      if (deriv) J.ds[col] = v * tD;  // driver.f90:228
      else {
        J.s[col] = v;
        if (J.flags) J.flags[col] = *s_mask != 0ull ? 1 : 0;
      }
    }
  }
}

// ---------------------------------------------------------------------------
// Grid kernel: lanes <-> z.  One CTA = one (t,r) column and a block of 32 z-values;
// one warp per p.  The per-(a,p) terms (ap_terms_fast) are computed lane-parallel for 32
// abscissae at a time and staged in shared memory; then every lane walks those 32
// abscissae for ITS z (one exp_pm + one sincos each), accumulating the tanh-sinh sum
// and the Gauss-Lobatto interval areas in abscissa order (the reference's own
// summation order, driver.f90:135,201).  Abscissae whose Re(eta) exceeds the fast-path
// bound take the literal path -- a warp-uniform branch in this layout.
struct StageEnt {
  cplx eta;
  Coef co[3];
};
struct CoefAosSink {   // ap_terms_fast_s sink: a layer's coefficients into a staged entry in shared memory
  Coef *co;
  __device__ __forceinline__ void set(int L, cplx k0, cplx cp, cplx cm) const {
    co[L].k0 = k0; co[L].cp = cp; co[L].cm = cm;
  }
  __device__ __forceinline__ void wt(cplx, cplx) const {}
};

__host__ __device__ inline size_t grid_smem_bytes(int np, int na_seq, int ZL) {
  size_t b = 0;
  b += (size_t)4 * np * sizeof(cplx);                       // p, lt, aux, aux2
  b += (size_t)2 * na_seq * sizeof(double);                 // a2, wj
  b += (size_t)np * 32 * ZL * sizeof(cplx);                 // totlap[p][z]
  size_t stage = (size_t)UNC_WARPS * 32 * sizeof(StageEnt) + (size_t)UNC_WARPS * 32 * sizeof(int);
  size_t scratch = (size_t)UNC_WARPS * 3 * np * sizeof(cplx);  // de Hoog scratch aliases the stage
  b += stage > scratch ? stage : scratch;
  b += 64;
  return (b + 15) & ~(size_t)15;
}

template <int ZL>
__global__ void __launch_bounds__(UNC_THREADS, 2)
lh_grid_kernel(const __grid_constant__ DevParams P, const __grid_constant__ Job J) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int ZB = 32 * ZL;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int np = P.np, nacc = P.nacc, G = P.G, N = P.N;
  const int NA = N + nacc * G;
  const int na_seq = (NA + 31) & ~31;
  const int nzb = (J.nz + ZB - 1) / ZB;
  const long long col = blockIdx.x / nzb;
  const int z0 = (int)(blockIdx.x % nzb) * ZB;
  const int nzv = min(ZB, J.nz - z0);

  unsigned char *sp = smem_raw;
  PTab T;
  T.p = (cplx *)sp; sp += np * sizeof(cplx);
  T.lt = (cplx *)sp; sp += np * sizeof(cplx);
  T.aux = (cplx *)sp; sp += np * sizeof(cplx);
  T.aux2 = (cplx *)sp; sp += np * sizeof(cplx);
  double *s_a2 = (double *)sp; sp += na_seq * sizeof(double);
  double *s_wj = (double *)sp; sp += na_seq * sizeof(double);
  cplx *s_tot = (cplx *)sp; sp += (size_t)np * ZB * sizeof(cplx);
  StageEnt *s_stage = (StageEnt *)sp;
  int *s_ok = (int *)(sp + (size_t)UNC_WARPS * 32 * sizeof(StageEnt));
  cplx *s_scr = (cplx *)sp;
  {
    size_t stage = (size_t)UNC_WARPS * 32 * sizeof(StageEnt) + (size_t)UNC_WARPS * 32 * sizeof(int);
    size_t scratch = (size_t)UNC_WARPS * 3 * np * sizeof(cplx);
    sp += stage > scratch ? stage : scratch;
  }
  int *s_misc = (int *)sp;  // [0] layer mask, [1] bits of max|z| (float)

  const long long tcol = col + J.col0;
  const double tD = J.tD[tcol / J.tdiv];
  const int sv = J.sv[tcol / J.tdiv];
  const double rD = J.rD[tcol % J.rmod];
  const double tee = P.tee_mult * tD;
  const double arg = P.j0z[sv - 1] / rD;                      // driver.f90:120
  const double tscale = J.ts_scale ? J.ts_scale[col] : arg;  // driver.f90:121-126
  const long long zbase = (J.zstride ? col * (long long)J.nz : 0) + z0;
  double myz[ZL];
  int mylay[ZL];
  bool zvalid[ZL];
#pragma unroll
  for (int k = 0; k < ZL; ++k) {
    const int zi = lane + 32 * k;
    zvalid[k] = zi < nzv;
    myz[k] = zvalid[k] ? J.zD[zbase + zi] : 0.0;
    mylay[k] = zvalid[k] ? J.zLay[zbase + zi] : 0;
  }

  // ---- prologue ---------------------------------------------------------------
  for (int i = tid; i < np; i += UNC_THREADS) {
    const double PI = 3.141592653589793;
    double sigma = P.alpha - P.log_tol / (2.0 * tee);   // invlap.f90:166-170
    cplx p = mk(sigma, PI * (double)i / tee);
    T.p[i] = p;
    T.lt[i] = laptime_dev(P, p);
    cplx aux = mk(0.0, 0.0), aux2 = mk(0.0, 0.0);
    if (P.model == 3) {
      for (int m = 0; m < P.moench_M; ++m) aux = aux + 1.0 / (1.0 + p * (1.0 / P.moench_gamma[m]));
    } else if (P.model == 2) {
      cplx xi = P.rDw * csqrt_g(p);
      cplx K[2];
      cbesk01_dev(xi, K);
      aux = 2.0 / (p * P.CDw * K[0] + xi * K[1]);
      aux2 = p * P.tDb + 1.0;
    }
    T.aux[i] = aux;
    T.aux2[i] = aux2;
  }
  for (int idx = tid; idx < na_seq; idx += UNC_THREADS) {
    double a = 0.0, w = 0.0;
    if (idx < N) {
      a = (P.ts_T[idx] * tscale) / 2.0;  // integration.f90:62
      w = P.ts_wc[idx] * (arg / 2.0);    // driver.f90:135,154 + Richardson (linear in tmp)
    } else if (idx < NA) {
      const int node = idx - N;
      const int j = node / G, m = node - j * G;
      const double lob = P.j0z[sv + j - 1] / rD;  // driver.f90:188-193
      const double hib = P.j0z[sv + j] / rD;
      const double width = hib - lob;
      a = fma(width, P.gl_x[m], hib + lob) / 2.0;
      w = P.gl_w[m] * (width / 2.0);
    }
    s_a2[idx] = a * a;
    s_wj[idx] = (w != 0.0) ? w * (a * j0_dev(a * rD)) : 0.0;  // laplace_hankel_solutions.f90:118
  }
  if (warp == 0) {
    int m = 0;
    float za = 0.f;
#pragma unroll
    for (int k = 0; k < ZL; ++k)
      if (zvalid[k]) { m |= 1 << (mylay[k] - 1); za = fmaxf(za, (float)fabs(myz[k]) * 1.0000002f); }
    for (int o = 16; o > 0; o >>= 1) {
      m |= __shfl_xor_sync(0xffffffffu, m, o);
      za = fmaxf(za, __shfl_xor_sync(0xffffffffu, za, o));
    }
    if (lane == 0) { s_misc[0] = m; s_misc[1] = __float_as_int(za); }
  }
  __syncthreads();
  const int lay_mask = s_misc[0];
  const double eta_max = fast_eta_max(P, lay_mask, (double)__int_as_float(s_misc[1]));
  const bool uniform = (lay_mask & (lay_mask - 1)) == 0;   // one layer in the whole block
  const int L0 = __ffs(lay_mask) - 1;
  int myL[ZL];
#pragma unroll
  for (int k = 0; k < ZL; ++k) {
    if (!zvalid[k]) { mylay[k] = L0 + 1; myz[k] = 0.5; }   // padding lanes mimic a present layer
    myL[k] = mylay[k] - 1;
  }

  // ---- phase A+B per p -----------------------------------------------------------
  StageEnt *stage = s_stage + warp * 32;
  int *okv = s_ok + warp * 32;
  unsigned long long stale[ZL];  // per z-slot: bit p = all-zero/NaN series for that p
#pragma unroll
  for (int k = 0; k < ZL; ++k) stale[k] = 0ull;
  for (int pi = warp; pi < np; pi += UNC_WARPS) {
    const cplx pp = T.p[pi], aux = T.aux[pi], aux2 = T.aux2[pi];
    cplx series[ZL][UNC_MAX_NACC];
    cplx acc[ZL], fin[ZL];
#pragma unroll
    for (int k = 0; k < ZL; ++k) { acc[k] = mk(0.0, 0.0); fin[k] = mk(0.0, 0.0); }
    int seg = 0;        // 0: tanh-sinh, j>=1: Gauss-Lobatto interval j
    int next_b = N;     // first abscissa index of the next segment
    for (int base = 0; base < NA; base += 32) {
      int ok = 1;
      {
        const int idx = base + lane;
        if (idx < NA) {
          // each layer's coefficients straight into the stage entry (no 20-double entry in registers)
          const CoefAosSink sink{stage[lane].co};
          cplx eta;
          ok = ap_terms_fast_s<-1>(P, pp, aux, aux2, s_a2[idx], s_wj[idx], lay_mask, eta_max, &eta, sink) ? 1 : 0;
          stage[lane].eta = eta;
        }
        okv[lane] = ok;
      }
      const bool all_ok = __all_sync(0xffffffffu, ok);
      __syncwarp();
      const int cnt = min(32, NA - base);
      int j = 0;
      while (j < cnt) {
        const int jend = min(cnt, next_b - base);
        if (all_ok && uniform) {
          // hot loop: 4 broadcast LDS.128 + ZL x ~59 FP64 instructions per abscissa, no branches
          for (; j < jend; ++j) {
            const cplx eta = stage[j].eta;
            const Coef c = stage[j].co[L0];
#pragma unroll
            for (int k = 0; k < ZL; ++k) acc[k] = caddf(acc[k], eval_z_fast(eta, c, myz[k]));
          }
        } else if (all_ok) {
          for (; j < jend; ++j) {
            const cplx eta = stage[j].eta;
#pragma unroll
            for (int k = 0; k < ZL; ++k) acc[k] = caddf(acc[k], eval_z_fast(eta, stage[j].co[myL[k]], myz[k]));
          }
        } else {
          for (; j < jend; ++j) {
            if (okv[j]) {
#pragma unroll
              for (int k = 0; k < ZL; ++k)
                acc[k] = caddf(acc[k], eval_z_fast(stage[j].eta, stage[j].co[myL[k]], myz[k]));
            } else {
              const int id = base + j;
              const double w = s_wj[id];
              const bool sure_nan = literal_is_nan(P, stage[j].eta);
              const double nanv = __longlong_as_double(0x7ff8000000000000LL);
#pragma unroll
              for (int k = 0; k < ZL; ++k) {
                if (sure_nan) { acc[k] = mk(nanv, nanv); continue; }
                cplx v = soln_literal_one(P, T, pi, s_a2[id], myz[k], mylay[k]);
                acc[k] = caddf(acc[k], mk(w * v.re, w * v.im));
              }
            }
          }
        }
        if (base + j == next_b && next_b < NA) {
#pragma unroll
          for (int k = 0; k < ZL; ++k) {
            if (seg == 0) fin[k] = acc[k]; else series[k][seg - 1] = acc[k];
            acc[k] = mk(0.0, 0.0);
          }
          seg += 1;
          next_b += G;
        }
      }
      __syncwarp();
    }
#pragma unroll
    for (int k = 0; k < ZL; ++k) { if (seg == 0) fin[k] = acc[k]; else series[k][seg - 1] = acc[k]; }
    // phase B: Wynn-epsilon (integration.f90:125-189), totlap (driver.f90:216)
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    const cplx lt = T.lt[pi];
#pragma unroll
    for (int k = 0; k < ZL; ++k) {
      bool any = false;
      for (int j = 0; j < nacc; ++j) {
        cplx a = series[k][j];
        a = is_finite_c(a) ? a * lt : mk(nan, nan);
        series[k][j] = a;
        if (cabs_d(a) > 0.0) any = true;  // driver.f90:209
      }
      cplx infint = mk(0.0, 0.0);
      if (any) infint = wynn_any(series[k], nacc);
      else stale[k] |= 1ull << pi;
      cplx f = fin[k];
      f = is_finite_c(f) ? f * lt : mk(nan, nan);
      s_tot[(size_t)pi * ZB + 32 * k + lane] = f + infint;
    }
  }
  // per-z stale flag: OR over the warps via shared memory
  __syncthreads();
  unsigned long long *s_flag = (unsigned long long *)s_scr;  // stage no longer needed
  if (tid < ZB) s_flag[tid] = 0ull;
  __syncthreads();
#pragma unroll
  for (int k = 0; k < ZL; ++k) if (stale[k]) atomicOr(&s_flag[32 * k + lane], stale[k]);
  __syncthreads();
  unsigned long long myflag[ZL];
#pragma unroll
  for (int k = 0; k < ZL; ++k) myflag[k] = s_flag[32 * k + lane];
  __syncthreads();

  // ---- phase C: de Hoog -------------------------------------------------------------
  cplx *scr = s_scr + (size_t)warp * 3 * np;
  for (int job = warp; job < 2 * nzv; job += UNC_WARPS) {
    const int zi = job >> 1, deriv = job & 1;
    double v = dehoog_warp(P, s_tot + zi, ZB, deriv ? T.p : nullptr, tD, tee, scr, scr + np,
                           scr + 2 * np, lane);
    unsigned long long fl = 0ull;
#pragma unroll
    for (int k = 0; k < ZL; ++k) {
      unsigned long long f = __shfl_sync(0xffffffffu, myflag[k], zi & 31);
      if ((zi >> 5) == k) fl = f;
    }
    if (lane == 0) {
      const long long o = col * (long long)J.nz + z0 + zi;
      if (deriv) J.ds[o] = v * tD;  // driver.f90:228
      else {
        J.s[o] = v;
        if (J.flags) J.flags[o] = fl != 0ull ? 1 : 0;
        if (J.smask) J.smask[o] = fl;
        if (J.nstale && fl != 0ull) atomicAdd(J.nstale, 1u);
      }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------
// Eight z-slots per lane, two Laplace parameters per warp (lh_grid8_kernel below).
#ifndef UNC_WYNN_LOZ2
#define UNC_WYNN_LOZ2 0   // 1: Wynn-epsilon with two anti-diagonals in lockstep (wynn.cuh: wynn_loz2) -- measured slower
#endif
struct StageEnt8 {   // register-side image of one staged abscissa; see st8_idx for the shared-memory layout
  cplx eta;
  Coef co[3];
  cplx sp, sm;    // exp(+-eta*D), D = z spacing between a lane's slots (16 grid steps)
  cplx spx, smx;  // cp, cm of the exception slot's OTHER layer times exp(+-eta*D*kx)
  cplx sp2, sm2;  // exp(+-2*eta*D)
};
// A warp's stage in shared memory: 32 entries (16 abscissae x the warp's two Laplace parameters) of
// ST8_NF complex fields, FIELD-MAJOR: field f of abscissa j of half-warp h at complex index
// f*32 + 2*j + h.  The 32 lanes of the producer (lane <-> entry) then store 512 contiguous bytes per
// field, and the two half-warps of the consumer read one 32-byte segment -- with entry-major
// 256-byte entries every lane of a store hit the same banks (measured: 95.3 instead of 90.5
// ms/step on C5a in spite of 13 % fewer FP64 instructions in the hot loop).
constexpr int ST8_NF = (int)(sizeof(StageEnt8) / sizeof(cplx));
static_assert(ST8_NF == 16 && sizeof(Coef) == 3 * sizeof(cplx), "stage field numbering");
enum { ST8_ETA = 0, ST8_CO = 1, ST8_SP = 10, ST8_SM = 11, ST8_SPX = 12, ST8_SMX = 13, ST8_SP2 = 14, ST8_SM2 = 15 };
__host__ __device__ __forceinline__ int st8_idx(int f, int j, int h) {
  return f * 32 + 2 * j + h;
}
// complex-index step from abscissa j to j+1 and from field f to f+1
#define ST8_JSTEP 2
#define ST8_FSTEP 32

// One abscissa for the eight slots of a lane.  The slot values of the common-layer slots are
// advanced ALREADY SCALED by the coefficients, P_k = cp e^{eta z_k}, M_k = cm e^{-eta z_k}.
// Anchors at the even slots advance by exp(+-2 eta D) (two first-order recurrences, each stable
// in its own direction); an odd slot is its anchor times exp(+-eta D), fused into the
// accumulation: acc += P*E is four FMA, where advancing P and adding it are four multiply/FMA
// plus two adds -- 36 instead of 44 FP64 instructions per direction for eight slots, and
// dependent chains of three instead of seven multiplies (every slot advanced from its neighbour
// before: profiles/r02_grid_kernel_variants.txt).
// Slot KX (if >= 0) has lane-dependent layers.  Lanes on the common layer (Lx == L) treat it like
// any other slot.  The other lanes all lie on ONE other layer (the caller checks that); the stage
// holds that layer's cp, cm already multiplied by exp(+-eta D KX), so their value is
// k0' + spx*E0 + smx*E0' from the unscaled start exponentials.  Both kinds run the same eight
// FMA on lane-selected operands (before: exponentials of slot KX from slot 0 in one step, then
// the per-lane layer's coefficients -- eight instructions more).
// K0Z: k0 of the common layer is exactly zero.
template <int KX, bool K0Z>
__device__ __forceinline__ void eval8_scaled(const cplx *e, int L, int Lx, double z0, cplx *acc) {
#define ST8F(f) e[(f) * ST8_FSTEP]
  double ep, em, cc, ss, s, cs;
  int kk;
  const cplx eta = ST8F(ST8_ETA);
  Coef c;
  c.cp = ST8F(ST8_CO + 3 * L + 1);
  c.cm = ST8F(ST8_CO + 3 * L + 2);
  if (!K0Z) c.k0 = ST8F(ST8_CO + 3 * L);
  exp_pm_core(eta.re * z0, &ep, &em, &cc, &ss, &kk);
  sincos_q(eta.im * z0, &s, &cs);
  const cplx Ep = mk(ep * cs, ep * s), Em = mk(em * cs, -(em * s));
  cplx Pk = cmulf(c.cp, Ep), Mk = cmulf(c.cm, Em);
  const cplx e1p = ST8F(ST8_SP), e1m = ST8F(ST8_SM), e2p = ST8F(ST8_SP2), e2m = ST8F(ST8_SM2);
  const bool isB = (KX >= 0) && Lx != L;
#pragma unroll
  for (int k = 0; k < 8; k += 2) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int q = k + h;
      if (q != KX) {
        if (h == 0) {
          double fr = Pk.re + Mk.re, fi = Pk.im + Mk.im;
          if (!K0Z) { fr += c.k0.re; fi += c.k0.im; }
          acc[q] = mk(acc[q].re + fr, acc[q].im + fi);
        } else {
          double fr = K0Z ? acc[q].re : acc[q].re + c.k0.re;
          double fi = K0Z ? acc[q].im : acc[q].im + c.k0.im;
          fr = fma(Pk.re, e1p.re, fr);
          fr = fma(-Pk.im, e1p.im, fr);
          fr = fma(Mk.re, e1m.re, fr);
          fr = fma(-Mk.im, e1m.im, fr);
          fi = fma(Pk.re, e1p.im, fi);
          fi = fma(Pk.im, e1p.re, fi);
          fi = fma(Mk.re, e1m.im, fi);
          fi = fma(Mk.im, e1m.re, fi);
          acc[q] = mk(fr, fi);
        }
      }
      else {
        // common-layer lanes: anchor (times exp(+-eta D) at an odd slot); the others: start
        // exponentials times the pre-scaled coefficients of their layer
        const cplx one = mk(1.0, 0.0);
        const cplx k0x = ST8F(ST8_CO + 3 * Lx);
        const cplx X1 = isB ? Ep : Pk, X2 = isB ? Em : Mk;
        const cplx Y1 = isB ? ST8F(ST8_SPX) : (h == 0 ? one : e1p), Y2 = isB ? ST8F(ST8_SMX) : (h == 0 ? one : e1m);
        double fr = acc[q].re + k0x.re, fi = acc[q].im + k0x.im;
        fr = fma(X1.re, Y1.re, fr);
        fr = fma(-X1.im, Y1.im, fr);
        fr = fma(X2.re, Y2.re, fr);
        fr = fma(-X2.im, Y2.im, fr);
        fi = fma(X1.re, Y1.im, fi);
        fi = fma(X1.im, Y1.re, fi);
        fi = fma(X2.re, Y2.im, fi);
        fi = fma(X2.im, Y2.re, fi);
        acc[q] = mk(fr, fi);
      }
    }
    if (k < 6) { Pk = cmulf(Pk, e2p); Mk = cmulf(Mk, e2m); }
  }
#undef ST8F
}

// A whole staged chunk in one call, segment ends included: when the abscissa that closes a
// quadrature segment (tanh-sinh part or a J0 interval) has been added, the eight sums go to
// areas[k][seg] and restart from zero.  seg_rel = chunk-relative index one past the last
// abscissa of the current segment; boundaries at or beyond lim_rel (= end of the whole
// quadrature) are left to the caller.  Returns the new segment index.  One call per chunk
// instead of one per segment piece: the per-call cost (eight accumulators through local memory,
// pipeline fill and drain) is paid 44 instead of ~60 times per job.
template <int KX, bool K0Z>
__device__ __noinline__ int hot8_chunk(const cplx *stage /* field 0 of the half-warp's abscissa 0 */, int cnt, double z0, int L, int Lx,
                                       cplx *acc_io, cplx *areas, int seg, int seg_rel, int lim_rel, int G) {
  constexpr int AST = UNC_MAX_NACC + 1;
  cplx acc[8];
  int ncl = 0, bad = 0, nz = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) acc[k] = acc_io[k];
  for (int j = 0; j < cnt; ++j) {
    eval8_scaled<KX, K0Z>(stage + j * ST8_JSTEP, L, Lx, z0, acc);
    if (j + 1 == seg_rel && seg_rel < lim_rel) {
      // fate of the interval just closed, from the registers: bit k of `bad` = not finite, of `nz` =
      // finite and non-zero (the caller's early-stop bookkeeping; re-reading the areas from thread-
      // local memory stalled on the load)
      if (ncl == 0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const bool f = is_finite_fastc(acc[k]);
          if (!f) bad |= 1 << k;
          if (f && (acc[k].re != 0.0 || acc[k].im != 0.0)) nz |= 1 << k;
        }
      }
      ncl += 1;
#pragma unroll
      for (int k = 0; k < 8; ++k) { areas[k * AST + seg] = acc[k]; acc[k] = mk(0.0, 0.0); }
      seg += 1;
      seg_rel += G;
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) acc_io[k] = acc[k];
  return seg | (min(ncl, 3) << 8) | (bad << 12) | (nz << 20);
}


// The same for the eight-slot kernel: also exp(+-eta*Dz), its square, and for the exception slot
// kx (>= 0; other layer Lb) exp(+-eta*Dz*kx) -- as a product of the powers 1, 2, 4 of exp(+-eta*Dz)
// (relative error a few ulp on top of kx times that of the factor, which is what the slot
// recurrences carry anyway) -- times that layer's cp, cm.
struct CoefStageSink {   // a layer's coefficients straight into the lane's stage entry
  cplx *out;
  __device__ __forceinline__ void set(int L, cplx k0, cplx cp, cplx cm) const {
    out[(ST8_CO + 3 * L) * ST8_FSTEP] = k0;
    out[(ST8_CO + 3 * L + 1) * ST8_FSTEP] = cp;
    out[(ST8_CO + 3 * L + 2) * ST8_FSTEP] = cm;
  }
  __device__ __forceinline__ void wt(cplx, cplx) const {}
};
template <int MODEL>
__device__ __noinline__ int ap_terms_stage8_t(const DevParams &P, cplx p, cplx aux, cplx aux2, double a2,
                                              double w, int lay_mask, double eta_max, bool zuni,
                                              double Dz, int kx, int Lb, cplx *out /* field 0 of this lane's entry */) {
  cplx eta;
  const CoefStageSink sink{out};
  const bool ok = ap_terms_fast_s<MODEL>(P, p, aux, aux2, a2, w, lay_mask, eta_max, &eta, sink);
  out[ST8_ETA * ST8_FSTEP] = eta;
  const cplx one = mk(1.0, 0.0);
  cplx sp = one, sm = one, spx = one, smx = one;
  cplx sp2 = one, sm2 = one;
  if (zuni && ok) {
    const cbundle S = cexp_bundle(eta.re * Dz, eta.im * Dz);
    sp = S.ep;
    sm = S.em;
    sp2 = cmulf(S.ep, S.ep);
    sm2 = cmulf(S.em, S.em);
    if (kx >= 1) {
      if (kx & 1) { spx = S.ep; smx = S.em; }
      if (kx & 2) {
        spx = (kx & 1) ? cmulf(spx, sp2) : sp2;
        smx = (kx & 1) ? cmulf(smx, sm2) : sm2;
      }
      if (kx & 4) {
        const cplx p4 = cmulf(sp2, sp2), m4 = cmulf(sm2, sm2);
        spx = (kx & 3) ? cmulf(spx, p4) : p4;
        smx = (kx & 3) ? cmulf(smx, m4) : m4;
      }
    }
    if (kx >= 0) {
      // the other layer's cp, cm read back from the stage (no dynamic indexing of registers)
      spx = cmulf(out[(ST8_CO + 3 * Lb + 1) * ST8_FSTEP], spx);
      smx = cmulf(out[(ST8_CO + 3 * Lb + 2) * ST8_FSTEP], smx);
    }
  }
  out[ST8_SP * ST8_FSTEP] = sp;
  out[ST8_SM * ST8_FSTEP] = sm;
  out[ST8_SPX * ST8_FSTEP] = spx;
  out[ST8_SMX * ST8_FSTEP] = smx;
  out[ST8_SP2 * ST8_FSTEP] = sp2;
  out[ST8_SM2 * ST8_FSTEP] = sm2;
  return ok ? 1 : 0;
}

// Per-item tables, built by the whole CTA (kept out of line: once per item, not on the
// per-abscissa path): de Hoog p (invlap.f90:166-170), lapTime(p), the Moench sum / wellbore
// storage factors, and per abscissa a^2 and weight*a*J0(a rD).
__device__ __noinline__ void item_tables(const DevParams &P, const PTab &T, double *s_a2, double *s_wj, double tD,
                                         int sv, double rD, double tscale, int tid, int nthreads) {
  const int np = P.np, nacc = P.nacc, G = P.G, N = P.N;
  const int NA = N + nacc * G;
  const int na_seq = (NA + 31) & ~31;
  const double tee = P.tee_mult * tD;
  const double arg = P.j0z[sv - 1] / rD;                      // driver.f90:120
  for (int i = tid; i < np; i += nthreads) {
    const double PI = 3.141592653589793;
    double sigma = P.alpha - P.log_tol / (2.0 * tee);   // invlap.f90:166-170
    cplx p = mk(sigma, PI * (double)i / tee);
    T.p[i] = p;
    T.lt[i] = laptime_dev(P, p);
    cplx aux = mk(0.0, 0.0), aux2 = mk(0.0, 0.0);
    if (P.model == 3) {
      for (int m = 0; m < P.moench_M; ++m) aux = aux + 1.0 / (1.0 + p * (1.0 / P.moench_gamma[m]));
    } else if (P.model == 2) {
      cplx xi = P.rDw * csqrt_g(p);
      cplx K[2];
      cbesk01_dev(xi, K);
      aux = 2.0 / (p * P.CDw * K[0] + xi * K[1]);
      aux2 = p * P.tDb + 1.0;
    }
    T.aux[i] = aux;
    T.aux2[i] = aux2;
  }
  for (int idx = tid; idx < na_seq; idx += nthreads) {
    double a = 0.0, w = 0.0;
    if (idx < N) {
      a = (P.ts_T[idx] * tscale) / 2.0;  // integration.f90:62
      w = P.ts_wc[idx] * (arg / 2.0);    // driver.f90:135,154 + Richardson (linear in tmp)
    } else if (idx < NA) {
      const int node = idx - N;
      const int j = node / G, m = node - j * G;
      const double lob = P.j0z[sv + j - 1] / rD;  // driver.f90:188-193
      const double hib = P.j0z[sv + j] / rD;
      const double width = hib - lob;
      a = fma(width, P.gl_x[m], hib + lob) / 2.0;
      w = P.gl_w[m] * (width / 2.0);
    }
    s_a2[idx] = a * a;
    s_wj[idx] = (w != 0.0) ? w * (a * j0_dev(a * rD)) : 0.0;  // laplace_hankel_solutions.f90:118
  }
}

// End of a p-job for the eight slots of a lane (kept out of line: it is not part of the
// per-abscissa path and its loops would otherwise weigh on the kernel's register allocation):
// areas[k][0] = finite part, areas[k][1..nacc] = interval areas, both still without lapTime.
// Applies lapTime (laplace_hankel_solutions.f90:118), runs Wynn-epsilon where some area is
// finite and non-zero (driver.f90:209; otherwise infint = 0 and the slot is flagged stale),
// stores totlap = finint + infint (driver.f90:216) at out[16 k] unless out is null.
__device__ __noinline__ int finish8(cplx *areas, int nacc, cplx lt, cplx *out, cplx *wscr) {
  constexpr int AST = UNC_MAX_NACC + 1;
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  int stale = 0;
  for (int k = 0; k < 8; ++k) {
    cplx *ar = areas + k * AST;
    bool any = false;
    for (int j0 = 1; j0 <= nacc; j0 += 4) {       // four thread-local loads in flight at a time
      cplx v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = ar[min(j0 + u, nacc)];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (j0 + u <= nacc) {
          cplx a = v[u];
          const bool fin_a = is_finite_fastc(a);
          a = fin_a ? a * lt : mk(nan, nan);
          ar[j0 + u] = a;
          if (fin_a && (a.re != 0.0 || a.im != 0.0)) any = true;  // abs(GLarea) > 0, driver.f90:209
        }
      }
    }
    cplx infint = mk(0.0, 0.0);
    if (any) {
#if defined(UNC_SKIP_WYNN)
      infint = ar[1];
#else
      // wscr: this lane's column of the warp's (now idle) stage, [table column][32 lanes]
#if UNC_WYNN_LOZ2
      if (wscr && nacc <= 14) infint = wynn_loz2(ar + 1, nacc, wscr, 32);
#else
      if (wscr && nacc <= 14) infint = wynn_loz(ar + 1, nacc, wscr, 32);
#endif
      else infint = wynn_grid(ar + 1, nacc);
#endif
    } else stale |= 1 << k;
    cplx f = ar[0];
    f = is_finite_fastc(f) ? f * lt : mk(nan, nan);
    if (out) out[16 * k] = f + infint;
  }
  return stale;
}

// Exact per-slot evaluation of staged abscissae j..jend-1 for the eight z of a lane: the fast
// closed form with one exponential per slot where the per-(a,p) terms exist (bit j of okbits), the literal
// path otherwise.  z, layers and the padding-slot rules are rebuilt exactly as in the kernel.
__device__ __noinline__ void slow8_run(const DevParams &P, const PTab &T, int pi, const cplx *stage,
                                       unsigned okbits, int base, int j, int jend, const double *s_wj,
                                       const double *s_a2, const double *zsrc, const int *lsrc, int nzv,
                                       int hl, int L0, bool zuni, double Dz, cplx *acc) {
  double myz[8];
  int mylay[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int zi = hl + 16 * k;
    const bool v = zi < nzv;
    myz[k] = v ? zsrc[zi] : 0.0;
    mylay[k] = v ? lsrc[zi] : 0;
  }
  const bool v0 = hl < nzv;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    if (!(hl + 16 * k < nzv)) {
      mylay[k] = L0 + 1;
      myz[k] = zuni ? myz[0] + k * Dz : 0.5;
      if (!v0) myz[k] = 0.5;
    }
  }
  for (; j < jend; ++j) {
    if ((okbits >> j) & 1u) {
#pragma unroll
      for (int k = 0; k < 8; ++k)
      {
        const cplx *e = stage + j * ST8_JSTEP;
        Coef c;
        const int fb = ST8_CO + 3 * (mylay[k] - 1);
        c.k0 = e[fb * ST8_FSTEP]; c.cp = e[(fb + 1) * ST8_FSTEP]; c.cm = e[(fb + 2) * ST8_FSTEP];
        acc[k] = caddf(acc[k], eval_z_fast(e[ST8_ETA * ST8_FSTEP], c, myz[k]));
      }
    } else {
      const int id = base + j;
      const double w = s_wj[id];
      const bool sure_nan = literal_is_nan(P, stage[j * ST8_JSTEP + ST8_ETA * ST8_FSTEP]);
      const double nanv = __longlong_as_double(0x7ff8000000000000LL);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        if (sure_nan) { acc[k] = mk(nanv, nanv); continue; }
        cplx v = soln_literal_one(P, T, pi, s_a2[id], myz[k], mylay[k]);
        acc[k] = caddf(acc[k], mk(w * v.re, w * v.im));
      }
    }
  }
}

__device__ __forceinline__ int ap_terms_stage8(const DevParams &P, cplx p, cplx aux, cplx aux2, double a2,
                                               double w, int lay_mask, double eta_max, bool zuni,
                                               double Dz, int kx, int Lb, cplx *out) {
#ifdef UNC_AP_RUNTIME_MODEL
  return ap_terms_stage8_t<-1>(P, p, aux, aux2, a2, w, lay_mask, eta_max, zuni, Dz, kx, Lb, out);
#else
  switch (P.model) {   // warp-uniform
    case 0: return ap_terms_stage8_t<0>(P, p, aux, aux2, a2, w, lay_mask, eta_max, zuni, Dz, kx, Lb, out);
    case 1: return ap_terms_stage8_t<1>(P, p, aux, aux2, a2, w, lay_mask, eta_max, zuni, Dz, kx, Lb, out);
    case 2: return ap_terms_stage8_t<2>(P, p, aux, aux2, a2, w, lay_mask, eta_max, zuni, Dz, kx, Lb, out);
    case 3: return ap_terms_stage8_t<3>(P, p, aux, aux2, a2, w, lay_mask, eta_max, zuni, Dz, kx, Lb, out);
    case 4: return ap_terms_stage8_t<4>(P, p, aux, aux2, a2, w, lay_mask, eta_max, zuni, Dz, kx, Lb, out);
    case 5: return ap_terms_stage8_t<5>(P, p, aux, aux2, a2, w, lay_mask, eta_max, zuni, Dz, kx, Lb, out);
    default: return ap_terms_stage8_t<6>(P, p, aux, aux2, a2, w, lay_mask, eta_max, zuni, Dz, kx, Lb, out);
  }
#endif
}

// test hook (unc_debug_cbesk01): K0, K1 of n complex arguments by the device routine
__global__ void cbesk01_test_kernel(int n, const double *z, double *out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  cplx K[2];
  cbesk01_dev(mk(z[2 * i], z[2 * i + 1]), K);
  out[4 * i] = K[0].re; out[4 * i + 1] = K[0].im; out[4 * i + 2] = K[1].re; out[4 * i + 3] = K[1].im;
}

// DFMA-chain microbenchmark: 8 independent chains per thread
__global__ void fp64_peak_kernel(double *out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5,
         a6 = a0 + 6, a7 = a0 + 7;
  const double b = 1.0000001, c = 1e-7;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
    a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

}  // namespace unc

#include "grid8.cuh"
