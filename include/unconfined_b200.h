/* unconfined_b200 -- C ABI of the B200-native Laplace-Hankel drawdown evaluator.
 *
 * Drop-in boundary for the hot path of klkuhlm/unconfined: the loop nest
 * driver.f90:100-231 (per time: de Hoog p-values; per (t,r): tanh-sinh finite part,
 * Gauss-Lobatto/Wynn-epsilon infinite part of the Hankel inversion of
 * lap_hank_soln, then de Hoog inversion of the value and of its log-time
 * derivative).  The reference has no plugin API; its seam is the alias
 *     use laplace_hankel_solutions, only : soln => lap_hank_soln   (driver.f90:34)
 * plus the calls to dehoog/pvalues/tanh_sinh_setup/gauss_lobatto_setup/
 * wynn_epsilon/extraptozero (driver.f90:37,40) inside that loop nest, and its only
 * FFI precedent is the bind(c) interface to arb_J/arb_Y
 * (laplace_hankel_solutions.f90:310-325).  The whole nest moves behind ONE call, so
 * no per-abscissa crossing remains; read_input (driver_io.f90:30) and the output
 * code (driver.f90:234-273) stay in the Fortran driver.  fortran/unconfined_b200_mod.f90
 * holds the ISO_C_BINDING interface for every entry point below; INTEGRATION.md shows
 * the modified driver.
 *
 * Conventions: plain pointers and sizes; the caller owns every array; the library
 * copies in and out and keeps no caller pointer after return.  Every function
 * returns 0 on success or a negative UNC_ERR_* code and never exits/throws.
 * Numerical pathologies are data exactly as in the reference: NaN, +-Inf, the
 * Wynn sentinel -999999.9 (integration.f90:147), 0 for an all-zero f(p)
 * (invlap.f90:139).  There is no CPU fallback: without a CUDA device every
 * evaluation entry point returns UNC_ERR_NO_DEVICE.
 */
#ifndef UNCONFINED_B200_H
#define UNCONFINED_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UNC_OK 0
#define UNC_ERR_BAD_ARG (-1)     /* invalid size / NULL pointer / parameter out of range */
#define UNC_ERR_UNSUPPORTED (-2) /* model 6 with MNtype 0/2 (ARB / finite differences), or a table limit exceeded */
#define UNC_ERR_NO_DEVICE (-3)   /* no usable CUDA device */
#define UNC_ERR_CUDA (-4)        /* CUDA runtime failure, see unc_last_error() */
#define UNC_ERR_IO (-5)          /* deck reader: cannot open / parse */

/* flag bits returned per output point by the *_ex entry points */
#define UNC_FLAG_STALE_INFINT 1  /* every Gauss-Lobatto area of some p was 0 or non-finite, so the
                                    reference does not assign infint(p,z) and keeps the value of the
                                    last (t,r) that did (driver.f90:205-214).  Grid calls in
                                    reference-compatible mode (ts_abscissa_scale given) reproduce
                                    that (unc_set_carry); otherwise infint = 0 is used.  The flag is
                                    set in both cases. */

/* Flattened types.f90 parameter structs (invLaplace :31, invHankel :88, GaussLobatto :98,
 * TanhSinh :117, well :131, formation :145, solution :174).  Fortran: type, bind(C). */
typedef struct unc_params {
  int32_t model;        /* s%model 0..5 (types.f90:185); 6 only with mn_type = 1 (below) */
  int32_t M;            /* l%M; np = 2M+1 (driver.f90:79) */
  double alpha;         /* l%alpha (types.f90:39) */
  double tol;           /* l%tol */
  double tee_mult;      /* TEE_MULT = 2.0 (driver.f90:54) */
  int32_t time_type;    /* l%timeType (types.f90:80) */
  int32_t n_time_par;   /* size(l%timePar) */
  const double *time_par; /* l%timePar(:) (types.f90:83) */
  int32_t ts_k;         /* ts%k (types.f90:118) */
  int32_t ts_R;         /* ts%R (types.f90:120) */
  int32_t gl_nacc;      /* gl%nacc (types.f90:99) */
  int32_t gl_ord;       /* gl%ord (types.f90:106) */
  int32_t n_j0z;        /* size(h%j0z) = max(j0s)+nacc+1 (driver_io.f90:628) */
  int32_t moench_M;     /* f%MoenchM */
  const double *j0z;    /* h%j0z(:): zeros of J0 as computed by driver_io.f90:628-647 */
  const double *moench_gamma; /* f%MoenchGamma(:) (driver_io.f90:550); may be NULL if M=0 */
  double kappa;         /* f%kappa */
  double alphaD;        /* f%alphaD (driver_io.f90:541) */
  double beta;          /* f%beta -- the DIMENSIONAL beta (laplace_hankel_solutions.f90:86) */
  double lD, dD, bD, rDw; /* w%lD, w%dD, w%bD, w%rDw (driver_io.f90:544-547) */
  double l, d, Ss, rDwobs, sF; /* model 2 only: w%l, w%d, f%Ss, s%rDwobs, s%sF
                                  (laplace_hankel_solutions.f90:248-251); Ss also model 6 */
  /* model 6, Mishra-Neuman: only s%MNtype = 1, the closed-form double-precision "Malama
   * finiteness" variant mishraNeumanMalama (laplace_hankel_solutions.f90:404-442), is
   * supported; MNtype 0 (ARB quad precision) and 2 (finite differences) return
   * UNC_ERR_UNSUPPORTED.  Ignored for models 0..5. */
  int32_t mn_type;      /* s%MNtype (types.f90:181) */
  int32_t mn_reserved;  /* padding, set to 0 */
  double mn_ak;         /* f%ak, conductivity sorptive number [1/L] (driver_io.f90:159) */
  double mn_psia, mn_psik; /* f%psia, f%psik [L] */
  double mn_b;          /* f%b, initial saturated thickness [L] */
  double mn_Sy;         /* f%Sy */
} unc_params;

/* One call = driver.f90:100-231 for the whole (t, r, z) grid.
 *   tD(nt), sv(nt)   s%tD, h%sv (1-based split index, driver_io.f90:664)
 *   rD(nr)           s%rD
 *   zD(nz), zLay(nz) s%zD, s%zLay (driver_io.f90:572-586)
 *   ts_abscissa_scale  (nr,nt) column-major, or NULL.  The `arg` that scales the
 *                    tanh-sinh ABSCISSAE of each (t,r).  NULL = j0z(sv(t))/rD(r) (fresh).
 *                    The reference computes the abscissae only for the first (t,r)
 *                    (driver.f90:121-126,274): a bug-compatible caller passes
 *                    j0z(sv(1))/rD(1) in every entry.  Passing it also selects the
 *                    reference's stale-infint carry (driver.f90:205-214, t outer / r inner
 *                    order, 0 before the first assignment; see unc_set_carry).
 *   ngpu             number of GPUs to shard the (t,r) columns over; 0 = all visible
 *   totint, totintd  out, column-major (nz,nr,nt): dimensionless drawdown and its
 *                    log-time derivative (driver.f90:221,228)
 */
int unc_eval_grid(const unc_params *prm, int32_t nt, const double *tD, const int32_t *sv,
                  int32_t nr, const double *rD, int32_t nz, const double *zD,
                  const int32_t *zLay, const double *ts_abscissa_scale, int32_t ngpu,
                  double *totint, double *totintd);
int unc_eval_grid_ex(const unc_params *prm, int32_t nt, const double *tD, const int32_t *sv,
                     int32_t nr, const double *rD, int32_t nz, const double *zD,
                     const int32_t *zLay, const double *ts_abscissa_scale, int32_t ngpu,
                     double *totint, double *totintd, int32_t *flags /* (nz,nr,nt) or NULL */);

/* Same computation for a flattened list of n independent (r,z,t) points (no carry between
 * points: a stale infint is 0 + flag). */
int unc_eval_points(const unc_params *prm, int64_t n, const double *tD, const int32_t *sv,
                    const double *rD, const double *zD, const int32_t *zLay,
                    const double *ts_abscissa_scale /* (n) or NULL */, int32_t ngpu, double *s,
                    double *ds);
int unc_eval_points_ex(const unc_params *prm, int64_t n, const double *tD, const int32_t *sv,
                       const double *rD, const double *zD, const int32_t *zLay,
                       const double *ts_abscissa_scale, int32_t ngpu, double *s, double *ds,
                       int32_t *flags);

/* Exact screen-averaged drawdown of n screened observation wells (no reference equivalent;
 * the reference averages zOrd point values with the rule of driver.f90:236-239).
 * Screen i is (tD[i], rD[i], zbot[i], ztop[i]) with 0 <= zbot < ztop <= 1 in dimensionless zD.
 * Its result is the point algorithm unchanged (tanh-sinh finite part, Gauss-Lobatto/Wynn
 * infinite part, de Hoog of the value and of p*F) with the integrand f(a,p,z) replaced by its
 * mean over [zbot, ztop]:
 *   - the screen is split at the layer boundaries 1-lD and 1-dD (those of unc_zlay) into at
 *     most three segments [u_i, v_i] in layers L_i; empty segments are dropped;
 *   - mean = sum_i (v_i-u_i)/(ztop-zbot) * mean_i;
 *   - mean_i = the layer function of L_i at m = (u_i+v_i)/2 with every z-dependent factor
 *     (cosh(eta(z-c)), cosh(eta(c-z)), exp(+-eta z), exp(eta(z-1))) multiplied by S(eta h),
 *     h = (v_i-u_i)/2, S(x) = sinh(x)/x; constant terms unchanged.  This is exact: the integral
 *     of cosh(eta(z-c)) over [m-h, m+h] is 2h cosh(eta(m-c)) S(eta h).  Model 0 has no z
 *     dependence, so its screen mean is the point value.
 * One inversion per screen instead of one per point across the screen.  Flags and stale
 * handling are those of unc_eval_points_ex: no carry between screens, a stale infint is 0 and
 * sets UNC_FLAG_STALE_INFINT.  Screens are sharded over ngpu devices as points are.
 * UNC_ERR_BAD_ARG (before any device is touched): NULL arrays, a non-finite bound, zbot < 0,
 * ztop > 1 or zbot >= ztop.  The _device variant checks the pointers only: its bounds are
 * in device memory and must satisfy the same conditions. */
int unc_eval_screens(const unc_params *prm, int64_t n, const double *tD, const int32_t *sv,
                     const double *rD, const double *zbot, const double *ztop,
                     const double *ts_abscissa_scale /* (n) or NULL */, int32_t ngpu,
                     double *s, double *ds, int32_t *flags /* (n) or NULL */);

/* Vertical drawdown gradient at n points (no reference equivalent):
 *   gz(tD, rD, zD) = d s_D / d z_D,   dgz = d gz / d ln tD.
 * z is measured upward from the aquifer bottom and zD = 1 is the water table; head is h0 - s,
 * so the vertical specific discharge is q_z = +K_z (Hc/Lc) gz.
 * The result is the point algorithm unchanged (tanh-sinh finite part, Gauss-Lobatto/Wynn
 * infinite part, de Hoog of the value and of p*F) with the integrand f(a,p,z) replaced by
 * df/dz.  Layers are geometric and there is no zLay argument: layer 1 if zD < 1-lD, otherwise
 * layer 2 if zD < 1-dD, otherwise layer 3 (so zD = 1 is layer 3, unlike unc_zlay; with dD = 0
 * layer 3 has zero width there and its formulas equal layer 2's).  The slope is continuous
 * across 1-lD and 1-dD.  Within a layer f(z) = k0 + cp e^(eta z) + cm e^(-eta z), so
 * df/dz = eta (cp e^(eta z) - cm e^(-eta z)); past the fast-path bound the derivatives of the
 * reference's own expressions are evaluated: cosh(eta z) -> eta sinh(eta z),
 * cosh(eta(c-z)) -> -eta sinh(eta(c-z)), exp(eta(z-1)) -> eta exp(eta(z-1)), constant terms
 * (the 1 of layer 2, udp of model 4, model 0 entirely) -> 0.
 * Flags and stale handling are those of unc_eval_points_ex: no carry, a stale infint is 0 and
 * sets UNC_FLAG_STALE_INFINT.  So model 0 returns gz = dgz = 0 with the flag set (every area is
 * 0), as does Hantush (models 1, 2) at zD = 0.  Points are sharded over ngpu devices.
 * UNC_ERR_BAD_ARG (before any device is touched): NULL arrays, a non-finite zD or one outside
 * [0, 1].  The _device variant checks the pointers only: its zD are in device memory and must
 * satisfy the same conditions. */
int unc_eval_points_dz(const unc_params *prm, int64_t n, const double *tD, const int32_t *sv,
                       const double *rD, const double *zD,
                       const double *ts_abscissa_scale /* (n) or NULL */, int32_t ngpu,
                       double *gz, double *dgz, int32_t *flags /* (n) or NULL */);

/* Device-resident variants: every array pointer is a DEVICE pointer on the current
 * device (unc_set_device), work is enqueued on `stream` (a cudaStream_t, NULL = default
 * stream) and the call returns without synchronising -- except unc_eval_grid_device with
 * d_ts_abscissa_scale given, whose carry post-pass reads two counters back (it synchronises
 * `stream`).  Scratch, tables and counters are kept per stream: calls on different streams may
 * overlap.  unc_params and the small arrays it points to stay on the host. */
int unc_eval_grid_device(const unc_params *prm, int32_t nt, const double *d_tD,
                         const int32_t *d_sv, int32_t nr, const double *d_rD, int32_t nz,
                         const double *d_zD, const int32_t *d_zLay,
                         const double *d_ts_abscissa_scale, double *d_totint, double *d_totintd,
                         int32_t *d_flags, void *stream);
int unc_eval_points_device(const unc_params *prm, int64_t n, const double *d_tD,
                           const int32_t *d_sv, const double *d_rD, const double *d_zD,
                           const int32_t *d_zLay, const double *d_ts_abscissa_scale, double *d_s,
                           double *d_ds, int32_t *d_flags, void *stream);
int unc_eval_screens_device(const unc_params *prm, int64_t n, const double *d_tD,
                            const int32_t *d_sv, const double *d_rD, const double *d_zbot,
                            const double *d_ztop, const double *d_ts_abscissa_scale, double *d_s,
                            double *d_ds, int32_t *d_flags, void *stream);
int unc_eval_points_dz_device(const unc_params *prm, int64_t n, const double *d_tD,
                              const int32_t *d_sv, const double *d_rD, const double *d_zD,
                              const double *d_ts_abscissa_scale, double *d_gz, double *d_dgz,
                              int32_t *d_flags, void *stream);

/* Set-up tables exactly as the reference computes them on the host (so that the
 * Fortran driver may also obtain them from here):
 *   unc_j0_zeros      driver_io.f90:628-647
 *   unc_split_index   driver_io.f90:658-664
 *   unc_zlay          driver_io.f90:572-586 */
int unc_j0_zeros(int32_t terms, double *j0z);
int unc_split_index(int32_t nt, const double *tD, int32_t j0s_a, int32_t j0s_b, int32_t *sv);
int unc_zlay(int32_t nz, const double *zD, double lD, double dD, int32_t *zLay);

/* Device selection / information / teardown. */
int unc_device_count(int32_t *ngpu);
int unc_set_device(int32_t device);       /* device used by the *_device entry points and by ngpu=1 */
int unc_device_info(int32_t *ngpu, double *fp64_peak_flops /* nominal: SMs*64*2*clock */);
int unc_measure_fp64_peak(double *flops); /* DFMA-chain microbenchmark on the current device */
int unc_kernel_launch_count(int64_t *n);  /* kernels launched by this library so far */
int unc_shutdown(void);                   /* frees cached device buffers */
int unc_release_stream(void *stream);     /* frees what the *_device entry points cached for this stream */
int unc_set_carry(int32_t on);            /* default 1: see UNC_FLAG_STALE_INFINT */
int unc_debug_cbesk01(int32_t n, const double *z /* [2n] */, double *out /* [4n]: K0, K1 */); /* test hook: device cbknu */
int unc_debug_force_kernel(int32_t which);/* test hook: 0 auto, 1 point kernel, 2 grid kernels,
                                             3 lanes<->z grid kernel even for nz >= 33,
                                             4 128-z persistent kernel from nz = 32 */
const char *unc_last_error(void);         /* thread-local message for the last failure */
const char *unc_version(void);

#ifdef __cplusplus
}
#endif
#endif /* UNCONFINED_B200_H */
