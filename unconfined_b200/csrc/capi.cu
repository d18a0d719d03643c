// C ABI of unconfined_b200 (include/unconfined_b200.h): host planner + launches.
//
// Host side = what the reference computes once per run on the host before its loop
// nest (driver.f90:79-91 level tables, integration.f90:31-120 quadrature set-up), plus
// sharding of the (t,r) columns over the GPUs of one box and the copies in/out.
// There is deliberately no CPU evaluation path here.
#include <cuda_runtime.h>
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <limits>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/unconfined_b200.h"
#include "kernels.cuh"
#include "carry.cuh"

namespace {

thread_local std::string g_err;
std::mutex g_mutex;                 // calls are serialised (SURVEY 8b: threading)
std::atomic<long long> g_launches{0};
int g_device = 0;

int fail(int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CK(call)                                                                      \
  do {                                                                                \
    cudaError_t e_ = (call);                                                          \
    if (e_ != cudaSuccess)                                                            \
      return fail(UNC_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                  __FILE__, __LINE__);                                                \
  } while (0)

// ---- host set-up tables -----------------------------------------------------
// integration.f90:45-62: weights of tanh-sinh level k (renormalised to sum 2) and,
// for the densest level, T = tanh(u2)+1 so that a = T*s/2.
void tanh_sinh_level(int k, std::vector<double> &w, std::vector<double> *T) {
  const int N = (1 << k) - 1, r = (N - 1) / 2;
  const double h = 4.0 / (double)(1 << k);
  const double piov2 = 2.0 * std::atan(1.0);
  w.resize(N);
  if (T) T->resize(N);
  double sum = 0.0;
  for (int i = -r; i <= r; ++i) {
    const double u1 = piov2 * std::cosh(h * i), u2 = piov2 * std::sinh(h * i);
    const double c = std::cosh(u2);
    w[i + r] = u1 / (c * c);
    if (T) (*T)[i + r] = std::tanh(u2) + 1.0;
  }
  for (int i = 0; i < N; ++i) sum += w[i];
  for (int i = 0; i < N; ++i) w[i] = 2.0 * w[i] / sum;
}

// integration.f90:192-237 is linear in y for fixed x: return the coefficient of each
// y_j in the value extrapolated to x=0 (Neville on unit vectors, long double).
std::vector<long double> richardson_coeffs(const std::vector<double> &x) {
  const int n = (int)x.size();
  std::vector<long double> coef(n);
  for (int u = 0; u < n; ++u) {
    std::vector<long double> c(n, 0.0L), d(n, 0.0L);
    c[u] = d[u] = 1.0L;
    int ns = 1;
    for (int i = 2; i <= n; ++i) if (x[i - 1] < x[ns - 1]) ns = i;
    long double y = c[ns - 1];
    ns -= 1;
    for (int m = 1; m <= n - 1; ++m) {
      for (int i = 1; i <= n - m; ++i) {
        long double den = (c[i] - d[i - 1]) / ((long double)x[i - 1] - (long double)x[i + m - 1]);
        d[i - 1] = (long double)x[i + m - 1] * den;
        c[i - 1] = (long double)x[i - 1] * den;
      }
      long double dy;
      if (2 * ns < n - m) dy = c[ns];
      else { dy = d[ns - 1]; ns -= 1; }
      y += dy;
    }
    coef[u] = y;
  }
  return coef;
}

// integration.f90:70-120: interior Gauss-Lobatto nodes and weights
void gauss_lobatto(int ord, std::vector<double> &gx, std::vector<double> &gw) {
  const int N = ord - 1, N1 = N + 1;
  const double pi = 4.0 * std::atan(1.0);
  std::vector<double> x(ord), xold(ord, 2.0), Pn(ord), Pn1(ord);
  for (int i = 0; i <= N; ++i) x[i] = std::cos(pi * i / N);
  for (;;) {
    double mx = 0.0;
    for (int i = 0; i < ord; ++i) mx = std::max(mx, std::fabs(x[i] - xold[i]));
    if (!(mx > std::numeric_limits<double>::epsilon())) break;
    xold = x;
    for (int i = 0; i < ord; ++i) {
      // Legendre recurrence up to P_N (Pn) and P_{N-1} (Pn1)
      double pkm1 = 1.0, pk = x[i];
      for (int k = 2; k <= N; ++k) {
        double pkp1 = ((2 * k - 1) * x[i] * pk - (k - 1) * pkm1) / k;
        pkm1 = pk;
        pk = pkp1;
      }
      Pn[i] = pk;
      Pn1[i] = pkm1;
      x[i] = xold[i] - (x[i] * pk - pkm1) / (N1 * pk);
    }
  }
  gx.resize(ord - 2);
  gw.resize(ord - 2);
  for (int i = 1; i < ord - 1; ++i) {
    gx[i - 1] = x[i];
    gw[i - 1] = 2.0 / ((double)(N * N1) * (Pn[i] * Pn[i]));
  }
}

struct HostPlan {
  unc::DevParams P;
  std::vector<double> blob;  // ts_T | ts_wc | gl_x | gl_w | j0z | time_par | moench_gamma
  size_t off_T, off_wc, off_glx, off_glw, off_j0z, off_tp, off_mg, off_lw;
};

int build_plan(const unc_params *prm, HostPlan &hp) {
  if (!prm) return fail(UNC_ERR_BAD_ARG, "prm is NULL");
  if (prm->model < 0 || prm->model > 6) return fail(UNC_ERR_BAD_ARG, "invalid model %d", prm->model);
  if (prm->model == 6) {
    if (prm->mn_type == 0 || prm->mn_type == 2)
      return fail(UNC_ERR_UNSUPPORTED, "model 6 MNtype %d (ARB quad precision / finite-difference "
                  "Mishra-Neuman) is out of scope; only MNtype 1 is supported", prm->mn_type);
    if (prm->mn_type != 1) return fail(UNC_ERR_BAD_ARG, "invalid MNtype %d (driver_io.f90:272)", prm->mn_type);
    if (!(prm->mn_b > 0.0) || !(prm->Ss > 0.0) || !(prm->mn_ak > 0.0))
      return fail(UNC_ERR_BAD_ARG, "model 6 needs mn_b, Ss, mn_ak > 0");
  }
  if (prm->M < 2) return fail(UNC_ERR_BAD_ARG, "de Hoog M must be >= 2 (driver_io.f90:308)");
  if (prm->M > 31) return fail(UNC_ERR_UNSUPPORTED, "de Hoog M > 31 not supported (2M+1 <= 63)");
  if (prm->ts_R < 1 || prm->ts_k - prm->ts_R < 2)
    return fail(UNC_ERR_BAD_ARG, "tanh-sinh needs R>=1 and k-R>=2 (driver_io.f90:317-328)");
  if (prm->ts_k > 12) return fail(UNC_ERR_UNSUPPORTED, "tanh-sinh k > 12 not supported");
  if (prm->gl_nacc < 2 || prm->gl_nacc > UNC_MAX_NACC)
    return fail(UNC_ERR_UNSUPPORTED, "gl_nacc must be in 2..%d", UNC_MAX_NACC);
  if (prm->gl_ord < 3) return fail(UNC_ERR_BAD_ARG, "gl_ord must be >= 3");
  if (!prm->j0z || prm->n_j0z < prm->gl_nacc + 2)
    return fail(UNC_ERR_BAD_ARG, "j0z must hold at least nacc+2 zeros");
  if (prm->time_type == 0 || prm->time_type > 8)
    return fail(UNC_ERR_BAD_ARG, "invalid time_type %d (time.f90:47-121)", prm->time_type);
  {
    int need = 2;
    if (prm->time_type < 0 && prm->time_type >= -100) need = 2 * (-prm->time_type) + 1;
    if (prm->time_type <= -101) need = 2 * (-prm->time_type - 100) + 1;
    if (!prm->time_par || prm->n_time_par < need)
      return fail(UNC_ERR_BAD_ARG, "time_par needs %d entries for time_type %d", need, prm->time_type);
  }
  if (prm->model == 3 && (prm->moench_M < 1 || !prm->moench_gamma))
    return fail(UNC_ERR_BAD_ARG, "model 3 needs moench_M >= 1 (driver_io.f90:144-149)");
  if (!(prm->tol > 0.0)) return fail(UNC_ERR_BAD_ARG, "tol must be > 0");

  unc::DevParams &P = hp.P;
  std::memset(&P, 0, sizeof P);
  P.model = prm->model;
  P.M = prm->M;
  P.np = 2 * prm->M + 1;            // driver.f90:79
  P.N = (1 << prm->ts_k) - 1;       // driver.f90:81
  P.R = prm->ts_R;
  P.G = prm->gl_ord - 2;
  P.nacc = prm->gl_nacc;
  P.gl_rounds = (P.nacc * P.G + 31) / 32;
  if (P.gl_rounds > P.G)
    return fail(UNC_ERR_UNSUPPORTED, "nacc*(ord-2)/32 must not exceed ord-2 (nacc <= 32)");
  P.nts_pad = ((P.N + 31) / 32) * 32;
  P.time_type = prm->time_type;
  P.n_time_par = prm->n_time_par;
  P.moench_M = prm->model == 3 ? prm->moench_M : 0;
  P.n_j0z = prm->n_j0z;
  P.alpha = prm->alpha;
  P.log_tol = std::log(prm->tol);   // invlap.f90:77,166 (glibc log, as the reference)
  P.tee_mult = prm->tee_mult;
  P.kappa = prm->kappa;
  P.alphaD = prm->alphaD;
  P.beta = prm->beta;
  P.lD = prm->lD; P.dD = prm->dD; P.bD = prm->bD; P.rDw = prm->rDw;
  P.lD1 = 1.0 - prm->lD;            // laplace_hankel_solutions.f90:159-160
  P.dD1 = 1.0 - prm->dD;
  if (prm->model == 6) {
    // laplace_hankel_solutions.f90:424-431 (run constants of mishraNeumanMalama)
    const double beta0 = prm->mn_ak * prm->mn_b;
    const double phiDa = prm->mn_psia / prm->mn_b;
    const double phiDk = prm->mn_psik / prm->mn_b;
    P.mn_vartheta = beta0 * prm->mn_Sy / (prm->Ss * prm->mn_b) * std::exp(-beta0 * (phiDa - phiDk));
    P.mn_u0 = beta0 / 2.0;
  }
  if (prm->model == 2) {
    const double PI = 4.0 * std::atan(1.0);
    P.CDw = prm->rDw * prm->rDw / (2.0 * (prm->l - prm->d) * prm->Ss);   // :248
    P.tDb = PI * prm->rDwobs * prm->rDwobs / (prm->sF * prm->Ss);        // :251
  }
  // quadrature tables
  std::vector<double> T, wc(P.N, 0.0), w;
  std::vector<double> hv(P.R);
  std::vector<std::vector<double>> lw(P.R);
  for (int m = 1; m <= P.R; ++m) {
    int kv = prm->ts_k - P.R + m;                    // driver.f90:86-91
    hv[m - 1] = 4.0 / (double)(1 << kv);
    tanh_sinh_level(kv, lw[m - 1], m == P.R ? &T : nullptr);
  }
  std::vector<long double> rc(P.R, 1.0L);
  if (P.R > 1) rc = richardson_coeffs(hv);
  for (int nn = 1; nn <= P.N; ++nn) {
    long double acc = 0.0L;
    for (int j = 1; j <= P.R; ++j) {
      int step = 1 << (P.R - j);                     // driver.f90:150
      if (nn % step == 0) acc += rc[j - 1] * (long double)lw[j - 1][nn / step - 1];
    }
    wc[nn - 1] = (double)acc;
  }
  std::vector<double> gx, gw;
  gauss_lobatto(prm->gl_ord, gx, gw);
  auto push = [&](const double *src, size_t n) {
    size_t off = hp.blob.size();
    hp.blob.insert(hp.blob.end(), src, src + n);
    if (hp.blob.size() % 2) hp.blob.push_back(0.0);
    return off;
  };
  hp.blob.clear();
  hp.off_T = push(T.data(), T.size());
  hp.off_wc = push(wc.data(), wc.size());
  hp.off_glx = push(gx.data(), gx.size());
  hp.off_glw = push(gw.data(), gw.size());
  hp.off_j0z = push(prm->j0z, prm->n_j0z);
  hp.off_tp = push(prm->time_par, prm->n_time_par);
  double zero = 0.0;
  hp.off_mg = P.moench_M ? push(prm->moench_gamma, P.moench_M) : push(&zero, 1);
  {
    std::vector<double> all;   // the levels' own weights (error-budget builds, UNC_BUDGET_NEVILLE)
    for (int m = 0; m < P.R; ++m) all.insert(all.end(), lw[m].begin(), lw[m].end());
    hp.off_lw = push(all.data(), all.size());
    P.ts_k = prm->ts_k;
  }
  return UNC_OK;
}

// The plan depends on the parameter struct only (quadrature set-up: ~250 libm calls and a
// Newton iteration, ~0.1 ms -- a third of the wall time of a 100-point deck), so the last one
// is kept.  Callers hold g_mutex.
struct PlanCache {
  bool valid = false;
  unc_params key;
  std::vector<double> j0z, tp, mg;
  HostPlan plan;
};
PlanCache g_plan_cache;

int make_plan(const unc_params *prm, HostPlan &hp) {
  if (!prm) return fail(UNC_ERR_BAD_ARG, "prm is NULL");
  PlanCache &c = g_plan_cache;
  if (c.valid) {
    unc_params k = *prm;
    k.j0z = nullptr; k.time_par = nullptr; k.moench_gamma = nullptr;
    const bool same = std::memcmp(&k, &c.key, sizeof k) == 0 && prm->j0z && prm->time_par &&
                      (int)c.j0z.size() == prm->n_j0z && (int)c.tp.size() == prm->n_time_par &&
                      std::equal(c.j0z.begin(), c.j0z.end(), prm->j0z) &&
                      std::equal(c.tp.begin(), c.tp.end(), prm->time_par) &&
                      (c.mg.empty() || (prm->moench_gamma && std::equal(c.mg.begin(), c.mg.end(), prm->moench_gamma)));
    if (same) { hp = c.plan; return UNC_OK; }
  }
  int rc = build_plan(prm, hp);
  if (rc) return rc;
  std::memset(&c.key, 0, sizeof c.key);
  c.key = *prm;
  c.key.j0z = nullptr; c.key.time_par = nullptr; c.key.moench_gamma = nullptr;
  c.j0z.assign(prm->j0z, prm->j0z + prm->n_j0z);
  c.tp.assign(prm->time_par, prm->time_par + prm->n_time_par);
  c.mg.clear();
  if (hp.P.moench_M > 0) c.mg.assign(prm->moench_gamma, prm->moench_gamma + hp.P.moench_M);
  c.plan = hp;
  c.valid = true;
  return UNC_OK;
}

// ---- per-device context -------------------------------------------------------
struct DevBuf {
  void *ptr = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return UNC_OK;
    if (ptr) cudaFree(ptr);
    ptr = nullptr; cap = 0;
    size_t want = std::max(bytes, (size_t)4096);
    CK(cudaMalloc(&ptr, want));
    cap = want;
    return UNC_OK;
  }
  void release() { if (ptr) cudaFree(ptr); ptr = nullptr; cap = 0; }
};

// Everything a launch writes lives in the resources of the stream it is enqueued on: the
// persistent grid kernel's totlap scratch and work counter, the uploaded tables and the
// carry post-pass buffers.  Two calls on different streams therefore never share mutable
// device state; calls on one stream are ordered by the stream.
struct StreamRes {
  DevBuf tables, scratch, counter;
  std::vector<double> blob_cached;
  // carry post-pass
  DevBuf mask, slot, need, src_slot, list, src_list, fix_src, fix_val, fix_out, counts, cin;
  DevBuf order, bins;   // cost-ordered unit list of large point sets
  void release() {
    for (DevBuf *b : {&tables, &scratch, &counter, &mask, &slot, &need, &src_slot, &list, &src_list,
                      &fix_src, &fix_val, &fix_out, &counts, &cin, &order, &bins})
      b->release();
  }
};

struct DevCtx {
  bool init = false;
  cudaStream_t stream = nullptr;
  DevBuf in, out;
  int sm_count = 0;
  bool smem_set[32] = {false};
  std::map<cudaStream_t, StreamRes> res;
};
DevCtx g_ctx[16];
std::atomic<int> g_carry{1};   // unc_set_carry
std::atomic<int> g_force{0};   // unc_debug_force_kernel: 0 auto, 1 point, 2 grid, 3 grid (lanes<->z kernel only), 4 grid (128-z kernel from nz = 32)
// columns of at least this many z go to the 128-z persistent kernel (its padding slots idle):
// measured on 1024 r x nz x 2 t of C5a, lanes<->z kernel vs 128-z kernel: nz=32 17.2 vs 19.2 ms,
// nz=40 30.9 vs 19.9, nz=48 31.3 vs 19.8, nz=64 32.4 vs 19.7, nz=96 60.1 vs 20.5
// (profiles/r02_nz_crossover.txt; before the padding slots were taken out of the early-stop
// condition the 128-z kernel needed 54 ms below nz = 64 and the crossover was 64)
#ifndef UNC_GRID8_MIN_NZ
#define UNC_GRID8_MIN_NZ 33
#endif

// the library switches devices internally; the caller's current device is restored on return
struct DeviceGuard {
  int prev = -1;
  DeviceGuard() { if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; } }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

int ensure_ctx(int dev) {
  if (dev < 0 || dev >= 16) return fail(UNC_ERR_BAD_ARG, "device %d out of range", dev);
  CK(cudaSetDevice(dev));
  DevCtx &c = g_ctx[dev];
  if (!c.init) {
    CK(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    CK(cudaDeviceGetAttribute(&c.sm_count, cudaDevAttrMultiProcessorCount, dev));
    c.init = true;
  }
  return UNC_OK;
}

int upload_tables(StreamRes &r, HostPlan &hp, cudaStream_t st) {
  size_t bytes = hp.blob.size() * sizeof(double);
  if (bytes > r.tables.cap) r.blob_cached.clear();
  int rc = r.tables.ensure(bytes);
  if (rc) return rc;
  if (r.blob_cached != hp.blob) {
    // tables are a few KB: synchronous semantics are fine, but stay on the job's stream
    CK(cudaMemcpyAsync(r.tables.ptr, hp.blob.data(), bytes, cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));
    r.blob_cached = hp.blob;
  }
  const double *b = (const double *)r.tables.ptr;
  hp.P.ts_T = b + hp.off_T;
  hp.P.ts_wc = b + hp.off_wc;
  hp.P.gl_x = b + hp.off_glx;
  hp.P.gl_w = b + hp.off_glw;
  hp.P.j0z = b + hp.off_j0z;
  hp.P.time_par = b + hp.off_tp;
  hp.P.moench_gamma = b + hp.off_mg;
  hp.P.ts_lw = b + hp.off_lw;
  return UNC_OK;
}

template <int ZT, int PT>
int launch_point(int dev, const unc::DevParams &P, const unc::Job &J, cudaStream_t st, long long nunits) {
  const int na = P.nts_pad + P.gl_rounds * 32;
  const size_t smem = unc::point_smem_bytes(P.np, P.nacc, na, ZT, PT);
  if (smem > 227 * 1024) return fail(UNC_ERR_UNSUPPORTED, "shared memory need %zu B exceeds 227 KB", smem);
  DevCtx &c = g_ctx[dev];
  if (!c.smem_set[ZT + 4 * (PT - 1)]) {
    CK(cudaFuncSetAttribute(unc::lh_point_kernel<ZT, PT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            227 * 1024));
    c.smem_set[ZT + 4 * (PT - 1)] = true;
  }
  const long long nblk = (nunits + PT - 1) / PT;
  if (nblk <= 0) return UNC_OK;
  if (nblk > 2147483647LL) return fail(UNC_ERR_UNSUPPORTED, "too many work items (%lld)", nblk);
  unc::lh_point_kernel<ZT, PT><<<(unsigned)nblk, UNC_PTHREADS, smem, st>>>(P, J);
  g_launches++;
  CK(cudaGetLastError());
  return UNC_OK;
}

// ZT z-values of one column per work unit; for ZT = 1 (scattered points, time series) a CTA can
// take several units so that its Wynn and de Hoog phases are fuller (UNC_POINT_PTMAX; measured
// below: one unit per CTA is best once large point sets are cost-ordered)
template <int ZT>
int launch_zt(int dev, const unc::DevParams &P, const unc::Job &J, cudaStream_t st, long long nunits_fix = -1) {
  const long long ntiles = (J.nz + ZT - 1) / ZT;
  const long long nunits = nunits_fix >= 0 ? nunits_fix : J.ncol * ntiles;
  if (ZT == 1) {
#ifndef UNC_POINT_PTMAX
#define UNC_POINT_PTMAX 1   // C5b, ms per 2^17 points, one / two / four units per CTA: 290 / 287 / 318 in input order
#endif                      // (instruction-cache misses), 278.5 / 281.7 / 290.2 with cost-ordered units
#ifndef UNC_BUDGET_SEQSUM
    const int na = P.nts_pad + P.gl_rounds * 32;
    const int cta_per_sm = 16 / UNC_PWARPS;
    const long long fill = (long long)cta_per_sm * g_ctx[dev].sm_count;
    if (UNC_POINT_PTMAX >= 4 && nunits >= 4 * fill &&
        cta_per_sm * unc::point_smem_bytes(P.np, P.nacc, na, 1, 4) <= 227 * 1024)
      return launch_point<1, 4>(dev, P, J, st, nunits);
    if (UNC_POINT_PTMAX >= 2 && nunits >= 2 * fill &&
        cta_per_sm * unc::point_smem_bytes(P.np, P.nacc, na, 1, 2) <= 227 * 1024)
      return launch_point<1, 2>(dev, P, J, st, nunits);
#endif
    return launch_point<1, 1>(dev, P, J, st, nunits);
  }
  return launch_point<ZT, 1>(dev, P, J, st, nunits);
}

template <int ZL>
int launch_grid_zl(int dev, const unc::DevParams &P, const unc::Job &J, cudaStream_t st) {
  const int NA = P.N + P.nacc * P.G;
  const size_t smem = unc::grid_smem_bytes(P.np, (NA + 31) & ~31, ZL);
  if (smem > 227 * 1024) return fail(UNC_ERR_UNSUPPORTED, "shared memory need %zu B exceeds 227 KB", smem);
  DevCtx &c = g_ctx[dev];
  if (!c.smem_set[10 + ZL]) {
    CK(cudaFuncSetAttribute(unc::lh_grid_kernel<ZL>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    c.smem_set[10 + ZL] = true;
  }
  const long long nblk = J.ncol * ((J.nz + 32 * ZL - 1) / (32 * ZL));
  if (nblk <= 0) return UNC_OK;
  if (nblk > 2147483647LL) return fail(UNC_ERR_UNSUPPORTED, "too many work items (%lld)", nblk);
  unc::lh_grid_kernel<ZL><<<(unsigned)nblk, UNC_THREADS, smem, st>>>(P, J);
  g_launches++;
  CK(cudaGetLastError());
  return UNC_OK;
}

// 128 z per work item, persistent CTAs drawing items from an atomic counter, eight z-slots per
// lane and two Laplace parameters per warp; totlap in a per-CTA global scratch slot
// (kernels.cuh: lh_grid8_kernel).  Scratch and counter belong to the launch stream.
// 128 z per work item, persistent CTAs drawing items from an atomic counter, eight z-slots per
// lane and two Laplace parameters per warp; totlap and the items' tables in per-CTA global
// scratch slots (grid8.cuh: lh_grid8_kernel).  Scratch and counter belong to the launch stream.
template <int NW>
int launch_grid8_nw(int dev, StreamRes &r, const unc::DevParams &P, const unc::Job &J, cudaStream_t st) {
  const int NA = P.N + P.nacc * P.G, na_seq = (NA + 31) & ~31;
  const size_t smem = unc::grid8_smem_bytes(P.np, na_seq, NW);
  if (smem > 227 * 1024) return fail(UNC_ERR_UNSUPPORTED, "shared memory need %zu B exceeds 227 KB", smem);
  DevCtx &c = g_ctx[dev];
  if (!c.smem_set[20]) {
    CK(cudaFuncSetAttribute(unc::lh_grid8_kernel<NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    c.smem_set[20] = true;
  }
  const long long nitems = J.ncol * ((J.nz + 127) / 128);
  if (nitems <= 0) return UNC_OK;
  if (nitems > 4000000000LL) return fail(UNC_ERR_UNSUPPORTED, "too many work items (%lld)", nitems);
  int occ = 1;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, unc::lh_grid8_kernel<NW>, NW * 32, smem));
  if (occ < 1) occ = 1;
  const int grid = (int)std::min<long long>(nitems, (long long)c.sm_count * occ);
  // per CTA: three totlap slots, two table slots, three stale-mask slots
  int rc = r.scratch.ensure(unc::grid8_scratch_bytes(P.np, na_seq, grid));
  if (rc) return rc;
  rc = r.counter.ensure(256);
  if (rc) return rc;
  // armed on the launch stream before every launch (the kernel also re-arms it when it ends, so
  // that a profiler's replays of the launch start from zero as well)
  CK(cudaMemsetAsync(r.counter.ptr, 0, 256, st));
  unc::lh_grid8_kernel<NW><<<grid, NW * 32, smem, st>>>(P, J, (unc::cplx *)r.scratch.ptr,
                                                         (unsigned int *)r.counter.ptr);
  g_launches++;
  CK(cudaGetLastError());
  return UNC_OK;
}

int launch_grid(int dev, StreamRes &r, const unc::DevParams &P, const unc::Job &J, cudaStream_t st) {
  const bool small_only = g_force.load() == 3;
  if ((J.nz >= UNC_GRID8_MIN_NZ && !small_only) || (g_force.load() == 4 && J.nz >= 32))
    return launch_grid8_nw<UNC_GRID8_NW>(dev, r, P, J, st);
  // two z per lane (64 z per CTA) halves the per-(a,p) work per point; keep one z per lane
  // for short columns and when the larger totlap tile would not fit twice per SM
  if (J.nz > 32 && P.np <= 53) return launch_grid_zl<2>(dev, P, J, st);
  return launch_grid_zl<1>(dev, P, J, st);
}

// lists of 16384 or more one-z columns (points, screens, gradients) run in cost order, most
// expensive (smallest rD) first; Jo gets the order list.  Jo is left as it is for smaller lists,
// when a kernel is forced, and in UNC_NO_COST_ORDER builds.
int cost_order(StreamRes &r, const unc::Job &J, cudaStream_t st, unc::Job &Jo) {
#ifndef UNC_NO_COST_ORDER
  if (J.ncol >= 16384 && g_force.load() == 0) {
    int rc = r.order.ensure((size_t)J.ncol * sizeof(int));
    if (rc) return rc;
    if ((rc = r.bins.ensure(128 * sizeof(unsigned int)))) return rc;
    unsigned int *bins = (unsigned int *)r.bins.ptr;
    const unsigned nb = (unsigned)((J.ncol + 255) / 256);
    CK(cudaMemsetAsync(bins, 0, 128 * sizeof(unsigned int), st));
    unc::cost_hist_kernel<<<nb, 256, 0, st>>>(J.rD, J.ncol, bins);
    unc::cost_scan_kernel<<<1, 32, 0, st>>>(bins);
    unc::cost_scatter_kernel<<<nb, 256, 0, st>>>(J.rD, J.ncol, bins, (int *)r.order.ptr);
    g_launches += 3;
    Jo.fix_mode = 3;
    Jo.fix_n = J.ncol;
    Jo.fix_list = (const int *)r.order.ptr;
  }
#endif
  return UNC_OK;
}

// kernel selection: lanes<->z (grid kernels) once a column has enough z to fill most of a
// warp; otherwise lanes<->abscissae (point kernel).  unc_debug_force_kernel overrides (tests).
int launch(int dev, StreamRes &r, const unc::DevParams &P, const unc::Job &J, cudaStream_t st) {
  const int force = g_force.load();
  bool grid = J.nz >= 12;
  // a small contour grid (fewer column CTAs than SMs) is a latency problem: the point kernel
  // spreads it over nz/4 times as many CTAs (hantush-contours deck, 30 r x 20 z: 6.9 ms -> <1 ms)
  if (grid && J.nz < 64 && J.ncol * ((J.nz + 31) / 32) < (long long)g_ctx[dev].sm_count) grid = false;
  if (force == 1) grid = false;
  if (force == 2 || force == 3 || force == 4) grid = true;
  if (grid) return launch_grid(dev, r, P, J, st);
  // large scattered point sets: most expensive (smallest rD) first, see carry.cuh
  if (J.zstride == 1 && J.nz == 1 && J.fix_mode == 0 && J.ncol < 2147483647LL && force == 0) {
    unc::Job Jo = J;
    int rc = cost_order(r, J, st, Jo);
    if (rc) return rc;
    if (Jo.fix_mode == 3) return launch_zt<1>(dev, P, Jo, st, J.ncol);
  }
#ifdef UNC_BUDGET_SEQSUM
  return launch_zt<1>(dev, P, J, st);   // error-budget builds: the sequential sums exist for one z per CTA only
#endif
  // the largest z tile whose shared memory fits: at the top of the accepted settings (M >= 27,
  // 32 Wynn terms, k = 12, ord = 100) four z per CTA exceed 227 KB while two still fit
  const int na = P.nts_pad + P.gl_rounds * 32;
  auto fits = [&](int zt) { return unc::point_smem_bytes(P.np, P.nacc, na, zt, 1) <= 227 * 1024; };
  if (J.nz >= 4 && fits(4)) return launch_zt<4>(dev, P, J, st);
  if (J.nz >= 2 && fits(2)) return launch_zt<2>(dev, P, J, st);
  return launch_zt<1>(dev, P, J, st);
}

// one observation per CTA (kernels.cuh: lh_column_kernel): screens, with `ztop` their tops, and
// vertical gradients, with `ztop` NULL; cost-ordered
template <int KIND>
int launch_column(int dev, StreamRes &r, const unc::DevParams &P, const unc::Job &J, const double *ztop,
                  cudaStream_t st) {
  const int na = P.nts_pad + P.gl_rounds * 32;
  const size_t smem = unc::column_smem_bytes(P.np, P.nacc, na, KIND);
  if (smem > 227 * 1024) return fail(UNC_ERR_UNSUPPORTED, "shared memory need %zu B exceeds 227 KB", smem);
  DevCtx &c = g_ctx[dev];
  if (!c.smem_set[21 + KIND]) {
    CK(cudaFuncSetAttribute(unc::lh_column_kernel<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    c.smem_set[21 + KIND] = true;
  }
  if (J.ncol <= 0) return UNC_OK;
  if (J.ncol > 2147483647LL) return fail(UNC_ERR_UNSUPPORTED, "too many work items (%lld)", J.ncol);
  unc::Job Jo = J;
  int rc = cost_order(r, J, st, Jo);
  if (rc) return rc;
  unc::lh_column_kernel<KIND><<<(unsigned)J.ncol, UNC_PTHREADS, smem, st>>>(P, Jo, ztop);
  g_launches++;
  CK(cudaGetLastError());
  return UNC_OK;
}

// ---- stale-infint carry (driver.f90:205-214), see carry.cuh --------------------------------
// d_mask: per point of the WHOLE job (global column order), bit p = infint(p,z) stale.
// Jg: the global job (col0 = 0; device pointers of the inputs; s/ds = device outputs to patch
// in place, or NULL).  On return *nf_out = number of re-inverted points; if h_list/h_s/h_ds are
// given they receive the compact results (point index, s, ds).  Synchronises `st` twice.
int carry_postpass(int dev, StreamRes &r, const unc::DevParams &P, unc::Job Jg, const unsigned long long *d_mask,
                   cudaStream_t st, long long *nf_out, std::vector<int> *h_list, std::vector<double> *h_s,
                   std::vector<double> *h_ds) {
  const long long npts = Jg.ncol * (long long)Jg.nz;
  *nf_out = 0;
  if (npts <= 0) return UNC_OK;
  if (npts > 2147483647LL) return fail(UNC_ERR_UNSUPPORTED, "carry post-pass: more than 2^31 points");
  const int np = P.np, nz = Jg.nz;
  int rc;
  if ((rc = r.counts.ensure(64))) return rc;
  if ((rc = r.slot.ensure((size_t)npts * sizeof(int)))) return rc;
  if ((rc = r.list.ensure((size_t)npts * sizeof(int)))) return rc;
  unsigned int *d_cnt = (unsigned int *)r.counts.ptr;
  CK(cudaMemsetAsync(d_cnt, 0, 64, st));
  const int TB = 256;
  const unsigned nb = (unsigned)((npts + TB - 1) / TB);
  unc::carry_list_kernel<<<nb, TB, 0, st>>>(d_mask, npts, (int *)r.list.ptr, (int *)r.slot.ptr, d_cnt);
  g_launches++;
  unsigned int h_cnt[2] = {0, 0};
  CK(cudaMemcpyAsync(&h_cnt[0], d_cnt, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const long long nf = h_cnt[0];
  if (nf == 0) return UNC_OK;
  // sources
  if ((rc = r.need.ensure((size_t)npts * sizeof(unsigned long long)))) return rc;
  if ((rc = r.fix_src.ensure((size_t)nf * np * sizeof(int)))) return rc;
  if ((rc = r.src_slot.ensure((size_t)npts * sizeof(int)))) return rc;
  if ((rc = r.src_list.ensure((size_t)npts * sizeof(int)))) return rc;
  CK(cudaMemsetAsync(r.need.ptr, 0, (size_t)npts * sizeof(unsigned long long), st));
  unc::carry_scan_kernel<<<(unsigned)((nz * np + 127) / 128), 128, 0, st>>>(
      d_mask, Jg.ncol, nz, np, (const int *)r.slot.ptr, (int *)r.fix_src.ptr, (unsigned long long *)r.need.ptr);
  unc::carry_list_kernel<<<nb, TB, 0, st>>>((const unsigned long long *)r.need.ptr, npts, (int *)r.src_list.ptr,
                                            (int *)r.src_slot.ptr, d_cnt + 1);
  g_launches += 2;
  CK(cudaMemcpyAsync(&h_cnt[1], d_cnt + 1, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const long long ns = h_cnt[1];
  if ((rc = r.fix_val.ensure((size_t)std::max<long long>(ns, 1) * np * 2 * sizeof(double)))) return rc;
  if ((rc = r.fix_out.ensure((size_t)nf * 2 * sizeof(double)))) return rc;
  unc::carry_link_kernel<<<(unsigned)((nf * np + TB - 1) / TB), TB, 0, st>>>(
      (const int *)r.list.ptr, nf, nz, np, d_mask, (const int *)r.src_slot.ptr, (int *)r.fix_src.ptr);
  g_launches++;
  CK(cudaGetLastError());
  // pass 1: Wynn results of the source points for the p somebody inherits
  unc::Job Js = Jg;
  Js.s = Js.ds = nullptr; Js.flags = nullptr; Js.smask = nullptr;
  Js.fix_mode = 1;
  Js.fix_n = ns;
  Js.fix_list = (const int *)r.src_list.ptr;
  Js.fix_need = (const unsigned long long *)r.need.ptr;
  Js.fix_val = (double *)r.fix_val.ptr;
  if (ns > 0 && (rc = launch_zt<1>(dev, P, Js, st, ns))) return rc;
  // pass 2: the flagged points again, with the inherited values
  unc::Job Jd = Jg;
  Jd.flags = nullptr; Jd.smask = nullptr;
  Jd.fix_mode = 2;
  Jd.fix_n = nf;
  Jd.fix_list = (const int *)r.list.ptr;
  Jd.fix_src = (const int *)r.fix_src.ptr;
  Jd.fix_val = (double *)r.fix_val.ptr;
  Jd.fix_s = (double *)r.fix_out.ptr;
  Jd.fix_ds = Jd.fix_s + nf;
  if ((rc = launch_zt<1>(dev, P, Jd, st, nf))) return rc;
  if (h_list) {
    h_list->resize(nf); h_s->resize(nf); h_ds->resize(nf);
    CK(cudaMemcpyAsync(h_list->data(), r.list.ptr, nf * sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h_s->data(), Jd.fix_s, nf * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h_ds->data(), Jd.fix_ds, nf * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  *nf_out = nf;
  return UNC_OK;
}

int check_common(const double *tD, const int32_t *sv, const double *rD, const double *zD,
                 const int32_t *zLay, const double *o1, const double *o2) {
  if (!tD || !sv || !rD || !zD || !zLay || !o1 || !o2) return fail(UNC_ERR_BAD_ARG, "NULL array argument");
  return UNC_OK;
}

int validate_sv(const unc_params *prm, long long n, const int32_t *sv) {
  for (long long i = 0; i < n; ++i)
    if (sv[i] < 1 || sv[i] + prm->gl_nacc > prm->n_j0z)
      return fail(UNC_ERR_BAD_ARG, "sv[%lld]=%d needs j0z(1..%d) but n_j0z=%d", i, sv[i],
                  sv[i] + prm->gl_nacc, prm->n_j0z);
  return UNC_OK;
}

int device_count() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

// Host-array evaluation of a contiguous range of columns on one device.
struct Shard {
  int dev;
  long long c0, c1;  // columns [c0,c1)
  int rc = 0;
  std::string err;
  long long nflagged = 0;
};

// What a call evaluates: host arrays for run_host, device arrays for run_device.
enum class JobKind { grid, points, screens, dz };

struct HostJob {
  JobKind kind;
  long long ncol;
  int nt = 0, nr = 0, nz = 1;    // grid: the t, r and z axes; lists: one z per column
  const double *tD; const int32_t *sv; const double *rD;
  const double *zD;              // screens: the bottoms
  const int32_t *zLay = nullptr; // grid, points
  const double *ztop = nullptr;  // screens: the tops
  const double *ts;
  double *s, *ds; int32_t *flags;  // dz: s/ds receive gz/dgz
  bool carry = false;            // grid jobs with ts given: reproduce the reference's stale infint
  unsigned long long *hmask = nullptr;  // carry: host copy of the per-point stale masks (global order)
};

// device addresses of a job's inputs.  upload_inputs copies those of columns [c0,c1): grid jobs
// get the whole t/r/z axes (a few KB) and address them by global column (Job::col0); point lists
// get their own slice
struct DevInputs {
  const double *tD, *rD, *zD, *ts, *ztop;
  const int32_t *sv, *lay;
};

int upload_inputs(DevBuf &buf, const HostJob &hj, long long c0, long long c1, cudaStream_t st, DevInputs &d) {
  const long long nc = c1 - c0;
  const bool grid = hj.kind == JobKind::grid;
  const size_t n_t = grid ? (size_t)hj.nt : (size_t)nc;
  const size_t n_r = grid ? (size_t)hj.nr : (size_t)nc;
  const size_t n_z = grid ? (size_t)hj.nz : (size_t)nc;
  const size_t n_ts = hj.ts ? (size_t)nc : 0;
  const size_t n_top = hj.ztop ? n_z : 0;
  const long long off = grid ? 0 : c0;
  int rc = buf.ensure((n_t + n_r + n_z + n_ts + n_top) * sizeof(double) + (n_t + n_z) * sizeof(int32_t) + 64);
  if (rc) return rc;
  double *tD = (double *)buf.ptr, *rD = tD + n_t, *zD = rD + n_r, *ts = zD + n_z, *ztop = ts + n_ts;
  int32_t *sv = (int32_t *)(ztop + n_top), *lay = sv + n_t;
  CK(cudaMemcpyAsync(tD, hj.tD + off, n_t * sizeof(double), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(sv, hj.sv + off, n_t * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(rD, hj.rD + off, n_r * sizeof(double), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(zD, hj.zD + off, n_z * sizeof(double), cudaMemcpyHostToDevice, st));
  if (hj.zLay) CK(cudaMemcpyAsync(lay, hj.zLay + off, n_z * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  if (hj.ztop) CK(cudaMemcpyAsync(ztop, hj.ztop + off, n_top * sizeof(double), cudaMemcpyHostToDevice, st));
  if (hj.ts) CK(cudaMemcpyAsync(ts, hj.ts + c0, n_ts * sizeof(double), cudaMemcpyHostToDevice, st));
  d = {tD, rD, zD, hj.ts ? ts : nullptr, hj.ztop ? ztop : nullptr, sv, lay};
  return UNC_OK;
}

unc::Job make_job(const HostJob &hj, const DevInputs &d, long long c0, long long nc) {
  unc::Job J;
  std::memset(&J, 0, sizeof J);
  J.ncol = nc;
  J.nz = hj.nz;
  J.tD = d.tD; J.sv = d.sv; J.rD = d.rD; J.zD = d.zD; J.zLay = d.lay;
  J.ts_scale = d.ts;
  if (hj.kind == JobKind::grid) {
    J.col0 = c0;          // global column c: t = c / nr, r = c % nr (driver.f90:100,113 loop order)
    J.tdiv = hj.nr;
    J.rmod = hj.nr;
    J.zstride = 0;
  } else {
    J.col0 = 0;
    J.tdiv = 1;
    J.rmod = nc;
    J.zstride = 1;
  }
  return J;
}

// the kernel family of the job's kind; `ztop` is the device copy of the screens' tops
int launch_job(JobKind kind, int dev, StreamRes &r, const unc::DevParams &P, const unc::Job &J, const double *ztop,
               cudaStream_t st) {
  switch (kind) {
    case JobKind::screens: return launch_column<unc::COL_SCREEN>(dev, r, P, J, ztop, st);
    case JobKind::dz: return launch_column<unc::COL_DZ>(dev, r, P, J, nullptr, st);
    default: return launch(dev, r, P, J, st);
  }
}

int run_shard(const unc_params *prm, const HostJob &hj, Shard &sh) {
  HostPlan hp;
  int rc = make_plan(prm, hp);
  if (rc) return rc;
  rc = ensure_ctx(sh.dev);
  if (rc) return rc;
  DevCtx &c = g_ctx[sh.dev];
  cudaStream_t st = c.stream;
  StreamRes &r = c.res[st];
  rc = upload_tables(r, hp, st);
  if (rc) return rc;
  const long long nc = sh.c1 - sh.c0;
  if (nc <= 0) return UNC_OK;
  const int nz = hj.nz;
  const size_t npts = (size_t)nc * nz;
  DevInputs di;
  rc = upload_inputs(c.in, hj, sh.c0, sh.c1, st, di);
  if (rc) return rc;
  // outputs: s | ds | masks (carry) | flags | flagged-count
  rc = c.out.ensure(npts * (2 * sizeof(double) + sizeof(unsigned long long) + sizeof(int32_t)) + 64);
  if (rc) return rc;
  double *d_s = (double *)c.out.ptr;
  double *d_ds = d_s + npts;
  unsigned long long *d_mask = (unsigned long long *)(d_ds + npts);
  int32_t *d_fl = (int32_t *)(d_mask + npts);
  unsigned int *d_cnt = (unsigned int *)(d_fl + npts);
  unc::Job J = make_job(hj, di, sh.c0, nc);
  J.s = d_s; J.ds = d_ds;
  J.flags = hj.flags ? d_fl : nullptr;
  J.smask = hj.carry ? d_mask : nullptr;
  J.nstale = hj.carry ? d_cnt : nullptr;      // the kernels count the points with a stale infint
  if (hj.carry) CK(cudaMemsetAsync(d_cnt, 0, sizeof(unsigned int), st));
  rc = launch_job(hj.kind, sh.dev, r, hp.P, J, di.ztop, st);
  if (rc) return rc;
  unsigned int h_cnt = 0;
  if (hj.carry) CK(cudaMemcpyAsync(&h_cnt, d_cnt, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(hj.s + sh.c0 * nz, d_s, npts * sizeof(double), cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(hj.ds + sh.c0 * nz, d_ds, npts * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (hj.flags)
    CK(cudaMemcpyAsync(hj.flags + sh.c0 * nz, d_fl, npts * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  sh.nflagged = h_cnt;
  if (hj.carry && h_cnt > 0) {
    CK(cudaMemcpyAsync(hj.hmask + sh.c0 * nz, d_mask, npts * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  return UNC_OK;
}

// carry post-pass for host-array jobs: after every shard has finished, on one device, over the
// whole job in the reference's column order (the chain crosses shard boundaries)
int carry_host(const unc_params *prm, const HostJob &hj, int dev) {
  HostPlan hp;
  int rc = make_plan(prm, hp);
  if (rc) return rc;
  rc = ensure_ctx(dev);
  if (rc) return rc;
  DevCtx &c = g_ctx[dev];
  cudaStream_t st = c.stream;
  StreamRes &r = c.res[st];
  rc = upload_tables(r, hp, st);
  if (rc) return rc;
  DevInputs di;
  rc = upload_inputs(r.cin, hj, 0, hj.ncol, st, di);
  if (rc) return rc;
  const size_t npts = (size_t)hj.ncol * hj.nz;
  rc = r.mask.ensure(npts * sizeof(unsigned long long));
  if (rc) return rc;
  CK(cudaMemcpyAsync(r.mask.ptr, hj.hmask, npts * sizeof(unsigned long long), cudaMemcpyHostToDevice, st));
  unc::Job J = make_job(hj, di, 0, hj.ncol);
  std::vector<int> list;
  std::vector<double> vs, vds;
  long long nf = 0;
  rc = carry_postpass(dev, r, hp.P, J, (const unsigned long long *)r.mask.ptr, st, &nf, &list, &vs, &vds);
  if (rc) return rc;
  for (long long i = 0; i < nf; ++i) {
    hj.s[list[i]] = vs[i];
    hj.ds[list[i]] = vds[i];
  }
  return UNC_OK;
}

int run_host(const unc_params *prm, HostJob hj, int ngpu) {
  std::lock_guard<std::mutex> lk(g_mutex);
  DeviceGuard guard;
  {
    HostPlan probe;   // parameter validation is host-only and comes before any device work
    int rc = make_plan(prm, probe);
    if (rc) return rc;
  }
  if (ngpu < 0) return fail(UNC_ERR_BAD_ARG, "ngpu < 0");
  const int avail = device_count();
  if (avail <= 0) return fail(UNC_ERR_NO_DEVICE, "no CUDA device available (there is no CPU fallback)");
  int use = ngpu == 0 ? avail : std::min(ngpu, avail);
  if (hj.ncol < use) use = (int)std::max<long long>(1, hj.ncol);
  std::vector<unsigned long long> hmask;
  if (hj.carry) {
    hmask.assign((size_t)hj.ncol * hj.nz, 0ull);
    hj.hmask = hmask.data();
  }
  // contiguous equal split of the columns (SURVEY 8e) over the devices g_device, g_device+1, ...
  std::vector<Shard> shards(use);
  for (int g = 0; g < use; ++g) {
    shards[g].dev = (g_device + g) % avail;
    shards[g].c0 = hj.ncol * g / use;
    shards[g].c1 = hj.ncol * (g + 1) / use;
  }
  if (use == 1) {
    shards[0].rc = run_shard(prm, hj, shards[0]);
    if (shards[0].rc) return shards[0].rc;
  } else {
    std::vector<std::thread> th;
    for (int g = 0; g < use; ++g)
      th.emplace_back([&, g]() {
        shards[g].rc = run_shard(prm, hj, shards[g]);
        if (shards[g].rc) shards[g].err = g_err;
      });
    for (auto &t : th) t.join();
    for (int g = 0; g < use; ++g)
      if (shards[g].rc) {
        g_err = shards[g].err;
        return shards[g].rc;
      }
  }
  if (hj.carry) {
    long long nfl = 0;
    for (auto &sh : shards) nfl += sh.nflagged;
    if (nfl > 0) return carry_host(prm, hj, shards[0].dev);
  }
  return UNC_OK;
}

// the *_device entries: the caller's device arrays, on g_device, enqueued on the caller's stream
int run_device(const unc_params *prm, const HostJob &hj, void *stream) {
  std::lock_guard<std::mutex> lk(g_mutex);
  DeviceGuard guard;
  if (device_count() <= 0) return fail(UNC_ERR_NO_DEVICE, "no CUDA device available");
  HostPlan hp;
  int rc = make_plan(prm, hp);
  if (rc) return rc;
  rc = ensure_ctx(g_device);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  StreamRes &r = g_ctx[g_device].res[st];
  rc = upload_tables(r, hp, st);
  if (rc) return rc;
  const DevInputs d{hj.tD, hj.rD, hj.zD, hj.ts, hj.ztop, hj.sv, hj.zLay};
  unc::Job J = make_job(hj, d, 0, hj.ncol);
  J.s = hj.s; J.ds = hj.ds; J.flags = hj.flags;
  if (hj.carry) {
    rc = r.mask.ensure((size_t)J.ncol * J.nz * sizeof(unsigned long long));
    if (rc) return rc;
    J.smask = (unsigned long long *)r.mask.ptr;
  }
  rc = launch_job(hj.kind, g_device, r, hp.P, J, d.ztop, st);
  if (rc || !hj.carry) return rc;
  // reference-compatible mode: patch the stale points in place (synchronises the stream)
  J.smask = nullptr;
  long long nf = 0;
  return carry_postpass(g_device, r, hp.P, J, (const unsigned long long *)r.mask.ptr, st, &nf, nullptr, nullptr, nullptr);
}

}  // namespace

extern "C" {


const char *unc_version(void) { return "unconfined_b200 0.1 (sm_100a)"; }
const char *unc_last_error(void) { return g_err.c_str(); }

int unc_device_count(int32_t *ngpu) {
  if (!ngpu) return fail(UNC_ERR_BAD_ARG, "NULL");
  *ngpu = device_count();
  return UNC_OK;
}

int unc_set_device(int32_t device) {
  if (device < 0 || device >= device_count()) return fail(UNC_ERR_NO_DEVICE, "device %d not available", device);
  g_device = device;
  return UNC_OK;
}

int unc_device_info(int32_t *ngpu, double *fp64_peak_flops) {
  int n = device_count();
  if (ngpu) *ngpu = n;
  if (fp64_peak_flops) {
    *fp64_peak_flops = 0.0;
    if (n > 0) {
      cudaDeviceProp pr;
      CK(cudaGetDeviceProperties(&pr, g_device));
      int khz = 0;
      CK(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, g_device));
      // 64 FP64 FMA lanes per SM per clock on sm_100 (2 flops each)
      *fp64_peak_flops = (double)pr.multiProcessorCount * 64.0 * 2.0 * (double)khz * 1e3;
    }
  }
  return UNC_OK;
}

int unc_kernel_launch_count(int64_t *n) {
  if (!n) return fail(UNC_ERR_BAD_ARG, "NULL");
  *n = g_launches.load();
  return UNC_OK;
}

int unc_measure_fp64_peak(double *flops) {
  if (!flops) return fail(UNC_ERR_BAD_ARG, "NULL");
  std::lock_guard<std::mutex> lk(g_mutex);
  DeviceGuard guard;
  if (device_count() <= 0) return fail(UNC_ERR_NO_DEVICE, "no CUDA device available");
  int rc = ensure_ctx(g_device);
  if (rc) return rc;
  cudaStream_t st = g_ctx[g_device].stream;
  cudaDeviceProp pr;
  CK(cudaGetDeviceProperties(&pr, g_device));
  const int blocks = pr.multiProcessorCount * 8, threads = 256, iters = 1 << 16;
  double *d = nullptr;
  CK(cudaMalloc(&d, (size_t)blocks * threads * sizeof(double)));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  unc::fp64_peak_kernel<<<blocks, threads, 0, st>>>(d, 1024);
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    CK(cudaEventRecord(e0, st));
    unc::fp64_peak_kernel<<<blocks, threads, 0, st>>>(d, iters);
    g_launches++;
    CK(cudaEventRecord(e1, st));
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    double f = (double)blocks * threads * (double)iters * 8.0 * 2.0 / (ms * 1e-3);
    best = std::max(best, f);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  *flops = best;
  return UNC_OK;
}

int unc_shutdown(void) {
  std::lock_guard<std::mutex> lk(g_mutex);
  DeviceGuard guard;
  for (int d = 0; d < 16; ++d) {
    DevCtx &c = g_ctx[d];
    if (!c.init) continue;
    cudaSetDevice(d);
    cudaDeviceSynchronize();
    c.in.release(); c.out.release();
    for (auto &kv : c.res) kv.second.release();
    cudaStreamDestroy(c.stream);
    c = DevCtx();
  }
  return UNC_OK;
}

/* frees the scratch, counters and tables the library keeps for `stream` on the current device
 * (they are otherwise cached until unc_shutdown); synchronises the stream first */
int unc_release_stream(void *stream) {
  std::lock_guard<std::mutex> lk(g_mutex);
  DeviceGuard guard;
  if (device_count() <= 0) return UNC_OK;
  DevCtx &c = g_ctx[g_device];
  if (!c.init) return UNC_OK;
  CK(cudaSetDevice(g_device));
  cudaStream_t st = (cudaStream_t)stream;
  auto it = c.res.find(st);
  if (it == c.res.end()) return UNC_OK;
  CK(cudaStreamSynchronize(st));
  it->second.release();
  c.res.erase(it);
  return UNC_OK;
}

/* 1 (default): grid calls that pass ts_abscissa_scale (reference-compatible mode) also
 * reproduce the reference's stale infint (driver.f90:205-214); 0: such points get infint = 0
 * and UNC_FLAG_STALE_INFINT only, as calls with ts_abscissa_scale = NULL always do */
int unc_set_carry(int32_t on) {
  g_carry.store(on ? 1 : 0);
  return UNC_OK;
}

/* test hook: the device cbknu (K0, K1 of n complex arguments, host arrays z[2n] -> out[4n]) */
int unc_debug_cbesk01(int32_t n, const double *z, double *out) {
  if (n < 0 || (n > 0 && (!z || !out))) return fail(UNC_ERR_BAD_ARG, "bad arguments");
  if (n == 0) return UNC_OK;
  std::lock_guard<std::mutex> lk(g_mutex);
  DeviceGuard guard;
  if (device_count() <= 0) return fail(UNC_ERR_NO_DEVICE, "no CUDA device available");
  int rc = ensure_ctx(g_device);
  if (rc) return rc;
  cudaStream_t st = g_ctx[g_device].stream;
  double *d = nullptr;
  CK(cudaMalloc(&d, (size_t)n * 6 * sizeof(double)));
  CK(cudaMemcpyAsync(d, z, (size_t)n * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
  unc::cbesk01_test_kernel<<<(n + 127) / 128, 128, 0, st>>>(n, d, d + 2 * (size_t)n);
  g_launches++;
  CK(cudaMemcpyAsync(out, d + 2 * (size_t)n, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  cudaFree(d);
  return UNC_OK;
}

/* test hook: pin the kernel family (0 auto, 1 point kernel, 2 grid kernels, 3 the lanes<->z
 * grid kernel even for nz >= 33; 4 the 128-z kernel from nz = 32); never needed by a caller of the product */
int unc_debug_force_kernel(int32_t which) {
  if (which < 0 || which > 4) return fail(UNC_ERR_BAD_ARG, "which must be 0..4");
  g_force.store(which);
  return UNC_OK;
}

int unc_eval_grid_ex(const unc_params *prm, int32_t nt, const double *tD, const int32_t *sv,
                     int32_t nr, const double *rD, int32_t nz, const double *zD,
                     const int32_t *zLay, const double *ts_abscissa_scale, int32_t ngpu,
                     double *totint, double *totintd, int32_t *flags) {
  if (nt < 0 || nr < 0 || nz < 0) return fail(UNC_ERR_BAD_ARG, "negative size");
  if (nt == 0 || nr == 0 || nz == 0) return UNC_OK;
  int rc = check_common(tD, sv, rD, zD, zLay, totint, totintd);
  if (rc) return rc;
  if (!prm) return fail(UNC_ERR_BAD_ARG, "prm is NULL");
  rc = validate_sv(prm, nt, sv);
  if (rc) return rc;
  // reference-compatible callers (ts_abscissa_scale given) also get the reference's stale infint
  const HostJob hj{.kind = JobKind::grid, .ncol = (long long)nt * nr, .nt = nt, .nr = nr, .nz = nz, .tD = tD,
                   .sv = sv, .rD = rD, .zD = zD, .zLay = zLay, .ts = ts_abscissa_scale, .s = totint,
                   .ds = totintd, .flags = flags, .carry = ts_abscissa_scale != nullptr && g_carry.load() != 0};
  return run_host(prm, hj, ngpu);
}

int unc_eval_grid(const unc_params *prm, int32_t nt, const double *tD, const int32_t *sv,
                  int32_t nr, const double *rD, int32_t nz, const double *zD,
                  const int32_t *zLay, const double *ts_abscissa_scale, int32_t ngpu,
                  double *totint, double *totintd) {
  return unc_eval_grid_ex(prm, nt, tD, sv, nr, rD, nz, zD, zLay, ts_abscissa_scale, ngpu, totint,
                          totintd, nullptr);
}

int unc_eval_points_ex(const unc_params *prm, int64_t n, const double *tD, const int32_t *sv,
                       const double *rD, const double *zD, const int32_t *zLay,
                       const double *ts_abscissa_scale, int32_t ngpu, double *s, double *ds,
                       int32_t *flags) {
  if (n < 0) return fail(UNC_ERR_BAD_ARG, "negative size");
  if (n == 0) return UNC_OK;
  int rc = check_common(tD, sv, rD, zD, zLay, s, ds);
  if (rc) return rc;
  if (!prm) return fail(UNC_ERR_BAD_ARG, "prm is NULL");
  rc = validate_sv(prm, n, sv);
  if (rc) return rc;
  // independent points: there is no "previous (t,r)" to inherit from
  const HostJob hj{.kind = JobKind::points, .ncol = n, .tD = tD, .sv = sv, .rD = rD, .zD = zD, .zLay = zLay,
                   .ts = ts_abscissa_scale, .s = s, .ds = ds, .flags = flags};
  return run_host(prm, hj, ngpu);
}

int unc_eval_points(const unc_params *prm, int64_t n, const double *tD, const int32_t *sv,
                    const double *rD, const double *zD, const int32_t *zLay,
                    const double *ts_abscissa_scale, int32_t ngpu, double *s, double *ds) {
  return unc_eval_points_ex(prm, n, tD, sv, rD, zD, zLay, ts_abscissa_scale, ngpu, s, ds, nullptr);
}

int unc_eval_grid_device(const unc_params *prm, int32_t nt, const double *d_tD,
                         const int32_t *d_sv, int32_t nr, const double *d_rD, int32_t nz,
                         const double *d_zD, const int32_t *d_zLay,
                         const double *d_ts_abscissa_scale, double *d_totint, double *d_totintd,
                         int32_t *d_flags, void *stream) {
  if (nt < 0 || nr < 0 || nz < 0) return fail(UNC_ERR_BAD_ARG, "negative size");
  if (nt == 0 || nr == 0 || nz == 0) return UNC_OK;
  int rc = check_common(d_tD, d_sv, d_rD, d_zD, d_zLay, d_totint, d_totintd);
  if (rc) return rc;
  const HostJob hj{.kind = JobKind::grid, .ncol = (long long)nt * nr, .nt = nt, .nr = nr, .nz = nz, .tD = d_tD,
                   .sv = d_sv, .rD = d_rD, .zD = d_zD, .zLay = d_zLay, .ts = d_ts_abscissa_scale, .s = d_totint,
                   .ds = d_totintd, .flags = d_flags,
                   .carry = d_ts_abscissa_scale != nullptr && g_carry.load() != 0};
  return run_device(prm, hj, stream);
}

int unc_eval_points_device(const unc_params *prm, int64_t n, const double *d_tD,
                           const int32_t *d_sv, const double *d_rD, const double *d_zD,
                           const int32_t *d_zLay, const double *d_ts_abscissa_scale, double *d_s,
                           double *d_ds, int32_t *d_flags, void *stream) {
  if (n < 0) return fail(UNC_ERR_BAD_ARG, "negative size");
  if (n == 0) return UNC_OK;
  int rc = check_common(d_tD, d_sv, d_rD, d_zD, d_zLay, d_s, d_ds);
  if (rc) return rc;
  const HostJob hj{.kind = JobKind::points, .ncol = n, .tD = d_tD, .sv = d_sv, .rD = d_rD, .zD = d_zD,
                   .zLay = d_zLay, .ts = d_ts_abscissa_scale, .s = d_s, .ds = d_ds, .flags = d_flags};
  return run_device(prm, hj, stream);
}

int unc_eval_screens(const unc_params *prm, int64_t n, const double *tD, const int32_t *sv,
                     const double *rD, const double *zbot, const double *ztop,
                     const double *ts_abscissa_scale, int32_t ngpu, double *s, double *ds,
                     int32_t *flags) {
  if (n < 0) return fail(UNC_ERR_BAD_ARG, "negative size");
  if (n == 0) return UNC_OK;
  if (!tD || !sv || !rD || !zbot || !ztop || !s || !ds) return fail(UNC_ERR_BAD_ARG, "NULL array argument");
  if (!prm) return fail(UNC_ERR_BAD_ARG, "prm is NULL");
  for (int64_t i = 0; i < n; ++i)
    if (!(std::isfinite(zbot[i]) && std::isfinite(ztop[i]) && zbot[i] >= 0.0 && ztop[i] <= 1.0 && zbot[i] < ztop[i]))
      return fail(UNC_ERR_BAD_ARG, "screen %lld: [%g, %g] is not a non-empty interval in [0, 1]", (long long)i,
                  zbot[i], ztop[i]);
  int rc = validate_sv(prm, n, sv);
  if (rc) return rc;
  const HostJob hj{.kind = JobKind::screens, .ncol = n, .tD = tD, .sv = sv, .rD = rD, .zD = zbot, .ztop = ztop,
                   .ts = ts_abscissa_scale, .s = s, .ds = ds, .flags = flags};
  return run_host(prm, hj, ngpu);
}

int unc_eval_screens_device(const unc_params *prm, int64_t n, const double *d_tD, const int32_t *d_sv,
                            const double *d_rD, const double *d_zbot, const double *d_ztop,
                            const double *d_ts_abscissa_scale, double *d_s, double *d_ds, int32_t *d_flags,
                            void *stream) {
  if (n < 0) return fail(UNC_ERR_BAD_ARG, "negative size");
  if (n == 0) return UNC_OK;
  if (!d_tD || !d_sv || !d_rD || !d_zbot || !d_ztop || !d_s || !d_ds)
    return fail(UNC_ERR_BAD_ARG, "NULL array argument");
  const HostJob hj{.kind = JobKind::screens, .ncol = n, .tD = d_tD, .sv = d_sv, .rD = d_rD, .zD = d_zbot,
                   .ztop = d_ztop, .ts = d_ts_abscissa_scale, .s = d_s, .ds = d_ds, .flags = d_flags};
  return run_device(prm, hj, stream);
}

int unc_eval_points_dz(const unc_params *prm, int64_t n, const double *tD, const int32_t *sv, const double *rD,
                       const double *zD, const double *ts_abscissa_scale, int32_t ngpu, double *gz, double *dgz,
                       int32_t *flags) {
  if (n < 0) return fail(UNC_ERR_BAD_ARG, "negative size");
  if (n == 0) return UNC_OK;
  if (!tD || !sv || !rD || !zD || !gz || !dgz) return fail(UNC_ERR_BAD_ARG, "NULL array argument");
  if (!prm) return fail(UNC_ERR_BAD_ARG, "prm is NULL");
  for (int64_t i = 0; i < n; ++i)
    if (!(std::isfinite(zD[i]) && zD[i] >= 0.0 && zD[i] <= 1.0))
      return fail(UNC_ERR_BAD_ARG, "point %lld: zD = %g is not in [0, 1]", (long long)i, zD[i]);
  int rc = validate_sv(prm, n, sv);
  if (rc) return rc;
  const HostJob hj{.kind = JobKind::dz, .ncol = n, .tD = tD, .sv = sv, .rD = rD, .zD = zD, .ts = ts_abscissa_scale,
                   .s = gz, .ds = dgz, .flags = flags};
  return run_host(prm, hj, ngpu);
}

int unc_eval_points_dz_device(const unc_params *prm, int64_t n, const double *d_tD, const int32_t *d_sv,
                              const double *d_rD, const double *d_zD, const double *d_ts_abscissa_scale,
                              double *d_gz, double *d_dgz, int32_t *d_flags, void *stream) {
  if (n < 0) return fail(UNC_ERR_BAD_ARG, "negative size");
  if (n == 0) return UNC_OK;
  if (!d_tD || !d_sv || !d_rD || !d_zD || !d_gz || !d_dgz) return fail(UNC_ERR_BAD_ARG, "NULL array argument");
  const HostJob hj{.kind = JobKind::dz, .ncol = n, .tD = d_tD, .sv = d_sv, .rD = d_rD, .zD = d_zD,
                   .ts = d_ts_abscissa_scale, .s = d_gz, .ds = d_dgz, .flags = d_flags};
  return run_device(prm, hj, stream);
}

// driver_io.f90:628-647
int unc_j0_zeros(int32_t terms, double *j0z) {
  if (terms < 0 || (terms > 0 && !j0z)) return fail(UNC_ERR_BAD_ARG, "bad arguments");
  const double PIEP = 4.0 * std::atan(1.0);
  for (int i = 0; i < terms; ++i) {
    double x = (i + 0.75) * PIEP;
    for (int it = 0; it < 100; ++it) {
      double dx = ::j0(x) / ::j1(x);
      x = x + dx;
      double sp = std::nextafter(std::fabs(x), std::numeric_limits<double>::infinity()) - std::fabs(x);
      if (std::fabs(dx) < sp) break;
    }
    j0z[i] = x;
  }
  return UNC_OK;
}

// driver_io.f90:658-664
int unc_split_index(int32_t nt, const double *tD, int32_t j0s_a, int32_t j0s_b, int32_t *sv) {
  if (nt < 0 || (nt > 0 && (!tD || !sv))) return fail(UNC_ERR_BAD_ARG, "bad arguments");
  const int lo = std::min(j0s_a, j0s_b), zrange = std::max(j0s_a, j0s_b) - lo;
  double mn = INFINITY, mx = -INFINITY;
  for (int i = 0; i < nt; ++i) {
    double l = std::log10(tD[i]);
    mn = std::min(mn, l);
    mx = std::max(mx, l);
  }
  const int minlsp = (int)std::floor(mn), maxlsp = (int)std::ceil(mx);
  const int spRange = maxlsp - minlsp + 1;
  for (int i = 0; i < nt; ++i)
    sv[i] = lo + (int)(zrange * ((maxlsp - std::log10(tD[i])) / spRange));
  return UNC_OK;
}

// driver_io.f90:572-586
int unc_zlay(int32_t nz, const double *zD, double lD, double dD, int32_t *zLay) {
  if (nz < 0 || (nz > 0 && (!zD || !zLay))) return fail(UNC_ERR_BAD_ARG, "bad arguments");
  for (int i = 0; i < nz; ++i) {
    if (zD[i] <= 0.0 || zD[i] < (1.0 - lD)) zLay[i] = 1;
    else if ((zD[i] - 1.0) >= 0.0 || zD[i] < (1.0 - dD)) zLay[i] = 2;
    else zLay[i] = 3;
  }
  return UNC_OK;
}

}  // extern "C"
