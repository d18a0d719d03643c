// unconfined_cli -- the reference's command line on top of the C ABI:
//     unconfined_cli [input.dat] [--fresh-abscissae] [--exact-screen] [--vertical-gradient] [--ngpu N] [--stdout]
//                    [--dump | --header-only]
// reads the deck exactly as read_input does (driver_io.f90:30-666), evaluates
// driver.f90:100-231 through ONE unc_eval_grid call on the GPU(s), and writes the
// reference's output file (headers driver_io.f90:668-845, rows driver.f90:234-272).
// There is no CPU evaluation path: without a CUDA device the call fails with the
// library's error.  --dump prints the parsed/derived deck (hex floats) and exits without
// touching the device (used by the CPU tests).  --exact-screen: for a time-series deck with a
// screened observation well (piezometer = F), each time's value is the exact drawdown averaged
// over [zBot, zTop]/b (one unc_eval_screens screen per time) instead of the reference's
// zOrd-point rule (driver.f90:236-239); the header is unchanged.  --vertical-gradient: for a
// piezometer time-series deck or a contour deck the rows carry gz = ds/dz and dgz = d gz/d ln t
// (unc_eval_points_dz) in place of s and ds, times Hc/Lc for a dimensional deck; the header is
// unchanged.  A screened time-series deck is refused: the screen mean of a gradient is a
// difference of two point drawdowns.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <stdexcept>
#include <string>
#include <vector>

#include "../include/unconfined_b200.h"
#include "deck_io.hpp"

using uncli::Deck;

static void fill_tables(Deck &d) {
  // driver_io.f90:572-586, 628-664 through the library's host routines
  const int terms = std::max(d.j0s[0], d.j0s[1]) + d.nacc + 1;
  d.j0z.resize(terms);
  if (unc_j0_zeros(terms, d.j0z.data())) throw std::runtime_error(unc_last_error());
  d.sv.resize(d.tD.size());
  if (unc_split_index((int32_t)d.tD.size(), d.tD.data(), d.j0s[0], d.j0s[1], d.sv.data()))
    throw std::runtime_error(unc_last_error());
  d.zLay.resize(d.zD.size());
  if (unc_zlay((int32_t)d.zD.size(), d.zD.data(), d.lD, d.dD, d.zLay.data())) throw std::runtime_error(unc_last_error());
}

static unc_params make_params(const Deck &d) {
  unc_params p;
  std::memset(&p, 0, sizeof p);
  p.model = d.model; p.M = d.M; p.alpha = d.alpha; p.tol = d.tol;
  p.tee_mult = 2.0;                                   // driver.f90:54
  p.time_type = d.timeType; p.n_time_par = (int32_t)d.timePar.size(); p.time_par = d.timePar.data();
  p.ts_k = d.ts_k; p.ts_R = d.ts_R; p.gl_nacc = d.nacc; p.gl_ord = d.ord;
  p.n_j0z = (int32_t)d.j0z.size(); p.j0z = d.j0z.data();
  p.moench_M = d.MoenchM; p.moench_gamma = d.MoenchM ? d.MoenchGamma.data() : nullptr;
  p.kappa = d.kappa; p.alphaD = d.alphaD; p.beta = d.beta;
  p.lD = d.lD; p.dD = d.dD; p.bD = d.bD; p.rDw = d.rDw;
  p.l = d.l; p.d = d.d; p.Ss = d.Ss; p.rDwobs = d.rDwobs; p.sF = d.sF;
  p.mn_type = d.MNtype; p.mn_ak = d.ak; p.mn_psia = d.psia; p.mn_psik = d.psik; p.mn_b = d.b; p.mn_Sy = d.Sy;
  return p;
}

static void dump(const Deck &d) {
  auto vec = [](const char *name, const std::vector<double> &v) {
    std::printf("%s %zu", name, v.size());
    for (double x : v) std::printf(" %a", x);
    std::printf("\n");
  };
  auto ivec = [](const char *name, const std::vector<int32_t> &v) {
    std::printf("%s %zu", name, v.size());
    for (int x : v) std::printf(" %d", x);
    std::printf("\n");
  };
  std::printf("model %d\ndimless %d\ntimeseries %d\npiezometer %d\n", d.model, d.dimless, d.timeseries, d.piezometer);
  std::printf("M %d\nts_k %d\nts_R %d\nj0s %d %d\nnacc %d\nord %d\ntimeType %d\nMNtype %d\nzOrd %d\n", d.M, d.ts_k,
              d.ts_R, d.j0s[0], d.j0s[1], d.nacc, d.ord, d.timeType, d.MNtype, d.zOrd);
  std::printf("scalars %a %a %a %a %a %a %a %a %a %a %a %a %a %a %a\n", d.alpha, d.tol, d.kappa, d.alphaD, d.beta, d.lD,
              d.dD, d.bD, d.rDw, d.rDwobs, d.Lc, d.Tc, d.Hc, d.l, d.d);
  vec("timePar", d.timePar); vec("MoenchGamma", d.MoenchGamma);
  vec("t", d.t); vec("r", d.r); vec("z", d.z); vec("tD", d.tD); vec("rD", d.rD); vec("zD", d.zD);
  vec("j0z", d.j0z); ivec("sv", d.sv); ivec("zLay", d.zLay);
  std::printf("outfile %s\n", d.outFileName.c_str());
}

int main(int argc, char **argv) {
  std::string input = "input.dat";   // driver_io.f90:66-70
  bool fresh = false, only_dump = false, to_stdout = false, header_only = false, exact_screen = false;
  bool vgrad = false;
  int ngpu = 0;
  for (int i = 1; i < argc; ++i) {
    std::string a = argv[i];
    if (a == "--fresh-abscissae") fresh = true;
    else if (a == "--exact-screen") exact_screen = true;
    else if (a == "--vertical-gradient") vgrad = true;
    else if (a == "--dump") only_dump = true;
    else if (a == "--stdout") to_stdout = true;
    else if (a == "--header-only") header_only = true;   // header text to stdout, no evaluation (no device needed)
    else if (a == "--format") {                          // RFMT / HFMT of the remaining arguments (tests)
      for (int k = i + 1; k < argc; ++k) {
        const double x = std::strtod(argv[k], nullptr);
        std::printf("[%s][%s]\n", uncli::RFMT(x).c_str(), uncli::HFMT(x).c_str());
      }
      return 0;
    }
    else if (a == "--ngpu" && i + 1 < argc) ngpu = std::atoi(argv[++i]);
    else if (a == "--help" || a == "-h") {
      std::puts("usage: unconfined_cli [input.dat] [--fresh-abscissae] [--exact-screen] [--vertical-gradient] [--ngpu N]\n"
                "                      [--dump] [--stdout]\n"
                "  --vertical-gradient  piezometer time-series and contour decks: the two value columns are\n"
                "                       gz = ds/dz and dgz = d gz/d ln t instead of s and ds (dimensionless, or\n"
                "                       times Hc/Lc for a dimensional deck); z points up, so the vertical\n"
                "                       specific discharge is q_z = K_z gz.  Headers are unchanged.");
      return 0;
    } else input = a;
  }
  try {
    Deck d = uncli::read_deck(input);
    if (vgrad && d.timeseries && !d.piezometer)
      throw std::runtime_error("--vertical-gradient: this deck has a screened observation well (piezometer = F); "
                               "the gradient is defined at points (the screen mean of a gradient is a "
                               "difference of two point drawdowns)");
    fill_tables(d);
    if (d.quiet > 0)
      for (const auto &w : d.warnings) std::cout << w << "\n";
    if (only_dump) { dump(d); return 0; }
    if (header_only) {
      std::string side;
      std::cout << (d.timeseries ? uncli::timeseries_header(d, &side) : uncli::contour_header(d, &side)) << side;
      return 0;
    }

    const int32_t nt = (int32_t)d.tD.size(), nr = (int32_t)d.rD.size(), nz = (int32_t)d.zD.size();
    // The reference builds the tanh-sinh abscissae only for the first (t,r) of a run
    // (driver.f90:121-126): reproduce that by default, --fresh-abscissae uses each (t,r)'s own
    std::vector<double> scale;
    if (!fresh) scale.assign((size_t)nt * nr, d.j0z[d.sv[0] - 1] / d.rD[0]);
    std::vector<double> s((size_t)nt * nr * nz), ds(s.size());
    unc_params p = make_params(d);
    // rows are written from a deck whose screen is one value per time: the exact screen mean, or
    // the point value where the screen has no length (zTop == zBot)
    Deck rows = d;
    const bool screen = exact_screen && d.timeseries && !d.piezometer;
    if (screen) { rows.z.resize(1); rows.zD.resize(1); rows.zOrd = 1; }
    int rc;
    if (vgrad) {
      // every (t, r, z) of the deck as an independent point, in the grid's order
      const size_t n = s.size();
      std::vector<double> tp(n), rp(n), zp(n), sc(fresh ? 0 : n);
      std::vector<int32_t> svp(n);
      for (size_t i = 0; i < n; ++i) {
        const size_t t = i / ((size_t)nr * nz), r = (i / nz) % nr, z = i % nz;
        tp[i] = d.tD[t]; svp[i] = d.sv[t]; rp[i] = d.rD[r]; zp[i] = d.zD[z];
        if (!fresh) sc[i] = scale[0];
      }
      rc = unc_eval_points_dz(&p, (int64_t)n, tp.data(), svp.data(), rp.data(), zp.data(),
                              fresh ? nullptr : sc.data(), ngpu, s.data(), ds.data(), nullptr);
      if (rc) throw std::runtime_error(std::string("unc_eval_points_dz: ") + unc_last_error());
      rows.Hc = d.Hc / d.Lc;   // output_rows scales dimensional rows by Hc: gz * (Hc/Lc)
    } else if (screen && d.zTop > d.zBot) {
      const std::vector<double> zb(nt, d.zBot / d.Lc), zt(nt, d.zTop / d.Lc), rD(nt, d.rD[0]);
      s.assign(nt, 0.0); ds.assign(nt, 0.0);
      rc = unc_eval_screens(&p, nt, d.tD.data(), d.sv.data(), rD.data(), zb.data(), zt.data(),
                            fresh ? nullptr : scale.data(), ngpu, s.data(), ds.data(), nullptr);
      if (rc) throw std::runtime_error(std::string("unc_eval_screens: ") + unc_last_error());
    } else {
      rc = unc_eval_grid(&p, nt, d.tD.data(), d.sv.data(), nr, d.rD.data(), nz, d.zD.data(), d.zLay.data(),
                         fresh ? nullptr : scale.data(), ngpu, s.data(), ds.data());
      if (rc) throw std::runtime_error(std::string("unc_eval_grid: ") + unc_last_error());
      if (screen) {   // zTop == zBot: the first of the zOrd identical points
        std::vector<double> s1(nt), ds1(nt);
        for (int i = 0; i < nt; ++i) { s1[i] = s[(size_t)i * nz]; ds1[i] = ds[(size_t)i * nz]; }
        s.swap(s1); ds.swap(ds1);
      }
    }

    std::string side;
    std::string text = d.timeseries ? uncli::timeseries_header(d, &side) : uncli::contour_header(d, &side);
    text += uncli::output_rows((screen || vgrad) ? rows : d, s, ds);
    std::cout << side;
    if (to_stdout) {
      std::cout << text;
    } else {
      std::ofstream f(d.outFileName, std::ios::trunc);
      if (!f) throw std::runtime_error("cannot open output file " + d.outFileName + " for writing");
      f << text;
    }
    unc_shutdown();
  } catch (const std::exception &e) {
    std::cerr << e.what() << "\n";
    return 1;
  }
  return 0;
}
