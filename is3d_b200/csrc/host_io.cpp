// host_io.cpp -- readers of the iS3D input files (see host_io.h).
#include "host_io.h"
#include "host_math.h"
#include <algorithm>
#include <cctype>
#include <cerrno>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>

namespace is3d {

static const double kHbarC = 0.197327053;   // GeV fm (reference iS3D.h:9)

static bool slurp(const std::string &path, std::string *out)
{
  std::ifstream f(path.c_str(), std::ios::binary);
  if (!f) return false;
  std::ostringstream ss; ss << f.rdbuf();
  *out = ss.str();
  return true;
}

// ------------------------------------------------------------------------------------------------ parameters
// The reference strips *every* blank and tab from both sides of '=' (arsenal.cpp:552-565) and lower-cases the name.
static std::string squeeze(const std::string &s)
{
  std::string t; t.reserve(s.size());
  for (char c : s) if (c != ' ' && c != '\t') t.push_back(c);
  return t;
}

bool Params::load(const std::string &path, std::string *err)
{
  std::string text;
  if (!slurp(path, &text)) { if (err) *err = "parameter file " + path + " does not exist"; return false; }
  std::istringstream in(text);
  std::string line;
  while (std::getline(in, line)) {
    if (squeeze(line).empty()) continue;
    const std::string body = squeeze(line.substr(0, line.find('#')));
    if (body.empty()) continue;
    const size_t eq = body.find('=');
    if (eq == std::string::npos) { if (err) *err = "parameter line without '=': " + line; return false; }
    std::string name = body.substr(0, eq);
    std::transform(name.begin(), name.end(), name.begin(), [](unsigned char c) { return (char)std::tolower(c); });
    std::istringstream rhs(body.substr(eq + 1) + " ");
    double v = 0.0; rhs >> v;
    if (!kv.count(name)) order.push_back(name);
    kv[name] = v;
  }
  return true;
}

bool Params::has(const std::string &name) const
{
  std::string n = squeeze(name);
  std::transform(n.begin(), n.end(), n.begin(), [](unsigned char c) { return (char)std::tolower(c); });
  return kv.count(n) != 0;
}

double Params::get(const std::string &name, std::string *err) const
{
  std::string n = squeeze(name);
  std::transform(n.begin(), n.end(), n.begin(), [](unsigned char c) { return (char)std::tolower(c); });
  auto it = kv.find(n);
  if (it == kv.end()) { if (err && err->empty()) *err = "parameter with name " + name + " not found"; return 0.0; }
  return it->second;
}

// ------------------------------------------------------------------------------------------------ block tables
static void line_values(const std::string &line, std::vector<double> *v)
{
  v->clear();
  std::istringstream ss(line + " ");
  double x;
  while (ss >> x) v->push_back(x);
}

bool BlockTable::load(const std::string &path, std::string *err)
{
  std::string text;
  cols.clear(); rows = 0;
  if (!slurp(path, &text)) { if (err) *err = "the data file " + path + " cannot be opened"; return false; }
  std::vector<double> vals;
  size_t pos = 0; bool first = true; size_t ncol = 0;
  // only lines that end in '\n' become rows: the reference pushes a line when the *next* getline has not hit EOF
  while (true) {
    const size_t nl = text.find('\n', pos);
    if (nl == std::string::npos) break;
    line_values(text.substr(pos, nl - pos), &vals);
    pos = nl + 1;
    if (first) {
      ncol = vals.size();
      if (ncol == 0) { if (err) *err = "table " + path + " has an empty first row"; return false; }
      cols.assign(ncol, std::vector<double>());
      first = false;
    }
    for (size_t c = 0; c < ncol; c++) cols[c].push_back(c < vals.size() ? vals[c] : 0.0);
    rows++;
  }
  if (first) { if (err) *err = "table " + path + " has no newline-terminated row"; return false; }
  return true;
}

// ------------------------------------------------------------------------------------------------ particle lists
static bool read_pdg_conventional(const std::string &path, std::vector<Particle> *out, std::string *err)
{
  std::string text;
  if (!slurp(path, &text)) { if (err) *err = "cannot open " + path; return false; }
  std::istringstream in(text);
  std::vector<Particle> v;
  // same extraction order and end-of-file behaviour as the reference loop: a trailing blank line produces one
  // empty record, which is dropped again below ("take account the final fake one", readindata.cpp:1539)
  while (!in.eof()) {
    Particle p;
    in >> p.mcid >> p.name >> p.mass >> p.width >> p.gspin >> p.baryon >> p.strange >> p.charm >> p.bottom >> p.gisospin >> p.charge >> p.decays;
    if (p.decays > 50) { if (err) *err = "too many decay channels in " + path; return false; }
    for (int j = 0; j < p.decays; j++) {
      long id; DecayChannel ch;
      in >> id >> ch.npart >> ch.branch_ratio >> ch.part[0] >> ch.part[1] >> ch.part[2] >> ch.part[3] >> ch.part[4];
      p.channels.push_back(ch);
    }
    p.stable = (!p.channels.empty() && p.channels[0].npart == 1) ? 1 : 0;      // readindata.cpp:1487-1488
    v.push_back(p);
    if (p.baryon > 0) {                                 // anti-baryon right behind its baryon (readindata.cpp:1491-1536)
      Particle a = p;
      a.mcid = -p.mcid; a.name = "Anti-baryon-" + p.name;
      a.baryon = -p.baryon; a.strange = -p.strange; a.charm = -p.charm; a.bottom = -p.bottom; a.charge = -p.charge;
      // daughters: the anti-particle, unless the daughter is a neutral non-strange meson (its own anti-particle in this table);
      // looked up among the particles read so far, first match (:1512-1530)
      for (auto &ch : a.channels)
        for (int k = 0; k < 5; k++) {
          if (ch.part[k] == 0) continue;
          bool neutral = false;
          for (const auto &q : v) if (q.mcid == ch.part[k]) { neutral = (q.baryon == 0 && q.charge == 0 && q.strange == 0); break; }
          if (!neutral) ch.part[k] = -ch.part[k];
        }
      v.push_back(a);
    }
  }
  if (v.empty()) { if (err) *err = "no particles in " + path; return false; }
  v.pop_back();
  for (auto &p : v) p.sign = (p.baryon % 2 == 0) ? -1 : 1;   // readindata.cpp:1541-1546
  *out = v;
  return true;
}

static bool read_pdg_smash_box(const std::string &path, std::vector<Particle> *out, std::string *err)
{
  std::ifstream f(path.c_str());
  if (!f) { if (err) *err = "cannot open " + path; return false; }
  std::vector<Particle> v;
  std::string line;
  while (std::getline(f, line)) {
    if (line.empty() || line[0] == '#') continue;
    std::istringstream ls(line);
    std::string name; double mass = 0, width = 0; char parity = 0; long ids[4] = {0, 0, 0, 0};
    ls >> name >> mass >> width >> parity;
    for (int k = 0; k < 4; k++) { long t; if (ls >> t) ids[k] = t; else break; }
    for (int k = 0; k < 4; k++) {
      if (ids[k] == 0) continue;
      // quantum numbers from the digits of the Monte-Carlo id (read_mcid, readindata.cpp:1201-1424)
      long x = std::labs(ids[k]); int d[10];
      for (int i = 0; i < 10; i++) { d[i] = (int)(x % 10); x /= 10; }
      const int nJ = d[0] + d[7], nq3 = d[1], nq2 = d[2], nq1 = d[3];
      const bool deuteron = (ids[k] == 1000010020L);
      const bool hadron = !deuteron && nq3 != 0 && nq2 != 0;
      const bool meson = hadron && nq1 == 0, bary = hadron && nq1 != 0;
      Particle p; p.name = name; p.mass = mass; p.width = width; p.mcid = ids[k];
      p.parity = (parity == '+') ? 1 : (parity == '-') ? -1 : 0;
      if (hadron) { p.gspin = (nJ > 0) ? nJ : 1; p.baryon = bary ? 1 : 0; p.sign = meson ? -1 : 1; }
      else if (deuteron) { p.gspin = 3; p.baryon = 2; p.sign = -1; }
      else { p.gspin = nq3 + 1; p.baryon = 0; p.sign = nq3 % 2; }
      const bool has_anti = hadron ? ((p.baryon != 0) || (nq2 != nq3)) : (deuteron ? true : (nq3 == 1));
      v.push_back(p);
      if (has_anti) { Particle a = p; a.name = "Anti-" + name; a.mcid = -ids[k]; a.baryon = -p.baryon; v.push_back(a); }
    }
  }
  *out = v;
  return true;
}

bool read_box_parities(const std::string &workdir, std::map<long, int> *out, std::string *err)
{
  std::vector<Particle> box;
  if (!read_pdg_smash_box(workdir + "/PDG/pdg_box.dat", &box, err)) {
    if (err) *err += " (polarization_feed_down = 1 reads the parities there)";
    return false;
  }
  out->clear();
  for (const Particle &p : box) if (p.parity != 0) out->emplace(std::labs(p.mcid), p.parity);       // first entry of an id wins
  return true;
}

bool read_weak_decays(const std::string &workdir, WeakTable *out, std::string *err)
{
  const std::string path = workdir + "/PDG/weak_decays.dat";
  std::ifstream f(path.c_str());
  if (!f) { if (err) *err = "cannot open " + path + " (polarization_weak_decays = 1 reads it)"; return false; }
  *out = WeakTable();
  std::string line;
  for (long n = 1; std::getline(f, line); n++) {
    const size_t hash = line.find('#');
    if (hash != std::string::npos) line.erase(hash);
    std::istringstream ls(line);
    std::string tok[7];
    int nt = 0;
    while (nt < 7 && ls >> tok[nt]) nt++;
    if (nt == 0) continue;
    long ids[3]; double v[3];
    bool ok = (nt == 6);
    for (int k = 0; ok && k < 6; k++) {
      char *end = nullptr;
      errno = 0;
      if (k < 3) ids[k] = std::strtol(tok[k].c_str(), &end, 10);
      else v[k - 3] = std::strtod(tok[k].c_str(), &end);
      ok = end && *end == '\0' && errno == 0;
    }
    if (!ok) { if (err) *err = path + ": line " + std::to_string(n) + " is not `parent daughter partner branching alpha phi`"; return false; }
    out->parent.push_back((int32_t)ids[0]); out->daughter.push_back((int32_t)ids[1]); out->partner.push_back((int32_t)ids[2]);
    out->branching.push_back(v[0]); out->alpha.push_back(v[1]); out->phi.push_back(v[2]);
  }
  return true;
}

bool read_pdg(const std::string &workdir, int hrg_eos, std::vector<Particle> *out, std::string *err)
{
  switch (hrg_eos) {
    case 1: return read_pdg_conventional(workdir + "/PDG/pdg-urqmd_v3.3+.dat", out, err);
    case 2: return read_pdg_conventional(workdir + "/PDG/pdg_smash.dat", out, err);
    case 3: return read_pdg_smash_box(workdir + "/PDG/pdg_box.dat", out, err);
    default: if (err) *err = "please choose hrg_eos = (1,2,3)"; return false;
  }
}

// ------------------------------------------------------------------------------------------------ surface
// strtod-based token reader: same result as `istream >> double` on well-formed files, and ~10x faster on 1M-cell files
struct Tokens {
  const char *p, *end;
  bool next(double *v)
  {
    while (p < end && std::isspace((unsigned char)*p)) p++;
    if (p >= end) return false;
    char *q = nullptr;
    *v = std::strtod(p, &q);
    if (q == p) return false;
    p = q;
    return true;
  }
};

// one newline-terminated line per surface cell, in surface order, with at least cols.size() numbers (`count` names that number)
static bool read_cell_columns(const std::string &path, const char *key, const std::vector<std::vector<double> *> &cols, const char *count,
                              int64_t n, std::string *err)
{
  std::string text;
  if (!slurp(path, &text)) { if (err) *err = "cannot open " + path + " (" + key + " = 1 reads it)"; return false; }
  int64_t lines = 0;
  for (char c : text) if (c == '\n') lines++;
  if (lines != n) {
    if (err) *err = path + " has " + std::to_string(lines) + " lines, the surface has " + std::to_string(n) + " cells";
    return false;
  }
  for (std::vector<double> *v : cols) v->assign((size_t)n, 0.0);
  const char *p = text.data(), *end = text.data() + text.size();
  for (int64_t i = 0; i < n; i++) {
    const char *eol = static_cast<const char *>(std::memchr(p, '\n', (size_t)(end - p)));
    Tokens tk{p, eol};
    for (std::vector<double> *v : cols)
      if (!tk.next(&(*v)[i])) {
        if (err) *err = path + ": line " + std::to_string(i + 1) + " has fewer than " + count + " numbers";
        return false;
      }
    p = eol + 1;
  }
  return true;
}

bool read_thermal_shear(const std::string &workdir, SurfaceData *s, std::string *err)
{
  return read_cell_columns(workdir + "/input/thermal_shear.dat", "thermal_shear_polarization",
                           {&s->xtt, &s->xtx, &s->xty, &s->xtn, &s->xxx, &s->xxy, &s->xxn, &s->xyy, &s->xyn, &s->xnn}, "ten", s->n, err);
}

bool read_baryon_gradient(const std::string &workdir, SurfaceData *s, std::string *err)
{
  return read_cell_columns(workdir + "/input/muB_over_T_gradient.dat", "spin_hall_polarization", {&s->gbt, &s->gbx, &s->gby, &s->gbn}, "four",
                           s->n, err);
}

bool read_surface(const std::string &workdir, const SurfaceFlags &fl, SurfaceData *s, std::string *err)
{
  const std::string path = workdir + "/input/surface.dat";
  std::string text;
  if (!slurp(path, &text)) { if (err) *err = "cannot open " + path; return false; }
  // cell count = newline-terminated lines (FO_data_reader::get_number_cells -> Table, readindata.cpp:122-131)
  int64_t n = 0;
  for (char c : text) if (c == '\n') n++;
  s->n = n;
  const int mode = fl.mode;
  if (mode < 0 || mode > 7 || mode == 3) {
    if (err) *err = "surface mode " + std::to_string(mode) + " has no smooth-spectra kernel (the reference reads mode 3 but never dispatches it)";
    return false;
  }
  auto rs = [&](std::vector<double> &v) { v.assign((size_t)n, 0.0); };
  rs(s->tau); rs(s->x); rs(s->y); rs(s->eta); rs(s->dat); rs(s->dax); rs(s->day); rs(s->dan); rs(s->ux); rs(s->uy); rs(s->un);
  rs(s->E); rs(s->T); rs(s->P); rs(s->pixx); rs(s->pixy); rs(s->pixn); rs(s->piyy); rs(s->piyn); rs(s->bulkPi);
  rs(s->muB); rs(s->nB); rs(s->Vx); rs(s->Vy); rs(s->Vn);
  const bool full_pi = (mode == 0 || mode == 2 || mode == 4 || mode == 6);     // formats that store all ten pi components
  if (full_pi) { rs(s->pitt); rs(s->pitx); rs(s->pity); rs(s->pitn); rs(s->pinn); }
  if (mode == 2) { rs(s->PL); rs(s->Wx); rs(s->Wy); rs(s->Lambda); rs(s->aL); rs(s->c0); rs(s->c1); rs(s->c2); rs(s->c3); rs(s->c4); }
  if (mode == 5) { rs(s->wtx); rs(s->wty); rs(s->wtn); rs(s->wxy); rs(s->wxn); rs(s->wyn); }

  Tokens tk{text.data(), text.data() + text.size()};
  double Tavg = 0, Eavg = 0, Pavg = 0, muBavg = 0, nBavg = 0, volume = 0;
  bool short_file = false;
  auto rd = [&](double *v) { if (!tk.next(v)) { short_file = true; *v = 0.0; } };
  auto rd_gev = [&](double *v) { double t; rd(&t); *v = t * kHbarC; };      // fm^-n -> GeV fm^(1-n), one multiply
  const bool writes_averages = (mode != 2 && mode != 5);                    // readindata.cpp: modes 2, 3, 5 never write the side file
  for (int64_t i = 0; i < n; i++) {
    double skip, muB = 0.0, nB = 0.0;
    rd(&s->tau[i]); rd(&s->x[i]); rd(&s->y[i]); rd(&s->eta[i]);
    const double tau = s->tau[i];
    if (mode == 4 || mode == 6 || mode == 7) {
      // boost-invariant formats (MUSIC old :552-681, MUSIC new :683-810, hic-eventgen :1059-1196): eta := 0, dsigma stored / tau
      s->eta[i] = 0.0;
      double a;
      rd(&a); s->dat[i] = a * tau; rd(&a); s->dax[i] = a * tau; rd(&a); s->day[i] = a * tau; rd(&a); s->dan[i] = a * tau;
      if (mode != 4 || fl.dimension == 2) s->dan[i] = 0.0;
    } else {
      rd(&s->dat[i]); rd(&s->dax[i]); rd(&s->day[i]); rd(&s->dan[i]);
      if (fl.dimension == 2 && s->dan[i] != 0 && mode == 0) {
        if (err) *err = "2+1d boost invariant surface read-in error at cell # " + std::to_string(i) + ": dsigma_eta is not zero";
        return false;                                                         // mode 0 exits here (readindata.cpp:183-187)
      }
    }
    double PLfile = 0, Pfile = 0, Tfile = 0;
    if (mode == 7) {
      // velocities instead of u^mu; every dissipative quantity already in GeV units
      double vx, vy, vn; rd(&vx); rd(&vy); rd(&vn);
      const double ut = std::sqrt(1.0 / (1.0 - (vx * vx) - (vy * vy)));
      s->ux[i] = ut * vx; s->uy[i] = ut * vy; s->un[i] = 0.0;
      double a;
      rd(&skip); rd(&skip); rd(&skip); rd(&skip);                             // pi^tt, pi^tx, pi^ty, pi^tz
      rd(&s->pixx[i]); rd(&s->pixy[i]); rd(&a); s->pixn[i] = a / tau; rd(&s->piyy[i]); rd(&a); s->piyn[i] = a / tau; rd(&skip);
      rd(&s->bulkPi[i]); rd(&s->T[i]); rd(&s->E[i]); rd(&s->P[i]); rd(&muB); s->muB[i] = muB;
    } else {
      if (mode == 0 || mode == 2 || mode == 4 || mode == 6) rd(&skip);          // u^tau column (recomputed from u^i)
      rd(&s->ux[i]); rd(&s->uy[i]); rd(&s->un[i]);
      if (mode == 4 || mode == 6) s->un[i] = s->un[i] / tau;
      double Efile;
      rd(&Efile); rd(&Tfile);
      s->E[i] = Efile * kHbarC; s->T[i] = Tfile * kHbarC;
      if (mode == 4 || mode == 6) {
        rd_gev(&muB); s->muB[i] = muB;                                           // always present in the MUSIC formats
        if (mode == 6) { rd(&skip); rd(&skip); }                                 // mu_S, mu_C
        double sdens; rd(&sdens);
        s->P[i] = sdens * s->T[i] - s->E[i];                                     // p = T s - e
      } else {
        rd(&Pfile); s->P[i] = Pfile * kHbarC;
      }
      if (mode == 2) { rd(&PLfile); s->PL[i] = PLfile * kHbarC; }
      if (full_pi) { rd_gev(&s->pitt[i]); rd_gev(&s->pitx[i]); rd_gev(&s->pity[i]); rd_gev(&s->pitn[i]); }
      rd_gev(&s->pixx[i]); rd_gev(&s->pixy[i]); rd_gev(&s->pixn[i]); rd_gev(&s->piyy[i]); rd_gev(&s->piyn[i]);
      if (full_pi) rd_gev(&s->pinn[i]);
      if (mode == 4 || mode == 6) {                                              // MUSIC stores tau * pi^{mu eta}
        s->pitn[i] = s->pitn[i] / tau; s->pixn[i] = s->pixn[i] / tau; s->piyn[i] = s->piyn[i] / tau; s->pinn[i] = s->pinn[i] / tau / tau;
      }
      if (mode == 2) { double wt, wn; rd(&wt); rd_gev(&s->Wx[i]); rd_gev(&s->Wy[i]); rd(&wn); }
      rd_gev(&s->bulkPi[i]);
      if (mode == 0 || mode == 1 || mode == 5) {
        if (fl.include_baryon) { rd_gev(&muB); s->muB[i] = muB; }
        if (fl.include_baryondiff_deltaf) {
          rd(&nB); s->nB[i] = nB;
          if (mode == 0 || mode == 5) rd(&skip);                                  // V^tau column
          rd(&s->Vx[i]); rd(&s->Vy[i]); rd(&s->Vn[i]);
        }
        if (mode == 5) { rd(&s->wtx[i]); rd(&s->wty[i]); rd(&s->wtn[i]); rd(&s->wxy[i]); rd(&s->wxn[i]); rd(&s->wyn[i]); }   // thermal vorticity
      }
    }
    if (writes_averages) {
      // surface averages weighted with |u.dsigma| + sqrt(|(u.dsigma)^2 - dsigma.dsigma|) (readindata.cpp:423-452).
      // (mode 7: the reference evaluates u.dsigma from uninitialised locals -- undefined behaviour; the stored u^mu is used here)
      const double ux = s->ux[i], uy = s->uy[i], un = s->un[i];
      const double ut = std::sqrt(1.0 + ux * ux + uy * uy + tau * tau * un * un);
      const double dat = s->dat[i], dax = s->dax[i], day = s->day[i], dan = s->dan[i];
      const double udsigma = ut * dat + ux * dax + uy * day + un * dan;
      const double dsds = dat * dat - dax * dax - day * day - dan * dan / (tau * tau);
      const double mag = std::fabs(udsigma) + std::sqrt(std::fabs(udsigma * udsigma - dsds));
      volume += mag;
      Eavg += (s->E[i] * mag); Tavg += (s->T[i] * mag); Pavg += (s->P[i] * mag); muBavg += (muB * mag); nBavg += (nB * mag);
    }
    if (mode == 2) {
      // conformal factorisation: alpha_L from PL/P, Lambda from T (readindata.cpp:905-918)
      if (!((PLfile / Pfile) < 3.0)) { if (err) *err = "pl is too large, stopping anisotropic variables"; return false; }
      const double aLv = aL_fit(PLfile / Pfile);
      const double Lam = Tfile / std::pow(0.5 * aLv * R200(aLv), 0.25);
      s->aL[i] = aLv; s->Lambda[i] = Lam * kHbarC;
    }
  }
  if (short_file) { if (err) *err = "surface file " + path + " has fewer values than " + std::to_string(n) + " cells need"; return false; }

  const std::string apath = workdir + "/average_thermodynamic_quantities.dat";
  if (writes_averages) {
    Tavg /= volume; Eavg /= volume; Pavg /= volume; muBavg /= volume; nBavg /= volume;
    // side file: 15 significant digits, default float format (readindata.cpp:463-466), re-read by
    // Plasma::load_thermodynamic_averages (:90-100) -- the round trip is part of the reference's arithmetic
    FILE *f = std::fopen(apath.c_str(), "w");
    if (!f) { if (err) *err = "cannot write " + apath; return false; }
    std::fprintf(f, "%.15g\n%.15g\n%.15g\n%.15g\n%.15g", Tavg, Eavg, Pavg, muBavg, nBavg);
    std::fclose(f);
  }
  if (mode != 2) {
    // modes that do not write the file read whatever an earlier run left there, like the reference
    FILE *f = std::fopen(apath.c_str(), "r");
    if (f && std::fscanf(f, "%lf\n%lf\n%lf\n%lf\n%lf", &s->avg[0], &s->avg[1], &s->avg[2], &s->avg[3], &s->avg[4]) == 5) s->averages_written = true;
    if (f) std::fclose(f);
    if (!s->averages_written && (writes_averages || fl.df_mode == 4)) { if (err) *err = "cannot read " + apath; return false; }
  }
  return true;
}

// ------------------------------------------------------------------------------------------------ delta-f tables
bool read_df_tables(const std::string &workdir, int hrg_eos, DfTables *t, std::string *err)
{
  const char *dir = hrg_eos == 1 ? "urqmd" : hrg_eos == 2 ? "smash" : hrg_eos == 3 ? "smash_box" : nullptr;
  if (!dir) { if (err) *err = "please choose hrg_eos = (1,2,3)"; return false; }
  const std::string base = workdir + "/deltaf_coefficients/vh/" + dir + "/";
  struct Item { const char *name; std::vector<double> *dst; } items[] = {
    {"c0", &t->c0}, {"c1", &t->c1}, {"c2", &t->c2}, {"c3", &t->c3}, {"c4", &t->c4}, {"F", &t->F}, {"G", &t->G},
    {"betabulk", &t->betabulk}, {"betaV", &t->betaV}, {"betapi", &t->betapi}};
  for (auto &it : items) {
    const std::string path = base + it.name + ".dat";
    FILE *f = std::fopen(path.c_str(), "r");
    if (!f) { if (err) *err = "couldn't open " + path; return false; }
    int nT = 0, nB = 0; char header[300];
    if (std::fscanf(f, "%d\n%d\n", &nT, &nB) != 2 || nT < 2) { std::fclose(f); if (err) *err = "bad header in " + path; return false; }
    if (!std::fgets(header, 100, f)) { std::fclose(f); if (err) *err = "bad header in " + path; return false; }
    t->n_T = nT; t->n_muB_file = nB;
    t->T.assign(nT, 0.0); it.dst->assign(nT, 0.0);
    for (int iT = 0; iT < nT; iT++) {                    // first block = muB = 0 (include_baryon = 0: points_muB forced to 1)
      double mu;
      if (std::fscanf(f, "%lf\t\t%lf\t\t%lf\n", &t->T[iT], &mu, &(*it.dst)[iT]) != 3) {
        std::fclose(f); if (err) *err = "short table " + path; return false;
      }
    }
    std::fclose(f);
  }
  return true;
}

bool read_laguerre(const std::string &path, Laguerre *g, std::string *err)
{
  FILE *f = std::fopen(path.c_str(), "r");
  if (!f) { if (err) *err = "couldn't open gauss laguerre file " + path; return false; }
  if (std::fscanf(f, "%d\t%d", &g->alpha, &g->points) != 2) { std::fclose(f); if (err) *err = "bad header in " + path; return false; }
  g->root.assign(g->alpha, std::vector<double>(g->points)); g->weight = g->root;
  for (int a = 0; a < g->alpha; a++)
    for (int j = 0; j < g->points; j++) {
      int dummy;
      if (std::fscanf(f, "%d\t%lf\t%lf", &dummy, &g->root[a][j], &g->weight[a][j]) != 3) { std::fclose(f); if (err) *err = "short file " + path; return false; }
    }
  std::fclose(f);
  return true;
}

// ------------------------------------------------------------------------------------------------ Jonah tables
void compute_jonah_tables(const std::vector<Particle> &pdg, double T, const Laguerre &gla, DfTables *tab)
{
  const int npts = 301;
  const double lam_min = -1.0, lam_max = 2.0, dlam = (lam_max - lam_min) / ((double)npts - 1.0);
  const std::vector<double> &root = gla.root[2], &wgt = gla.weight[2];
  tab->jonah_x.assign(npts, 0.0); tab->jonah_lambda2.assign(npts, 0.0); tab->jonah_z.assign(npts, 0.0);
  tab->bulkPi_over_Peq_max = -1.0;
  // kinetic-theory energy density / pressure integrands with momenta rescaled by (1 + lambda), gaussThermal.cpp:100-115
  auto e_term = [](double pbar, double mbar, double lam, double sign) {
    const double sc2 = (1.0 + lam) * (1.0 + lam), Ebar = std::sqrt(pbar * pbar + mbar * mbar);
    return std::sqrt(pbar * pbar * sc2 + mbar * mbar) * std::exp(pbar) / (std::exp(Ebar) + sign);
  };
  auto p_term = [](double pbar, double mbar, double lam, double sign) {
    const double sc2 = (1.0 + lam) * (1.0 + lam), Ebar = std::sqrt(pbar * pbar + mbar * mbar);
    return pbar * pbar * sc2 / std::sqrt(pbar * pbar * sc2 + mbar * mbar) * std::exp(pbar) / (std::exp(Ebar) + sign);
  };
  for (int i = 0; i < npts; i++) {
    const double lam = lam_min + (double)i * dlam;
    double E = 0, P = 0, Em = 0, Pm = 0;
    for (const Particle &h : pdg) {
      if (h.mass == 0.0) continue;                        // photon: breaks down at lambda = -1
      const double g = (double)h.gspin, sgn = (double)h.sign, mbar = h.mass / T;
      double e0 = 0, p0 = 0, e1 = 0, p1 = 0;
      for (size_t k = 0; k < root.size(); k++) e0 += wgt[k] * e_term(root[k], mbar, 0.0, sgn);
      for (size_t k = 0; k < root.size(); k++) p0 += wgt[k] * p_term(root[k], mbar, 0.0, sgn);
      for (size_t k = 0; k < root.size(); k++) e1 += wgt[k] * e_term(root[k], mbar, lam, sgn);
      for (size_t k = 0; k < root.size(); k++) p1 += wgt[k] * p_term(root[k], mbar, lam, sgn);
      E += g * e0; P += (1.0 / 3.0) * g * p0; Em += g * e1; Pm += (1.0 / 3.0) * g * p1;
    }
    const double z = E / Em, x = (Pm / P) * z - 1.0;
    tab->jonah_lambda2[i] = lam * lam; tab->jonah_z[i] = z; tab->jonah_x[i] = x;
    tab->bulkPi_over_Peq_max = std::max(tab->bulkPi_over_Peq_max, x);
  }
}

// ------------------------------------------------------------------------------------------------ anisotropic helpers
double aL_fit(double x)
{
  // rational fit alpha_L(PL/Peq), conformal factorisation approximation: coefficients from arsenal.cpp:1021-1025
  static const double num[15] = {2.307660683188896e-22, 1.7179667824677117e-16, 7.2725449826862375e-12, 4.2846163672079405e-8,
    0.00004757224421671691, 0.011776118846199547, 0.7235583305942909, 11.582755440134724, 44.45243622597357, 12.673594148032494,
    -33.75866652773691, 8.04299287188939, 1.462901772148128, -0.6320131889637761, 0.048528166213735346};
  static const double den[15] = {5.595674409987461e-19, 8.059757191879689e-14, 1.2033043382301483e-9, 2.9819348588423508e-6,
    0.0015212379997299082, 0.18185453852532632, 5.466199358534425, 40.1581708710626, 44.38310108782752, -55.213789667214364,
    1.5449108423263358, 11.636087951096759, -4.005934533735304, 0.4703844693488544, -0.014599143701745957};
  double xp = 1.0, a = 0.0, b = 0.0;
  for (int k = 0; k < 15; k++) { a += num[k] * xp; b += den[k] * xp; xp *= x; }
  return a / b;
}

double R200(double aL)
{
  const double x = (1.0 / (aL * aL)) - 1.0, delta = 0.01;
  double t200;
  if (x > delta) t200 = 1.0 + (1.0 + x) * std::atan(std::sqrt(x)) / std::sqrt(x);
  else if (x < -delta && x > -1.0) t200 = 1.0 + (1.0 + x) * std::atanh(std::sqrt(-x)) / std::sqrt(-x);
  else if (x >= -delta && x <= delta)
    t200 = 2.0 + x * (0.6666666666666667 + x * (-0.1333333333333333 + x * (0.05714285714285716 + x * (-0.031746031746031744 +
           x * (0.020202020202020193 + x * (-0.013986013986013984 + (0.010256410256410262 - 0.00784313725490196 * x) * x))))));
  else return NAN;
  return aL * t200;
}

// bilinear lookup of one cell's c0..c4 in the (Lambda [fm^-1], alpha_L) tables; tables are [iL * naL + iaL]
bool vah_lookup(int nL, int naL, const double *L, const double *aLv, const double *const c[5], double Lam_fm, double a, double out[5])
{
  // first table cell with Lambda < L[i1] and aL < aL[i2] (i1, i2 >= 1), as the loops of src/cuda/deltafReader.cu:222-277 find it
  int i2 = 1; while (i2 < naL && !(a < aLv[i2])) i2++;
  int i1 = 1; while (i1 < nL && !(Lam_fm < L[i1])) i1++;
  if (i1 >= nL || i2 >= naL) return false;
  const double hbarC3 = kHbarC * kHbarC * kHbarC;
  const double L1 = L[i1 - 1], L2 = L[i1], a1 = aLv[i2 - 1], a2 = aLv[i2];
  for (int k = 0; k < 5; k++) {
    const double f11 = c[k][(size_t)(i1 - 1) * naL + (i2 - 1)], f21 = c[k][(size_t)i1 * naL + (i2 - 1)];
    const double f12 = c[k][(size_t)(i1 - 1) * naL + i2], f22 = c[k][(size_t)i1 * naL + i2];
    const double v = ((f11 * (L2 - Lam_fm) + f21 * (Lam_fm - L1)) * (a2 - a) + (f12 * (L2 - Lam_fm) + f22 * (Lam_fm - L1)) * (a - a1)) / ((a2 - a1) * (L2 - L1));
    out[k] = v / hbarC3;
  }
  return true;
}

bool read_vah_tables(const std::string &workdir, VahTables *t, std::string *err)
{
  for (int k = 0; k < 5; k++) {
    const std::string path = workdir + "/deltaf_coefficients/vah/c" + std::to_string(k) + "_vah1.dat";
    FILE *f = std::fopen(path.c_str(), "r");
    if (!f) { if (err) *err = "couldn't open " + path; return false; }
    char header[300];
    if (std::fscanf(f, "%d\n%d\n", &t->nL, &t->naL) != 2 || !std::fgets(header, 100, f)) { std::fclose(f); if (err) *err = "bad header in " + path; return false; }
    t->L.assign(t->nL, 0.0); t->aL.assign(t->naL, 0.0); t->c[k].assign((size_t)t->nL * t->naL, 0.0);
    for (int i2 = 0; i2 < t->naL; i2++)
      for (int i1 = 0; i1 < t->nL; i1++)
        if (std::fscanf(f, "%lf\t\t%lf\t\t%lf\n", &t->L[i1], &t->aL[i2], &t->c[k][(size_t)i1 * t->naL + i2]) != 3) { std::fclose(f); if (err) *err = "short table " + path; return false; }
    std::fclose(f);
  }
  return true;
}

bool fill_vah_coefficients(const std::string &workdir, SurfaceData *s, std::string *err)
{
  VahTables t;
  if (!read_vah_tables(workdir, &t, err)) return false;
  const double *c[5] = {t.c[0].data(), t.c[1].data(), t.c[2].data(), t.c[3].data(), t.c[4].data()};
  for (int64_t i = 0; i < s->n; i++) {
    double out[5];
    if (!vah_lookup(t.nL, t.naL, t.L.data(), t.aL.data(), c, s->Lambda[i] / kHbarC, s->aL[i], out)) {
      if (err) *err = "cell " + std::to_string(i) + ": (Lambda, alpha_L) outside the vah coefficient table"; return false;
    }
    s->c0[i] = out[0]; s->c1[i] = out[1]; s->c2[i] = out[2]; s->c3[i] = out[3]; s->c4[i] = out[4];
  }
  return true;
}

}  // namespace is3d
