// els_host -- C++ host program above the C ABI (include/afesp_gpu.h): the drop-in stand-in for AFESP's `els.x`.
//
// The reference's main program (src/main.F90:20-187) is Fortran; this image has no Fortran compiler (SURVEY.md K5), so
// the host side of the boundary is written in C++ and follows main.F90 step by step:
//   read_system_in      els.in namelist                    src/system.f90:81-165
//   read_integrals_in   s.dat t.dat v.dat eri.dat           src/integrals.f90:48-165   (8-fold packing :196-210)
//   read_geometry_in    geom.dat, nel, E_nuc                src/geometry.f90:8-95
//   do_rhf              symmetric orthogonalisation, DIIS   src/hf.f90:21-151, 197-385  (host: outside the hot path)
//   do_mp2_spatial      -> afesp_gpu_ao2mo / afesp_gpu_mp2_energy
//   do_ccsd_*           -> afesp_gpu_ccsd_init / _iterate / _diis / _finalize   (host keeps loop, table, convergence)
//   do_ccsd_t_*         -> afesp_gpu_ccsd_t_spatial / _spinorb                   (host assembles the printed energies)
// and prints the same els.out (formats of the shipped sample outputs; only dates and wall-clock times differ), writes
// guess_out.dat (src/hf.f90:172-191) and FCIDUMP (src/mp2.f90:451-487) into the working directory, and stops with the
// reference's error block + exit status 999 & 0xff on failure (src/error_handling.f90:6-20).
//
//   usage:  els_host [--device N] [directory]        (directory defaults to the current one, as for els.x)
//
// Everything from the AO->MO transform on runs on the GPU through the C ABI; there is no CPU fallback.
#include <algorithm>
#include <cctype>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <fstream>
#include <map>
#include <sstream>
#include <string>
#include <vector>

#include <unistd.h>

#include "../include/afesp_gpu.h"

namespace {

using Clock = std::chrono::steady_clock;
double since(Clock::time_point t0) { return std::chrono::duration<double>(Clock::now() - t0).count(); }

// ---------------------------------------------------------------------------------------------- error handling
[[noreturn]] void fail(const std::string& procedure, const std::string& msg) {  // src/error_handling.f90:6-20
  std::fprintf(stderr, " ERROR.\n Programme stops in procedure: %s.\n Reason: %s.\n EXITING...\nSTOP 999\n",
               procedure.c_str(), msg.c_str());
  std::fflush(stdout);
  std::exit(999 & 0xff);
}

// host/gint.c: Gaussian integrals over a built-in basis set (returns nbf; outputs may be NULL)
extern "C" int afesp_gint_named(int natom, const double* Z, const double* xyz, const char* basis, double* Smat, double* Tmat,
                                double* Vmat, double* eri);

afesp_handle g_h = nullptr;
void check(const char* fn, int rc) {
  if (rc != 0) fail(std::string("afesp_gpu::") + fn, afesp_gpu_last_error(g_h));
}

// ---------------------------------------------------------------------------------------------- input
struct Sys {
  std::string calc_type = "CCSD(T)_spatial", els_in_text;
  double scf_e_tol = 1e-6, scf_d_tol = 1e-6, ccsd_e_tol = 1e-6, ccsd_t_tol = 1e-6;
  int scf_diis_n_errmat = 6, ccsd_diis_n_errmat = 8, scf_maxiter = 50, ccsd_maxiter = 50;
  bool write_fcidump = false, scf_read_guess = false, scf_write_guess = false;
  int frozen_core = 0;   // frozen doubly occupied orbitals (extension of the namelist; 0 = all-electron)
  int nbasis = 0, nel = 0;
  double e_nuc = 0.0;
  std::vector<double> ovlp, hcore, eri, guess;  // n x n row-major (symmetric), packed ERIs
  // calc_type flags (src/system.f90:116-165)
  int level = 0;  // 0 HF, 1 MP2, 2 CCSD, 3 CCSD(T)
  bool restricted = true, paren = false, renorm = false, comp_renorm = false;
};

std::string trim(const std::string& s) {
  size_t a = s.find_first_not_of(" \t\r\n"), b = s.find_last_not_of(" \t\r\n");
  return a == std::string::npos ? "" : s.substr(a, b - a + 1);
}
std::string lower(std::string s) {
  for (char& c : s) c = (char)std::tolower((unsigned char)c);
  return s;
}

void set_calc_type(Sys& s) {
  struct Row { const char* name; int level; bool restricted, paren, renorm, cr; };
  static const Row rows[] = {
      {"RHF", 0, true, false, false, false},          {"UHF", 0, false, false, false, false},
      {"MP2_spinorb", 1, false, false, false, false}, {"MP2_spatial", 1, true, false, false, false},
      {"CCSD_spinorb", 2, false, false, false, false}, {"CCSD_spatial", 2, true, false, false, false},
      {"CCSD(T)_spinorb", 3, false, false, false, false}, {"CCSD(T)_spatial", 3, true, true, false, false},
      {"CCSD[T]_spatial", 3, true, false, false, false},  {"RCCSD(T)_spatial", 3, true, true, true, false},
      {"RCCSD[T]_spatial", 3, true, false, true, false},  {"CRCCSD(T)_spatial", 3, true, true, false, true},
      {"CRCCSD[T]_spatial", 3, true, false, false, true}};
  for (const Row& r : rows)
    if (s.calc_type == r.name) {
      s.level = r.level; s.restricted = r.restricted; s.paren = r.paren; s.renorm = r.renorm; s.comp_renorm = r.cr;
      return;
    }
  fail("system::read_system_in", "Unrecognised calculation type!");
}

void read_system_in(Sys& s) {
  std::ifstream f("els.in");
  if (!f) fail("system::read_system_in", "input file els.in does not exist");
  std::stringstream ss;
  ss << f.rdbuf();
  s.els_in_text = ss.str();
  // `read(unit=ir, nml=elsinput)` (src/system.f90:105) with Fortran namelist rules: the group starts at `&elsinput` (any
  // case) and ends at the first `/` outside a string; `!` starts a comment; assignments are separated by commas, blanks
  // or line ends; names are case-insensitive.  Whatever the runtime would refuse is the reference's error (:107).
  auto bad = [&]() { fail("system::read_system_in", "invalid input file format!"); };
  std::string flat;
  {
    char quote = 0;
    bool comment = false;
    for (char ch : s.els_in_text) {
      if (ch == '\n') { comment = false; flat.push_back(ch); continue; }
      if (comment) continue;
      if (quote) { if (ch == quote) quote = 0; }
      else if (ch == '"' || ch == '\'') quote = ch;
      else if (ch == '!') { comment = true; continue; }
      flat.push_back(ch);
    }
  }
  const std::string lo = lower(flat);
  size_t pos = lo.find("&elsinput");
  if (pos == std::string::npos) bad();
  pos += 9;
  if (pos < lo.size() && (std::isalnum((unsigned char)lo[pos]) || lo[pos] == '_')) bad();
  auto skip_sep = [&]() {
    bool comma = false;
    while (pos < flat.size() && (std::isspace((unsigned char)flat[pos]) || (flat[pos] == ',' && !comma))) {
      if (flat[pos] == ',') comma = true;
      ++pos;
    }
  };
  auto as_bool = [&](const std::string& x) {
    std::string y = lower(x);
    while (!y.empty() && y[0] == '.') y.erase(0, 1);
    if (y.empty() || (y[0] != 't' && y[0] != 'f')) bad();
    return y[0] == 't';
  };
  auto as_real = [&](std::string x) {
    for (char& c : x) if (c == 'd' || c == 'D') c = 'e';
    char* end = nullptr;
    double r = std::strtod(x.c_str(), &end);
    if (end == x.c_str() || *end != 0) bad();
    return r;
  };
  auto as_int = [&](const std::string& x) {
    char* end = nullptr;
    long r = std::strtol(x.c_str(), &end, 10);
    if (end == x.c_str() || *end != 0) bad();
    return (int)r;
  };
  bool closed = false;
  while (!closed) {
    skip_sep();
    if (pos >= flat.size()) bad();   // group never closed
    if (flat[pos] == '/') { closed = true; break; }
    if (lo.compare(pos, 4, "&end") == 0) { closed = true; break; }
    size_t k0 = pos;
    while (pos < flat.size() && (std::isalnum((unsigned char)flat[pos]) || flat[pos] == '_')) ++pos;
    if (pos == k0) bad();
    const std::string k = lo.substr(k0, pos - k0);
    while (pos < flat.size() && std::isspace((unsigned char)flat[pos])) ++pos;
    if (pos >= flat.size() || flat[pos] != '=') bad();
    ++pos;
    while (pos < flat.size() && std::isspace((unsigned char)flat[pos])) ++pos;
    std::string v;
    if (pos < flat.size() && (flat[pos] == '"' || flat[pos] == '\'')) {
      const char q = flat[pos++];
      size_t e = flat.find(q, pos);
      if (e == std::string::npos) bad();
      v = flat.substr(pos, e - pos);
      pos = e + 1;
    } else {
      size_t v0 = pos;
      while (pos < flat.size() && !std::isspace((unsigned char)flat[pos]) && flat[pos] != ',' && flat[pos] != '/') ++pos;
      v = flat.substr(v0, pos - v0);
      if (v.empty()) bad();
    }
    if (k == "calc_type") s.calc_type = trim(v);
    else if (k == "scf_e_tol") s.scf_e_tol = as_real(v);
    else if (k == "scf_d_tol") s.scf_d_tol = as_real(v);
    else if (k == "ccsd_e_tol") s.ccsd_e_tol = as_real(v);
    else if (k == "ccsd_t_tol") s.ccsd_t_tol = as_real(v);
    else if (k == "scf_diis_n_errmat") s.scf_diis_n_errmat = as_int(v);
    else if (k == "ccsd_diis_n_errmat") s.ccsd_diis_n_errmat = as_int(v);
    else if (k == "scf_maxiter") s.scf_maxiter = as_int(v);
    else if (k == "ccsd_maxiter") s.ccsd_maxiter = as_int(v);
    else if (k == "write_fcidump") s.write_fcidump = as_bool(v);
    else if (k == "scf_read_guess") s.scf_read_guess = as_bool(v);
    else if (k == "scf_write_guess") s.scf_write_guess = as_bool(v);
    else if (k == "frozen_core") s.frozen_core = as_int(v);
    else bad();
  }
  set_calc_type(s);
}

inline long long pair_index(long long i, long long j) { return i >= j ? i * (i + 1) / 2 + j : j * (j + 1) / 2 + i; }

// free-format "i j value" triples of a symmetric matrix (src/integrals.f90:101-141)
std::vector<double> read_sym(const char* file, int n) {
  std::ifstream f(file);
  if (!f) fail("integrals::read_integrals_in", std::string("cannot open ") + file);
  std::vector<double> m((size_t)n * n, 0.0);
  long long i, j;
  double v;
  while (f >> i >> j >> v) {
    if (i < 1 || j < 1 || i > n || j > n) fail("integrals::read_integrals_in", std::string("index out of range in ") + file);
    m[(size_t)(i - 1) * n + (j - 1)] = v;
    m[(size_t)(j - 1) * n + (i - 1)] = v;
  }
  return m;
}

void read_integrals_in(Sys& s) {
  {  // first pass over s.dat finds nbasis (src/integrals.f90:81-93)
    std::ifstream f("s.dat");
    if (!f) fail("integrals::read_integrals_in", "cannot open s.dat");
    long long i, j;
    double v;
    int n = 0;
    while (f >> i >> j >> v) n = (int)std::max<long long>(n, std::max(i, j));
    if (n <= 0) fail("integrals::read_integrals_in", "s.dat is empty");
    s.nbasis = n;
  }
  const int n = s.nbasis;
  s.ovlp = read_sym("s.dat", n);
  std::vector<double> ke = read_sym("t.dat", n), en = read_sym("v.dat", n);
  s.hcore.resize((size_t)n * n);
  for (size_t k = 0; k < s.hcore.size(); ++k) s.hcore[k] = ke[k] + en[k];
  const long long npair = (long long)n * (n + 1) / 2;
  s.eri.assign((size_t)(npair * (npair + 1) / 2), 0.0);
  {
    // Extension for large basis sets (SURVEY.md section 8f-3): a text eri.dat at nbf = 400 would be ~3e9 lines and the
    // reference's default-integer pair index overflows there.  If `eri.bin` is present it is taken instead: the packed
    // 8-fold-unique array itself (npair(npair+1)/2 little-endian doubles, canonical order of src/integrals.f90:196-210,
    // 64-bit indices).
    std::ifstream fb("eri.bin", std::ios::binary);
    if (fb) {
      fb.read(reinterpret_cast<char*>(s.eri.data()), (std::streamsize)(s.eri.size() * sizeof(double)));
      if ((size_t)fb.gcount() != s.eri.size() * sizeof(double) || fb.peek() != EOF)
        fail("integrals::read_integrals_in", "eri.bin does not hold npair(npair+1)/2 doubles for this basis");
      return;
    }
  }
  std::ifstream f("eri.dat");
  if (!f) {
    // Extension (SURVEY.md section 8f-4): no eri.dat in the run directory (the reference checkout ships none for
    // sample_data/h2o-cc-pvtz).  If the basis set is named -- a one-line file `basis.dat`, or AFESP_BASIS in the
    // environment -- the two-electron integrals are generated from geom.dat by the built-in integral code (host/gint.c,
    // Psi4 conventions; the shipped s/t/v.dat are reproduced to 1e-14, tests/test_gint.py).
    std::string basis;
    { std::ifstream fbas("basis.dat"); if (fbas) fbas >> basis; }
    if (basis.empty()) if (const char* env = std::getenv("AFESP_BASIS")) basis = env;
    if (basis.empty()) fail("integrals::read_integrals_in", "cannot open eri.dat");
    std::ifstream fg("geom.dat");
    if (!fg) fail("integrals::read_integrals_in", "cannot open eri.dat (and no geom.dat to generate it from)");
    int nat = 0;
    fg >> nat;
    std::vector<double> Z(nat), xyz((size_t)3 * nat);
    for (int a = 0; a < nat; ++a)
      if (!(fg >> Z[a] >> xyz[3 * a] >> xyz[3 * a + 1] >> xyz[3 * a + 2]))
        fail("integrals::read_integrals_in", "geom.dat is truncated");
    const int nb = afesp_gint_named(nat, Z.data(), xyz.data(), basis.c_str(), nullptr, nullptr, nullptr, nullptr);
    if (nb == -2) fail("integrals::read_integrals_in", "no built-in parameters for basis set " + basis + " on these atoms");
    if (nb != n) fail("integrals::read_integrals_in", "basis set " + basis + " does not match s.dat (" + std::to_string(nb) +
                                                      " functions, s.dat has " + std::to_string(n) + ")");
    std::vector<double> S((size_t)n * n);
    afesp_gint_named(nat, Z.data(), xyz.data(), basis.c_str(), S.data(), nullptr, nullptr, s.eri.data());
    double dmax = 0.0;   // the generated overlap must be the one in s.dat: same basis, ordering, normalisation
    for (size_t q = 0; q < S.size(); ++q) dmax = std::max(dmax, std::fabs(S[q] - s.ovlp[q]));
    if (dmax > 1e-10) fail("integrals::read_integrals_in", "generated overlap matrix differs from s.dat (basis set " + basis + "?)");
    return;
  }
  long long i, j, k, l;
  double v;
  while (f >> i >> j >> k >> l >> v) {
    if (std::min({i, j, k, l}) < 1 || std::max({i, j, k, l}) > n)
      fail("integrals::read_integrals_in", "index out of range in eri.dat");
    s.eri[(size_t)pair_index(pair_index(i - 1, j - 1), pair_index(k - 1, l - 1))] = v;
  }
}

void read_geometry_in(Sys& s) {
  std::ifstream f("geom.dat");
  if (!f) fail("geometry::read_geometry_in", "cannot open geom.dat");
  int nat = 0;
  f >> nat;
  std::vector<int> z(nat);
  std::vector<double> xyz((size_t)3 * nat);
  for (int a = 0; a < nat; ++a) {
    double charge;
    if (!(f >> charge >> xyz[3 * a] >> xyz[3 * a + 1] >> xyz[3 * a + 2]))
      fail("geometry::read_geometry_in", "geom.dat is truncated");
    z[a] = (int)charge;  // charges(i) = int(charge)
  }
  s.nel = 0;
  for (int q : z) s.nel += q;
  s.e_nuc = 0.0;  // get_e_nuc (src/geometry.f90:74-95)
  for (int b = 1; b < nat; ++b)
    for (int a = 0; a < b; ++a) {
      double d2 = 0.0;
      for (int c = 0; c < 3; ++c) d2 += (xyz[3 * a + c] - xyz[3 * b + c]) * (xyz[3 * a + c] - xyz[3 * b + c]);
      s.e_nuc += z[a] * z[b] / std::sqrt(d2);
    }
}

// ---------------------------------------------------------------------------------------------- small dense algebra
// Cyclic Jacobi for a real symmetric matrix (row-major n x n): eigenvalues ascending in w, eigenvectors as the COLUMNS
// of V.  The reference calls LAPACK dsyev (src/linalg.fpp:18-36); both are accurate to a few ulps of |A|, which is far
// inside the 1e-10 the SCF table is printed with.
void eigh(std::vector<double> A, int n, std::vector<double>& w, std::vector<double>& V) {
  V.assign((size_t)n * n, 0.0);
  for (int i = 0; i < n; ++i) V[(size_t)i * n + i] = 1.0;
  for (int sweep = 0; sweep < 100; ++sweep) {
    double off = 0.0, diag = 0.0;
    for (int i = 0; i < n; ++i)
      for (int j = 0; j < n; ++j) (i == j ? diag : off) += A[(size_t)i * n + j] * A[(size_t)i * n + j];
    if (off <= 1e-60 || off <= 1e-34 * diag) break;
    for (int p = 0; p < n - 1; ++p)
      for (int q = p + 1; q < n; ++q) {
        const double apq = A[(size_t)p * n + q];
        if (apq == 0.0) continue;
        const double theta = (A[(size_t)q * n + q] - A[(size_t)p * n + p]) / (2.0 * apq);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double c = 1.0 / std::sqrt(t * t + 1.0), sn = t * c;
        for (int k = 0; k < n; ++k) {
          const double akp = A[(size_t)k * n + p], akq = A[(size_t)k * n + q];
          A[(size_t)k * n + p] = c * akp - sn * akq;
          A[(size_t)k * n + q] = sn * akp + c * akq;
        }
        for (int k = 0; k < n; ++k) {
          const double apk = A[(size_t)p * n + k], aqk = A[(size_t)q * n + k];
          A[(size_t)p * n + k] = c * apk - sn * aqk;
          A[(size_t)q * n + k] = sn * apk + c * aqk;
        }
        for (int k = 0; k < n; ++k) {
          const double vkp = V[(size_t)k * n + p], vkq = V[(size_t)k * n + q];
          V[(size_t)k * n + p] = c * vkp - sn * vkq;
          V[(size_t)k * n + q] = sn * vkp + c * vkq;
        }
      }
  }
  std::vector<int> order(n);
  for (int i = 0; i < n; ++i) order[i] = i;
  std::stable_sort(order.begin(), order.end(),
                   [&](int a, int b) { return A[(size_t)a * n + a] < A[(size_t)b * n + b]; });
  w.resize(n);
  std::vector<double> Vs((size_t)n * n);
  for (int c = 0; c < n; ++c) {
    w[c] = A[(size_t)order[c] * n + order[c]];
    for (int r = 0; r < n; ++r) Vs[(size_t)r * n + c] = V[(size_t)r * n + order[c]];
  }
  V.swap(Vs);
}

std::vector<double> matmul(const std::vector<double>& A, const std::vector<double>& B, int n, bool ta = false,
                           bool tb = false) {
  std::vector<double> C((size_t)n * n, 0.0);
  for (int i = 0; i < n; ++i)
    for (int k = 0; k < n; ++k) {
      const double a = ta ? A[(size_t)k * n + i] : A[(size_t)i * n + k];
      if (a == 0.0) continue;
      for (int j = 0; j < n; ++j) C[(size_t)i * n + j] += a * (tb ? B[(size_t)j * n + k] : B[(size_t)k * n + j]);
    }
  return C;
}

// Gaussian elimination with partial pivoting (the DIIS system is at most 9 x 9; the reference uses dsysv).
bool solve(std::vector<double> A, std::vector<double> b, int n, std::vector<double>& x) {
  for (int c = 0; c < n; ++c) {
    int piv = c;
    for (int r = c + 1; r < n; ++r)
      if (std::fabs(A[(size_t)r * n + c]) > std::fabs(A[(size_t)piv * n + c])) piv = r;
    if (A[(size_t)piv * n + c] == 0.0) return false;
    if (piv != c) {
      for (int k = 0; k < n; ++k) std::swap(A[(size_t)c * n + k], A[(size_t)piv * n + k]);
      std::swap(b[c], b[piv]);
    }
    for (int r = c + 1; r < n; ++r) {
      const double f = A[(size_t)r * n + c] / A[(size_t)c * n + c];
      if (f == 0.0) continue;
      for (int k = c; k < n; ++k) A[(size_t)r * n + k] -= f * A[(size_t)c * n + k];
      b[r] -= f * b[c];
    }
  }
  x.assign(n, 0.0);
  for (int r = n - 1; r >= 0; --r) {
    double acc = b[r];
    for (int k = r + 1; k < n; ++k) acc -= A[(size_t)r * n + k] * x[k];
    x[r] = acc / A[(size_t)r * n + r];
  }
  return true;
}

// ---------------------------------------------------------------------------------------------- RHF (src/hf.f90)
struct Scf {
  double energy = 0.0;
  bool converged = false;
  int iterations = 0;
  std::vector<double> coeff;  // C(mo, ao) row-major == canon_coeff(mo,ao)
  std::vector<double> eps;
  std::vector<double> fock;   // AO Fock matrix of the last diagonalisation (guess_out.dat)
};

void build_fock(const Sys& s, const std::vector<double>& D, std::vector<double>& F) {
  // F = H + sum_kl D_kl [2 (ij|kl) - (ik|jl)]   (src/hf.f90:319-385)
  const int n = s.nbasis;
  F = s.hcore;
  for (int i = 0; i < n; ++i)
    for (int j = 0; j <= i; ++j) {
      double acc = 0.0;
      const long long ij = pair_index(i, j);
      for (int k = 0; k < n; ++k)
        for (int l = 0; l < n; ++l) {
          const double d = D[(size_t)k * n + l];
          if (d == 0.0) continue;
          acc += d * (2.0 * s.eri[(size_t)pair_index(ij, pair_index(k, l))] -
                      s.eri[(size_t)pair_index(pair_index(i, k), pair_index(j, l))]);
        }
      F[(size_t)i * n + j] += acc;
      if (i != j) F[(size_t)j * n + i] += acc;
    }
}

Scf do_rhf(const Sys& s) {
  const int n = s.nbasis, nocc = s.nel / 2;
  Scf r;
  // X = S^{-1/2} by symmetric orthogonalisation (src/hf.f90:53-80)
  std::vector<double> w, U;
  eigh(s.ovlp, n, w, U);
  std::vector<double> Us = U;
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) Us[(size_t)i * n + j] = U[(size_t)i * n + j] / std::sqrt(w[j]);
  const std::vector<double> X = matmul(Us, U, n, false, true);
  std::vector<double> F = (s.scf_read_guess && !s.guess.empty()) ? s.guess : s.hcore;
  if (s.scf_read_guess && !s.guess.empty()) std::printf(" Reading previous AO Fock matrix as guess...\n");
  std::printf("%s\n Iteration        Energy           deltaE           delta RMS D      Time  \n%s\n",
              std::string(75, '-').c_str(), std::string(75, '-').c_str());
  const int nerr = s.scf_diis_n_errmat;
  const bool use_diis = nerr >= 2;
  std::vector<std::vector<double>> Fs(std::max(nerr, 1)), Es(std::max(nerr, 1));
  int slot = 0, n_active = 0;
  double energy = 0.0;
  std::vector<double> D_old((size_t)n * n, 0.0), D((size_t)n * n), Cp;
  auto t0 = Clock::now();
  for (int it = 1; it <= s.scf_maxiter; ++it) {
    std::vector<double> Fo = matmul(matmul(X, F, n, true, false), X, n);   // F' = X^T F X
    eigh(Fo, n, r.eps, Cp);
    r.fock = F;
    const std::vector<double> C = matmul(X, Cp, n);                        // AO x MO
    r.coeff.assign((size_t)n * n, 0.0);
    for (int mo = 0; mo < n; ++mo)
      for (int ao = 0; ao < n; ++ao) r.coeff[(size_t)mo * n + ao] = C[(size_t)ao * n + mo];
    for (int a = 0; a < n; ++a)
      for (int b = 0; b < n; ++b) {
        double acc = 0.0;
        for (int i = 0; i < nocc; ++i) acc += r.coeff[(size_t)i * n + a] * r.coeff[(size_t)i * n + b];
        D[(size_t)a * n + b] = acc;
      }
    const double e_old = energy;
    energy = 0.0;
    double rms = 0.0;
    for (size_t k = 0; k < D.size(); ++k) {
      energy += D[k] * (s.hcore[k] + F[k]);
      rms += (D[k] - D_old[k]) * (D[k] - D_old[k]);
    }
    rms = std::sqrt(rms);
    r.converged = rms < s.scf_d_tol && std::fabs(energy - e_old) < s.scf_e_tol;
    D_old = D;
    std::printf(" %9d   %15.10f   %15.10f   %15.10f   %8.6f\n", it, energy, energy - e_old, rms, since(t0));
    t0 = Clock::now();
    r.iterations = it;
    if (r.converged) {
      std::printf("%s\n Convergence reached within tolerance.\n", std::string(75, '-').c_str());
      std::printf(" Final SCF Energy (Hartree): %15.8f\n Orbital energies (Hartree):\n", energy);
      for (int i = n; i >= 1; --i) std::printf(" %3d %15.8f\n", i, r.eps[i - 1]);
      break;
    }
    build_fock(s, D, F);
    if (use_diis) {  // update_diis (src/hf.f90:197-242)
      slot = slot < nerr ? slot + 1 : 1;
      n_active = std::min(n_active + 1, nerr);
      Fs[slot - 1] = F;
      const std::vector<double> FDS = matmul(matmul(F, D, n), s.ovlp, n), SDF = matmul(matmul(s.ovlp, D, n), F, n);
      Es[slot - 1].resize((size_t)n * n);
      for (size_t k = 0; k < FDS.size(); ++k) Es[slot - 1][k] = FDS[k] - SDF[k];
      const int na = n_active;
      if (na > 1) {
        std::vector<double> B((size_t)(na + 1) * (na + 1), 0.0), rhs(na + 1, 0.0), c;
        for (int i = 0; i < na; ++i)
          for (int j = 0; j <= i; ++j) {
            double acc = 0.0;
            for (size_t k = 0; k < Es[i].size(); ++k) acc += Es[i][k] * Es[j][k];
            B[(size_t)i * (na + 1) + j] = B[(size_t)j * (na + 1) + i] = acc;
          }
        for (int i = 0; i < na; ++i) B[(size_t)na * (na + 1) + i] = B[(size_t)i * (na + 1) + na] = -1.0;
        rhs[na] = -1.0;
        if (!solve(B, rhs, na + 1, c)) fail("linalg::linsolve", "DIIS linear solve failed");
        std::fill(F.begin(), F.end(), 0.0);
        for (int i = 0; i < na; ++i)
          for (size_t k = 0; k < F.size(); ++k) F[k] += c[i] * Fs[i][k];
      }
    }
  }
  r.energy = energy;
  return r;
}

// ---------------------------------------------------------------------------------------------- files the program writes
void write_scf_guess(const std::vector<double>& F, int n) {  // src/hf.f90:172-191, (I0, 1X, I0, 1X, ES16.9)
  FILE* f = std::fopen("guess_out.dat", "w");
  if (!f) fail("hf::write_out_scf_guess", "cannot open guess_out.dat");
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) std::fprintf(f, "%d %d %16.9E\n", i + 1, j + 1, F[(size_t)i * n + j]);
  std::fclose(f);
}

void write_fcidump(const std::vector<double>& eri_mo, int n) {  // src/mp2.f90:451-487, (I3,I3,I3,I3,ES17.9)
  FILE* f = std::fopen("FCIDUMP", "w");
  if (!f) fail("mp2::write_fcidump", "cannot open FCIDUMP");
  const double thr = (double)1e-7f;  // the reference compares with a default-real literal
  size_t pqrs = 0;
  for (int p = 1; p <= n; ++p)
    for (int q = 1; q <= p; ++q)
      for (int r = 1; r <= p; ++r) {
        const int s_up = (p == r) ? q : r;
        for (int s = 1; s <= s_up; ++s, ++pqrs)
          if (std::fabs(eri_mo[pqrs]) > thr) std::fprintf(f, "%3d%3d%3d%3d%17.9E\n", p, q, r, s, eri_mo[pqrs]);
      }
  std::fclose(f);
}

void stamp(const char* what) {
  std::time_t t = std::time(nullptr);
  std::tm tmv;
  localtime_r(&t, &tmv);
  std::printf(" %s running on %02d/%02d/%04d at %02d:%02d:%02d\n", what, tmv.tm_mday, tmv.tm_mon + 1, tmv.tm_year + 1900,
              tmv.tm_hour, tmv.tm_min, tmv.tm_sec);
}

// '(1X, A, 1X, F16.8, A)' of src/main.F90:43-115 (the shipped N2/F2 logs predate it and print F7.4)
void taken(const std::string& label, double s) { std::printf(" Time taken for %s: %16.8fs\n", label.c_str(), s); }
std::string bar(int n, char c) { return std::string(n, c); }
// Fortran Ew.d: mantissa in [0.1, 1), e.g. E15.6 of 3.5e-7 is "   0.350000E-06" (C's %E would print 3.500000E-07)
std::string fortran_e(double x, int width, int digits) {
  int ex = 0;
  double mant = x;
  if (x != 0.0 && std::isfinite(x)) {
    ex = (int)std::floor(std::log10(std::fabs(x))) + 1;
    mant = x / std::pow(10.0, ex);
    char probe[64];
    std::snprintf(probe, sizeof probe, "%.*f", digits, mant);
    if (std::fabs(std::atof(probe)) >= 1.0) { ++ex; mant = x / std::pow(10.0, ex); }   // rounding carried into the leading digit
  }
  char buf[96];
  std::snprintf(buf, sizeof buf, "%.*fE%+03d", digits, mant, ex);
  std::string out(buf);
  if ((int)out.size() < width) out.insert(0, (size_t)width - out.size(), ' ');
  return out;
}

}  // namespace

int main(int argc, char** argv) {
  int device = 0;
  for (int a = 1; a < argc; ++a) {
    if (!std::strcmp(argv[a], "--device") && a + 1 < argc) device = std::atoi(argv[++a]);
    else if (chdir(argv[a]) != 0) fail("main", std::string("cannot enter directory ") + argv[a]);
  }
  auto t_glob = Clock::now();
  std::printf(" %s\n A Fortran Electronic Structure Programme (AFESP)\n %s\n", bar(64, '=').c_str(), bar(64, '=').c_str());
  stamp("Started");
  auto t0 = Clock::now();

  Sys s;
  read_system_in(s);
  std::printf(" %s\n Integral read-in\n %s\n", bar(16, '-').c_str(), bar(16, '-').c_str());
  std::printf(" Getting number of basis functions...\n Allocating integral store...\n Reading overlap matrix...\n"
              " Reading kinetic integrals...\n Reading nuclear-electron integrals...\n Constructing core Hamiltonian...\n"
              " Reading two-body integrals...\n");
  read_integrals_in(s);
  std::printf(" Done reading integrals!\n");
  read_geometry_in(s);
  const int n = s.nbasis, nocc = s.nel / 2;
  if (s.frozen_core < 0 || s.frozen_core >= nocc)   // at least one doubly occupied orbital stays active
    fail("system::read_system_in", "frozen_core = " + std::to_string(s.frozen_core) + " is outside 0.." +
                                       std::to_string(nocc - 1) + " (nocc - 1)!");
  // print_sys_info (src/integrals.f90:223-249)
  std::printf(" %s\n System information\n %s\n", bar(20, '-').c_str(), bar(20, '-').c_str());
  std::printf(" Number of electrons: %d\n Number of basis functions: %d\n Number of occupied orbitals: %d\n"
              " Number of virtual orbitals: %d\n",
              s.nel, n, s.restricted ? nocc : s.nel, s.restricted ? n - nocc : 2 * (n - nocc));   // src/geometry.f90:40-46
  if (s.frozen_core > 0) std::printf(" Number of frozen core orbitals: %d\n", s.frozen_core);
  std::printf(" E_nuc: %15.8E\n scf_e_tol: %8.2E\n scf_d_tol: %8.2E\n ccsd_e_tol: %8.2E\n"
              " ccsd_t_tol: %8.2E\n Number of SCF DIIS error matrices: %d\n Number of CCSD DIIS error matrices: %d\n"
              " Maximum number of SCF iterations: %d\n Maximum number of CCSD iterations: %d\n"
              " Printing out the input file...\n%s\n",
              s.e_nuc, s.scf_e_tol, s.scf_d_tol, s.ccsd_e_tol, s.ccsd_t_tol,
              s.scf_diis_n_errmat, s.ccsd_diis_n_errmat, s.scf_maxiter, s.ccsd_maxiter, bar(30, '-').c_str());
  {
    std::istringstream in(s.els_in_text);
    std::string ln;
    while (std::getline(in, ln)) {
      size_t e = ln.find_last_not_of(" \t\r");
      std::printf("%s\n", e == std::string::npos ? "" : ln.substr(0, e + 1).c_str());
    }
  }
  std::printf("%s\n", bar(30, '-').c_str());
  taken("system initialisation", since(t0));
  // calc_type "UHF": the reference has no UHF (do_uhf is a stub, src/hf.f90:193); its main program runs do_rhf for every
  // unrestricted calc_type (src/main.F90:49-56) and, for "UHF", goes straight to the final table.  Same here.

  // ---- RHF
  t0 = Clock::now();
  std::printf(" %s\n Restricted Hartree-Fock\n %s\n", bar(23, '-').c_str(), bar(23, '-').c_str());
  if (s.scf_read_guess) {
    std::ifstream f("guess_in.dat");
    if (!f) fail("hf::read_in_scf_guess", "cannot open guess_in.dat");
    s.guess.assign((size_t)n * n, 0.0);
    long long i, j;
    double v;
    while (f >> i >> j >> v)
      if (i >= 1 && j >= 1 && i <= n && j <= n) s.guess[(size_t)(i - 1) * n + (j - 1)] = v;
  }
  Scf scf = do_rhf(s);
  if (!scf.converged) std::printf(" Convergence not reached, please increase maxiter.\n");
  else if (s.scf_write_guess) {
    std::printf(" Writing AO Fock matrix for future use...\n");
    write_scf_guess(scf.fock, n);
  }
  taken("restricted Hartree-Fock", since(t0));
  const double e_hf = scf.energy;
  double e_mp2 = 0.0, e_ccsd = 0.0, t1_diag = 0.0, highest = 0.0;
  std::map<std::string, double> en;
  bool cc_conv = false;

  if (s.level >= 1) {
    if (afesp_gpu_open(device, &g_h) != 0) fail("afesp_gpu::afesp_gpu_open", afesp_gpu_last_error(nullptr));
    // Library switches (parity switches Q1-Q3, thresholds; include/afesp_gpu.h) from the environment, the way a Fortran
    // host would pass them on: AFESP_GPU_OPTIONS="key=value,key=value"
    if (const char* env = std::getenv("AFESP_GPU_OPTIONS")) {
      std::string all(env);
      size_t pos = 0;
      while (pos < all.size()) {
        size_t end = all.find(',', pos);
        if (end == std::string::npos) end = all.size();
        const std::string kv = all.substr(pos, end - pos);
        const size_t eq = kv.find('=');
        if (eq != std::string::npos)
          check("set_option", afesp_gpu_set_option(g_h, kv.substr(0, eq).c_str(), std::atof(kv.substr(eq + 1).c_str())));
        pos = end + 1;
      }
    }
    // MP2, CCSD and the triples correlate orbitals frozen_core.. only
    if (s.frozen_core > 0) check("set_option", afesp_gpu_set_option(g_h, "frozen_core", s.frozen_core));
    // coeff(mo,ao) column-major as the Fortran host holds canon_coeff: element (mo,ao) at mo + n*ao
    std::vector<double> coeff_f((size_t)n * n);
    for (int mo = 0; mo < n; ++mo)
      for (int ao = 0; ao < n; ++ao) coeff_f[(size_t)mo + (size_t)n * ao] = scf.coeff[(size_t)mo * n + ao];
    // ---- MP2 (src/mp2.f90:261-449)
    t0 = Clock::now();
    std::printf(" ----------\n MP2\n ----------\n Performing AO to MO ERI transformation...\n");
    std::vector<double> eri_mo;
    if (s.write_fcidump) eri_mo.resize(s.eri.size());
    check("ao2mo", afesp_gpu_ao2mo(g_h, n, s.eri.data(), coeff_f.data(), s.write_fcidump ? eri_mo.data() : nullptr));
    std::printf(" Calculating MP2 energy...\n");
    check("mp2_energy", afesp_gpu_mp2_energy(g_h, nocc, scf.eps.data(), &e_mp2));
    std::printf(" MP2 correlation energy (Hartree): %15.8f\n", e_mp2);
    highest = e_mp2;
    if (s.write_fcidump) {
      std::printf(" Writing FCIDUMP file...\n");
      write_fcidump(eri_mo, n);
      std::printf(" Done writing FCIDUMP file!\n");
    }
    taken("restricted MP2", since(t0));
  }
  if (s.level >= 2) {
    // ---- CCSD (src/ccsd.f90:279-402 / 71-277): the GPU does one iteration per call, the host keeps the loop
    t0 = Clock::now();
    std::printf(" ----------\n CCSD\n ----------\n");
    auto ti = Clock::now();
    double e = 0.0, rms = 0.0;
    const int rc_init = afesp_gpu_ccsd_init(g_h, nocc, s.restricted ? 1 : 0, scf.eps.data(), s.ccsd_diis_n_errmat, &e, &rms);
    if (!s.restricted) {
      // src/ccsd.f90:106-202.  The (2n)^4 tensor is never formed: the nine slices are gathered straight from the packed MO
      // integrals (first timer) and the reference's symmetry assertion runs on the device over the same index set (second
      // timer); nothing is left for the third banner.  Status 5 = the assertion fired (:161-164).
      double info[4] = {0, 0, 0, 0};
      if (rc_init == 0 || rc_init == 5) check("ccsd_init_info", afesp_gpu_ccsd_init_info(g_h, info));
      if (rc_init == 5) {
        std::printf(" Forming antisymmetrised spinorbital ERIs...\n Time taken: %8.6f s\n\n", info[1]);
        std::printf(" Checking that the permuational symmetry of the antisymmetrised integrals hold...\n");
        std::printf(" Permutational symmetry error: %s\n", fortran_e(info[0], 15, 6).c_str());   // E15.6, src/ccsd.f90:165
        fail("ccsd::do_ccsd", "Permutational symmetry of antisymmetrised integrals does not hold");
      }
      check("ccsd_init", rc_init);
      std::printf(" Forming antisymmetrised spinorbital ERIs...\n Time taken: %8.6f s\n\n", info[1]);
      std::printf(" Checking that the permuational symmetry of the antisymmetrised integrals hold...\n Time taken: %8.6f s\n\n", info[2]);
      std::printf(" Forming slices of antisymmetrised spinorbital ERIs\n Time taken: %8.6f s\n\n", 0.0);
    }
    check("ccsd_init", rc_init);
    std::printf(" Initialise CC intermediate tensors and DIIS auxilliary arrays...\n Forming energy denominator matrices...\n"
                " Allocating amplitude tensors...\n");
    std::printf(" Forming ERI slices...\n Forming initial amplitude guesses...\n Allocating stored intermediate tensors...\n");  // :477-526, both formulations
    std::printf(" Time taken: %8.6f s\n\n Initialisation done, now entering iterative CC solver...\n", since(ti));
    std::printf("%s\n Iteration        Energy           deltaE          delta RMS T2      Time  \n%s\n", bar(75, '-').c_str(),
                bar(75, '-').c_str());
    std::printf(" %9s   %15.12f   %15.12f   %15.12f\n", "MP1", e, e, rms);
    double e_old = e;
    for (int it = 1; it <= s.ccsd_maxiter; ++it) {
      auto tit = Clock::now();
      check("ccsd_iterate", afesp_gpu_ccsd_iterate(g_h, &e, &rms));
      std::printf(" %9d   %15.12f   %15.12f   %15.12f   %8.6f\n", it, e, e - e_old, rms, since(tit));
      if (std::sqrt(rms) < s.ccsd_t_tol && std::fabs(e - e_old) < s.ccsd_e_tol) { cc_conv = true; break; }  // :1805
      e_old = e;
      check("ccsd_diis", afesp_gpu_ccsd_diis(g_h));
    }
    e_ccsd = e;
    if (cc_conv) {
      std::printf("%s\n Convergence reached within tolerance.\n Final CCSD Energy (Hartree): %15.12f\n", bar(75, '-').c_str(),
                  e_ccsd);
      highest = e_ccsd;
    }
    check("ccsd_finalize", afesp_gpu_ccsd_finalize(g_h, s.comp_renorm ? 1 : 0, &t1_diag, nullptr, nullptr));
    if (s.restricted && cc_conv) {
      std::printf(" T1 diagnostic: %8.5f\n", t1_diag);
      if (t1_diag > 0.02) std::printf(" Significant multireference character detected, CCSD result might be unreliable!\n");
    }
    taken(s.restricted ? "restricted CCSD" : "unrestricted CCSD", since(t0));
  }
  if (s.level >= 3 && cc_conv) {
    t0 = Clock::now();
    std::printf(" ----------\n CCSD(T)\n ----------\n");
    std::string name = "CCSD(T)";
    if (s.restricted) {
      double sums[6], dconst = 0.0;
      check("ccsd_t_spatial", afesp_gpu_ccsd_t_spatial(g_h, s.paren, s.renorm, s.comp_renorm, sums, &dconst));
      // energy assembly of do_ccsd_t_spatial (src/ccsd.f90:2239-2276)
      double e_T = sums[0], e_TT = sums[1], D_T = sums[2], D_TT = sums[3], e_CR = sums[4], e_CRT = sums[5];
      const bool ren = s.renorm || s.comp_renorm;
      if (ren) { D_T += dconst; if (s.paren) D_TT += dconst; }
      en["e_ccsd_t"] = e_ccsd + e_T; highest = en["e_ccsd_t"];
      if (s.paren) { en["e_ccsd_tt"] = e_ccsd + e_TT; highest = en["e_ccsd_tt"]; }
      if (ren) {
        en["e_rccsd_t"] = e_ccsd + e_T / D_T; en["D_T"] = D_T; highest = en["e_rccsd_t"];
        if (s.paren) { en["e_rccsd_tt"] = e_ccsd + e_TT / D_TT; highest = en["e_rccsd_tt"]; }
        if (s.comp_renorm) {
          en["e_crccsd_t"] = e_ccsd + e_CR / D_T; en["D_TT"] = D_TT; highest = en["e_crccsd_t"];
          if (s.paren) { en["e_crccsd_tt"] = e_ccsd + e_CRT / D_TT; highest = en["e_crccsd_tt"]; }
        }
      }
      name = s.paren ? "CCSD(T)" : "CCSD[T]";
      if (s.renorm) name = "renormalised " + name;
      if (s.comp_renorm) name = "completely renormalised " + name;
      std::printf(" Restricted %s correlation energy (Hartree): %15.9f\n", name.c_str(), highest);
    } else {
      double e_T = 0.0;
      check("ccsd_t_spinorb", afesp_gpu_ccsd_t_spinorb(g_h, &e_T));
      en["e_ccsd_t"] = e_ccsd + e_T; highest = en["e_ccsd_t"];
      std::printf(" Unrestricted CCSD(T) correlation energy (Hartree): %15.9f\n", highest);
    }
    taken((s.restricted ? "restricted " : "unrestricted ") + name, since(t0));
  }
  if (g_h) { afesp_gpu_close(g_h); g_h = nullptr; }

  // ---- final energy breakdown (src/main.F90:123-175)
  const double base = e_hf + s.e_nuc;
  auto line = [](const char* label, double v) { std::printf(" %-31s %15.10f\n", label, v); };
  auto two = [&](const std::string& label, double corr) {
    line((label + " correlation energy:").c_str(), corr);
    line((label + " energy:").c_str(), corr + base);
  };
  std::printf(" %s\n Final energy breakdown\n", bar(64, '=').c_str());
  line("RHF energy:", base);
  if (s.level >= 1) two("MP2", e_mp2);
  if (s.level >= 2) two("CCSD", e_ccsd);
  if (s.level >= 3 && !en.empty()) {
    if (s.restricted) {
      two("CCSD[T]", en["e_ccsd_t"]);
      if (s.paren) two("CCSD(T)", en["e_ccsd_tt"]);
      if (s.renorm || s.comp_renorm) {
        two("R-CCSD[T]", en["e_rccsd_t"]);
        if (s.paren) two("R-CCSD(T)", en["e_rccsd_tt"]);
        if (s.comp_renorm) {
          two("CR-CCSD[T]", en["e_crccsd_t"]);
          if (s.paren) two("CR-CCSD(T)", en["e_crccsd_tt"]);
        }
      }
    } else {
      two("CCSD(T)", en["e_ccsd_t"]);
    }
  }
  if (s.level >= 2 && s.restricted) {
    std::printf(" %s\n", bar(47, '-').c_str());
    line("T1 diagnostic:", t1_diag);
  }
  if ((s.renorm || s.comp_renorm) && !en.empty()) {
    line("D[T]:", en["D_T"]);
    if (s.paren) line("D(T):", en.count("D_TT") ? en["D_TT"] : 0.0);
  }
  std::printf(" %s\n", bar(47, '-').c_str());
  line("Total electronic energy:", e_hf + highest);
  line("Nuclear repulsion:", s.e_nuc);
  line("Total energy:", e_hf + highest + s.e_nuc);
  std::printf(" %s\n", bar(64, '=').c_str());
  stamp("Finished");
  std::printf(" Total execution time: %16.8f\n", since(t_glob));   // src/main.F90:185
  return 0;
}
