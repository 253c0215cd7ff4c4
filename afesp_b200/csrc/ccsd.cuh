// Device-resident coupled-cluster state behind the C-ABI handle (include/afesp_gpu.h).
#pragma once
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "integrals.cuh"
#include "kernels.cuh"
#include "tensor.cuh"

namespace afesp {

// CC-DIIS ring (src/ccsd.f90:46-67, 577-676): stores the un-extrapolated amplitudes T_i and e_i = T_i - T'_{i-1}.
struct CCDiis {
  int nerr = 8;
  bool use = false;   // set by init(); a default-constructed ring (after finalize) must not be extrapolated
  int slot = 0, n_active = 0;
  std::vector<Tensor> t1, t2, e1, e2;
  Tensor t1_s, t2_s;
  std::vector<double> B;  // (nerr x nerr) cache of e_i . e_j, row-major, filled for active slots
  void init(int nerr_, int o, int v);
};

struct Options {
  bool q1_transposed_foo = true;   // spin-orbital build_F dgemm lands transposed (src/ccsd.f90:793-795)
  bool q3a_truncated_e = true;     // `do e = 1, nocc` over a virtual index (src/ccsd.f90:2535)
  bool q3b_stale_intermediates = true;  // CR intermediates read I_vo/asym_t2 of the last iteration's input (:2377)
  bool triples_ijk_symmetry = true;     // (T): loop unique i<=j<=k with multiplicities instead of all o^3
  long long triples_batch_bytes = 6LL << 30;
  bool finalize_keep_ccsd = false;      // keep DIIS history and intermediates after finalize (benchmark loops)
  double spinorb_symmetry_tol = 1e-12;  // depsilon (src/const.F90:19): abort threshold of the check at src/ccsd.f90:161
};

struct CCState {
  Engine eng;
  Options opt;
  int n = 0, nocc_spatial = 0;
  int nfrozen = 0;   // frozen doubly occupied orbitals 0..nfrozen-1: the CC equations see orbitals nfrozen..n-1 only
  bool restricted = true;
  int o = 0, v = 0;  // occupied / virtual counts in the active formulation (spin-orbital counts when !restricted)

  // inputs resident on the device
  DBuf eri_mo;       // packed MO ERIs
  DBuf eps;          // spatial orbital energies (n)
  Tensor eo, ev;     // energies of the active formulation, split occupied/virtual
  std::vector<double> eps_host;

  // amplitudes
  Tensor t1, t2, t1n, t2n, t2_old;
  DBuf red_out;      // small device array for reduction results
  double energy = 0.0, energy_old = 0.0, rms = 0.0;
  int iterations = 0;
  CCDiis diis;

  // spin-free integrals / intermediates (Piecuch et al.; src/ccsd.f90:507-512, 1040-1312)
  std::map<std::string, Tensor> T;  // named tensors: v_oovv, v_ovov, ..., I_vv, ...
  Tensor& get(const std::string& name) {
    auto it = T.find(name);
    AFESP_REQUIRE(it != T.end(), "unknown tensor " + name);
    return it->second;
  }
  Tensor& make(const std::string& name, std::vector<int> dims) {
    Tensor& t = T[name];
    if (t.dims != dims) t.init(dims);
    return t;
  }
  bool has(const std::string& name) const { return T.count(name) != 0; }
  void drop(const std::string& name) { T.erase(name); }

  // spin-orbital integral preparation (src/ccsd.f90:106-202): error of the permutational-symmetry self-check and the
  // device milliseconds of the slice gather and of the check (afesp_gpu_ccsd_init_info)
  double sym_err = 0.0, ms_slices = 0.0, ms_symcheck = 0.0;

  bool finalized = false;
  bool have_cr = false;
  bool vpm_sharded = false;  // V_plus / V_minus hold only this rank's column slab (ccsd_spatial_init)
};

// ---- spin-free (ccsd_spatial.cu)
void ccsd_spatial_init(CCState& s, int diis_n);
void ccsd_spatial_iterate(CCState& s);
void ccsd_spatial_cr_intermediates(CCState& s);  // build I_vovv_pp / I_ooov_pp (src/ccsd.f90:2338-2551)
// ---- spin-orbital (ccsd_spinorb.cu)
void ccsd_spinorb_init(CCState& s, int diis_n);
void ccsd_spinorb_iterate(CCState& s);
// ---- common (ccsd_common.cu)
void cc_update_energy(CCState& s);     // energy, rms <- current t1,t2 ; t2_old <- t2   (src/ccsd.f90:1734-1810)
void cc_diis_stash(CCState& s);        // t_s <- t   (src/ccsd.f90:342-343)
void cc_diis_update(CCState& s);       // src/ccsd.f90:617-676
double cc_t1_norm2(CCState& s);        // sum t1^2

// ---- triples (triples.cu): accumulators of do_ccsd_t_spatial / do_ccsd_t_spinorb for the triples owned by
//      (rank, nranks); sums[6] = e_T, e_TT, D_T, D_TT, e_CR, e_CRT (partial, without the constant of :2243)
void triples_spatial(CCState& s, bool paren, bool renorm, bool comp_renorm, int rank, int nranks, double sums[6]);
double triples_denominator_constant(CCState& s);  // 1 + 2 sum t1^2 + sum asym_t2 * c   (src/ccsd.f90:2243)
void triples_spinorb(CCState& s, int rank, int nranks, double* e_T);
// number of (i,j,k) work units each rank owns under the round-robin deal (host only, no device needed)
void triples_partition_counts(int o, bool symmetric, bool strict, int nranks, long long* counts);

}  // namespace afesp
