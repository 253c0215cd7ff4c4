// Packed-ERI kernels (integrals.cu).
#pragma once
#include "tensor.cuh"

namespace afesp {

long long npair_of(int n);    // n(n+1)/2
long long npacked_of(int n);  // npair(npair+1)/2

// eri_mo[packed] = sum C C C C eri_ao[packed];  C is C(mo,ao) column-major n x n (src/hf.f90:102).  All device.
void ao2mo_packed(Engine& e, int n, const double* eri_ao, const double* C, double* eri_mo,
                  long long block_bytes = 3LL << 30);

// Synthetic packed AO integrals eri = sum_P B(ij,P) B(kl,P) from device-resident factors B (npair x naux).
void synth_eri_from_factors(Engine& e, int n, int naux, const double* B, double* eri, long long block_bytes = 2LL << 30);

// MP2 correlation energy (src/mp2.f90:418-438) from packed MO integrals; result in out_dev[0].  The occupied sums run
// over the active orbitals nfrozen..nocc-1 (frozen core), the virtual ones over nocc..n-1.
void mp2_energy(Engine& e, int n, int nocc, int nfrozen, const double* eri_mo, const double* eps, double* out_dev);

// out(p,q,r,s) = <PQ|RS> = (PR|QS) with P = lo[0]+p ...; spatial orbitals (src/ccsd.f90:496-512)
void slice_phys(Engine& e, double* out, const double* eri_mo, const int lo[4], const int cnt[4]);
// out(P,Q,R,S) = <PQ||RS> over spin-orbital index ranges (src/ccsd.f90:111-143, 182-194)
void slice_spinorb(Engine& e, double* out, const double* eri_mo, const int lo[4], const int cnt[4]);

// err of the permutational-symmetry self-check of <pq||rs> (src/ccsd.f90:150-167), evaluated from the packed MO integrals
// over the spin-orbitals lo..2n-1 (lo = 2 x frozen core orbitals); result in out_dev[0].
void spinorb_symmetry_error(Engine& e, int n, int lo, const double* eri_mo, double* out_dev);

// Particle-particle ladder in (+/-)-symmetrised virtual-pair form (half the flop and memory of the dense v^4 slice):
//   sum_ef c(ij,ef) <ef|ab> = 1/2 [ S Vp + A Vm ](ij,ab),  S/A = symmetric/antisymmetric parts of c in (e,f)
// sign +1: Vp (P+ x P+), -1: Vm (P- x P-); columns [col0, col0 + ncols) only (ncols < 0: through the last column) --
// with several GPUs each rank keeps just the column slab of Vp / Vm its share of the ladder GEMM reads.
// The v virtual orbitals start at voff (= nocc) in the packed MO array.
void build_vpm(Engine& e, double* V, const double* eri_mo, int voff, int v, int sign, long long col0 = 0,
               long long ncols = -1);
void pack_c(Engine& e, double* S, double* A, const double* c, int oo, int v);
void unpack_ladder(Engine& e, double* X, const double* Lp, const double* Lm, int oo, int v, double alpha);

}  // namespace afesp
