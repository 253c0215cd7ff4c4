// Spin-free (closed-shell) CCSD on the device: Piecuch et al. CPC 149 (2002) 71, as coded by the reference in
// src/ccsd.f90:404-575 (init_cc), 1040-1312 (update_restricted_intermediates), 1538-1732
// (update_amplitudes_restricted) and 2338-2551 (build_cr_ccsd_t_intermediates).
//
// Every contraction -- including the ones the reference leaves as naive OpenMP loop nests (SURVEY.md §2.3, e.g. the
// three o^3 v^3 ring terms at :1680-1695) -- is a labelled einsum lowered to FP64 DMMA GEMMs (contract.cu).
// Tensor names and index orders follow the reference (SURVEY.md App. A); all arrays are column-major.
//
// Deviations that do not change results beyond rounding:
//  * the in-place antisymmetrise/deantisymmetrise round trips on the integral slices (:1089-1126) are replaced by
//    a constant tensor built once (A_oovv = 2 v_oovv - v_oovv^(ab)) and by two-step contractions for the v_vvov term;
//  * the particle-particle ladder (:1669) runs in (+/-)-symmetrised virtual-pair form, 1/2 [S Vp + A Vm]: two GEMMs
//    o^2 x P x P with P ~ v^2/2 -- half the flop and half the memory of the dense v^4 slice, which is never formed
//    (it would be 134 GB at nbf=400);
//  * I_vovv_p (o v^3, :1261-1299) is never materialised: its only consumer, t1 * I_vovv_p (:1700), is expanded into
//    one o^2v^3 GEMM against v_vvov and two o^3v^2 two-step products;
//  * energy denominators are evaluated from the orbital energies inside the divide kernel.
#include "ccsd.cuh"

namespace afesp {

namespace {
inline TView V(Tensor& t) { return t.view(); }
}  // namespace

void ccsd_spatial_init(CCState& s, int diis_n) {
  // active occupied orbitals start at nf (frozen core), virtual ones at nocc
  const int n = s.n, nocc = s.nocc_spatial, nf = s.nfrozen, o = nocc - nf, v = n - nocc;
  s.restricted = true;
  s.o = o; s.v = v;
  AFESP_REQUIRE(o > 0 && v > 0, "ccsd init: need at least one occupied and one virtual orbital");
  Engine& e = s.eng;
  Trace tr(e.stream);
  s.eo.init({o}); s.ev.init({v});
  AFESP_CUDA_CHECK(cudaMemcpyAsync(s.eo.p(), s.eps.p + nf, o * 8, cudaMemcpyDeviceToDevice, e.stream));
  AFESP_CUDA_CHECK(cudaMemcpyAsync(s.ev.p(), s.eps.p + nocc, v * 8, cudaMemcpyDeviceToDevice, e.stream));
  // integral slices, physicist order (src/ccsd.f90:507-512)
  struct Sl { const char* name; char k[5]; };
  const Sl sl[] = {{"v_oovv", "oovv"}, {"v_ovov", "ovov"}, {"v_vvov", "vvov"},
                   {"v_oovo", "oovo"}, {"v_oooo", "oooo"}};
  for (const Sl& x : sl) {
    int lo[4], cnt[4];
    std::vector<int> dims;
    for (int d = 0; d < 4; ++d) {
      lo[d] = x.k[d] == 'o' ? nf : nocc;
      cnt[d] = x.k[d] == 'o' ? o : v;
      dims.push_back(cnt[d]);
    }
    Tensor& t = s.make(x.name, dims);
    slice_phys(e, t.p(), s.eri_mo.p, lo, cnt);
  }
  tr.lap(0);
  Tensor& v_oovv = s.get("v_oovv");
  // A_oovv(i,j,a,b) = 2 v_oovv(i,j,a,b) - v_oovv(i,j,b,a)      (antisymmetrise '1243', :1089)
  Tensor& A = s.make("A_oovv", {o, o, v, v});
  transpose(e, "ijab->ijba", -1.0, V(v_oovv), 0.0, V(A));
  axpby(e.stream, A.size(), 2.0, v_oovv.p(), 1.0, A.p());
  // (+/-)-symmetrised <ef|ab> over virtual pairs for the ladder (replaces the dense v_vvvv slice of :512).
  // With several GPUs each rank builds and keeps only its column slab (ab in its range): W_abef-type memory and flop
  // are divided by the number of ranks; the o^2 x P result slabs are exchanged over NVLink after the GEMM.
  {
    const long long Pp = (long long)v * (v + 1) / 2, Pm = (long long)v * (v - 1) / 2;
    AFESP_REQUIRE(Pp < (1LL << 31), "too many virtual pairs");
    const Dist& d = e.dist;
    s.vpm_sharded = d.active() && Pm >= 64LL * d.nranks;
    long long p0 = 0, p1 = Pp, m0 = 0, m1 = Pm;
    if (s.vpm_sharded) { d.col_range(Pp, d.rank, &p0, &p1); d.col_range(Pm, d.rank, &m0, &m1); }
    Tensor& Vp = s.make("V_plus", {(int)Pp, (int)std::max<long long>(p1 - p0, 1)});
    build_vpm(e, Vp.p(), s.eri_mo.p, nocc, v, +1, p0, p1 - p0);
    if (Pm > 0) {
      Tensor& Vm = s.make("V_minus", {(int)Pm, (int)std::max<long long>(m1 - m0, 1)});
      build_vpm(e, Vm.p(), s.eri_mo.p, nocc, v, -1, m0, m1 - m0);
    }
  }

  tr.lap(1);
  s.t1.init({o, v}); s.t1n.init({o, v});
  s.t2.init({o, o, v, v}); s.t2n.init({o, o, v, v}); s.t2_old.init({o, o, v, v});
  fill(e.stream, s.t1.size(), 0.0, s.t1.p());
  fill(e.stream, s.t2_old.size(), 0.0, s.t2_old.p());
  divide_d2(e.stream, s.t2.p(), v_oovv.p(), s.eo.p(), s.ev.p(), o, v);  // MP1 guess (:520-521)
  // stored intermediates (:527-554)
  s.make("I_vo", {v, o}); s.make("I_vv", {v, v}); s.make("I_oo_p", {o, o}); s.make("I_oo", {o, o});
  s.make("c_oovv", {o, o, v, v}); s.make("asym_t2", {o, o, v, v});
  s.make("x_voov", {v, o, o, v}); s.make("I_oooo", {o, o, o, o}); s.make("I_ovov", {o, v, o, v});
  s.make("I_voov", {v, o, o, v}); s.make("I_ooov_p", {o, o, o, v});
  tr.lap(2);
  s.diis.init(diis_n, o, v);
  s.energy = s.energy_old = 0.0;
  s.iterations = 0;
  s.finalized = false; s.have_cr = false;
  tr.lap(3);
  {
    const char* names[] = {"init slices", "init V+/-", "init amps", "init diis"};
    tr.report(names, 4);
  }
}

void ccsd_spatial_iterate(CCState& s) {
  Engine& e = s.eng;
  cudaStream_t st = e.stream;
  const int o = s.o, v = s.v;
  Tensor &t1 = s.t1, &t2 = s.t2;
  Tensor &v_oovv = s.get("v_oovv"), &v_ovov = s.get("v_ovov"), &v_vvov = s.get("v_vvov"), &v_oovo = s.get("v_oovo"),
         &v_oooo = s.get("v_oooo"), &A = s.get("A_oovv");
  Tensor &I_vo = s.get("I_vo"), &I_vv = s.get("I_vv"), &I_oo_p = s.get("I_oo_p"), &I_oo = s.get("I_oo"),
         &c = s.get("c_oovv"), &asym = s.get("asym_t2"), &x_voov = s.get("x_voov"), &I_oooo = s.get("I_oooo"),
         &I_ovov = s.get("I_ovov"), &I_voov = s.get("I_voov"), &I_ooov_p = s.get("I_ooov_p");
  auto E = [&](const char* spec, double alpha, Tensor& a, Tensor& b, double beta, Tensor& cc) {
    einsum(e, spec, alpha, a.view(), b.view(), beta, cc.view());
  };
  auto copy = [&](Tensor& dst, Tensor& src) {
    AFESP_CUDA_CHECK(cudaMemcpyAsync(dst.p(), src.p(), src.size() * 8, cudaMemcpyDeviceToDevice, st));
  };

  // ---------------- update_restricted_intermediates (src/ccsd.f90:1040-1312) ----------------
  // asym_t2 = 2 t2 - t2(j,i,a,b)  (:1063-1064);  c = t2 + t1 (x) t1  (:1071-1079)
  transpose(e, "ijab->jiab", -1.0, V(t2), 0.0, V(asym));
  axpby(st, asym.size(), 2.0, t2.p(), 1.0, asym.p());
  t2_plus_t1t1(st, c.p(), t2.p(), t1.p(), o, v, 1.0, 0.0);
  // I_vo(a,i) = A(i,m,a,e) t1(m,e)                                                        (:1089-1092)
  E("imae,me->ai", 1.0, A, t1, 0.0, I_vo);
  // I_vv(b,a) = [2v(e,b,m,a) - v(b,e,m,a)] t1(m,e) - A(m,n,e,b) c(m,n,e,a)                (:1101-1111)
  {
    // 2 v(e,b,m,a) t1(m,e): Z(n,b,m,a) = t1(n,e) v_vvov(e,b,m,a) (one GEMM on v_vvov in place), then the n == m diagonal
    Scratch z(e.pool, (size_t)t2.size());
    TView Z(z.p, {o, v, o, v});
    einsum(e, "ne,ebma->nbma", 1.0, V(t1), V(v_vvov), 0.0, Z);
    diag_sum_nbma(st, I_vv.p(), z.p, o, v, 2.0);
    // - v(b,e,m,a) t1(m,e): for each a, I_vv(:,a) -= v_vvov(:,(e,m),a) t1^T(e,m)   (batched GEMV on v_vvov in place)
    Tensor t1T({v, o});
    transpose(e, "me->em", 1.0, V(t1), 0.0, V(t1T));
    GemmBatch bt;
    bt.count = v; bt.strideA = (long long)v * v * o; bt.strideB = 0; bt.strideC = v;
    dgemm(st, 'N', 'N', v, 1, v * o, -1.0, v_vvov.p(), v, t1T.p(), (long long)v * o, 1.0, I_vv.p(), v, &bt);
    AFESP_CUDA_CHECK(cudaStreamSynchronize(st));  // t1T is freed at scope exit
  }
  E("mneb,mnea->ba", -1.0, A, c, 1.0, I_vv);
  // I_oo_p(j,i) = [2v_oovo(m,i,e,j) - v_oovo(i,m,e,j)] t1(m,e) + asym_t2(j,m,f,e) v_oovv(m,i,e,f)   (:1121-1131)
  E("miej,me->ji", 2.0, v_oovo, t1, 0.0, I_oo_p);
  E("imej,me->ji", -1.0, v_oovo, t1, 1.0, I_oo_p);
  E("jmfe,mief->ji", 1.0, asym, v_oovv, 1.0, I_oo_p);
  // I_oo(j,i) = I_oo_p + t1(j,e) I_vo(e,i)                                                (:1136-1137)
  copy(I_oo, I_oo_p);
  E("je,ei->ji", 1.0, t1, I_vo, 1.0, I_oo);
  // I_oooo(k,l,i,j) = v_oooo + c(k,l,e,f) v_oovv(i,j,e,f) + P[t1(k,e) v_oovo(i,l,e,j)]     (:1143-1155)
  copy(I_oooo, v_oooo);
  E("klef,ijef->klij", 1.0, c, v_oovv, 1.0, I_oooo);
  {
    Scratch scr(e.pool, (size_t)I_oooo.size());
    TView S(scr.p, {o, o, o, o});
    einsum(e, "ke,ilej->klij", 1.0, V(t1), V(v_oovo), 0.0, S);
    axpby(st, I_oooo.size(), 1.0, scr.p, 1.0, I_oooo.p());
    transpose(e, "klij->lkji", 1.0, S, 1.0, V(I_oooo));
  }
  // I_ovov(j,b,i,a) = v_ovov - 1/2 v_oovv(m,i,b,e) c(m,j,a,e) - v_oovo(m,i,b,j) t1(m,a) + t1(j,e) v_vvov(e,b,i,a)   (:1165-1191)
  copy(I_ovov, v_ovov);
  E("mibe,mjae->jbia", -0.5, v_oovv, c, 1.0, I_ovov);
  E("mibj,ma->jbia", -1.0, v_oovo, t1, 1.0, I_ovov);
  E("je,ebia->jbia", 1.0, t1, v_vvov, 1.0, I_ovov);
  // x_voov(b,j,i,a) = v_vvov(b,e,i,a) t1(j,e), read as v_vvov(b,a,i,e) (real-orbital symmetry)   (:1279-1290)
  E("baie,je->bjia", 1.0, v_vvov, t1, 0.0, x_voov);
  // I_voov(b,j,i,a)                                                                        (:1205-1252)
  transpose(e, "jiab->bjia", 1.0, V(v_oovv), 0.0, V(I_voov));
  E("imbe,mjea->bjia", 0.5, A, t2, 1.0, I_voov);
  E("imbe,mjae->bjia", -0.5, v_oovv, c, 1.0, I_voov);
  E("imbj,ma->bjia", -1.0, v_oovo, t1, 1.0, I_voov);
  axpby(st, I_voov.size(), 1.0, x_voov.p(), 1.0, I_voov.p());
  // I_ooov_p(j,k,i,a) = v_oovo(k,j,a,i) + t2(j,k,e,f) v_vvov(e,f,i,a) + t1(j,e) x_voov(e,k,i,a)   (:1306-1308)
  transpose(e, "kjai->jkia", 1.0, V(v_oovo), 0.0, V(I_ooov_p));
  E("jkef,efia->jkia", 1.0, t2, v_vvov, 1.0, I_ooov_p);
  E("je,ekia->jkia", 1.0, t1, x_voov, 1.0, I_ooov_p);

  // ---------------- update_amplitudes_restricted (src/ccsd.f90:1538-1732) ----------------
  Tensor &r1 = s.t1n, &X = s.t2n;
  E("ie,ea->ia", 1.0, t1, I_vv, 0.0, r1);                 // :1571
  E("im,ma->ia", -1.0, I_oo_p, t1, 1.0, r1);              // :1572
  E("em,miea->ia", 1.0, I_vo, asym, 1.0, r1);             // :1580-1589
  E("me,miea->ia", 2.0, t1, v_oovv, 1.0, r1);
  E("me,maie->ia", -1.0, t1, v_ovov, 1.0, r1);
  E("mien,mnea->ia", -1.0, v_oovo, asym, 1.0, r1);        // :1606-1607
  E("efma,mief->ia", 1.0, v_vvov, asym, 1.0, r1);         // :1618-1630
  E("ijae,eb->ijab", 1.0, t2, I_vv, 0.0, X);              // :1647
  E("miba,jm->ijab", -1.0, t2, I_oo, 1.0, X);             // :1654-1664
  {
    // :1669  particle-particle ladder (dominant): 1/2 c(ij,ef) <ef|ab> = 1/4 [S Vp + A Vm] unpacked over (a,b)
    const long long Pp = (long long)v * (v + 1) / 2, Pm = (long long)v * (v - 1) / 2;
    const int oo = o * o;
    Scratch sS(e.pool, (size_t)(oo * Pp)), sA(e.pool, (size_t)std::max<long long>(oo * Pm, 1));
    Scratch sLp(e.pool, (size_t)(oo * Pp)), sLm(e.pool, (size_t)std::max<long long>(oo * Pm, 1));
    pack_c(e, sS.p, sA.p, c.p(), oo, v);
    const bool sh = s.vpm_sharded;   // V_plus / V_minus hold this rank's column slab only
    dgemm_sharded(e, 'N', 'N', oo, (int)Pp, (int)Pp, 1.0, sS.p, oo, s.get("V_plus").p(), Pp, 0.0, sLp.p, sh, sh);
    if (Pm > 0)
      dgemm_sharded(e, 'N', 'N', oo, (int)Pm, (int)Pm, 1.0, sA.p, oo, s.get("V_minus").p(), Pm, 0.0, sLm.p, sh, sh);
    unpack_ladder(e, X.p(), sLp.p, sLm.p, oo, v, 0.5);
  }
  E("ijmn,mnab->ijab", 0.5, I_oooo, c, 1.0, X);           // :1673
  E("mjae,iemb->ijab", -1.0, t2, I_ovov, 1.0, X);         // :1680-1695 (three o^3v^3 rings)
  E("iema,mjeb->ijab", -1.0, I_ovov, t2, 1.0, X);
  E("miea,ejmb->ijab", 1.0, asym, I_voov, 1.0, X);
  {
    // t1(i,e) I_vovv_p(e,j,a,b) with I_vovv_p(c,i,a,b) = v_vvov(b,a,i,c) - v_oovv(m,i,c,b) t1(m,a)
    //                                                  - v_ovov(m,a,i,c) t1(m,b)            (:1261-1299, :1700)
    Scratch tmp(e.pool, (size_t)X.size());
    TView T1(tmp.p, {o, v, v, o});
    einsum(e, "ie,baje->ibaj", 1.0, V(t1), V(v_vvov), 0.0, T1);
    transpose(e, "ibaj->ijab", 1.0, T1, 1.0, V(X));
    Scratch q(e.pool, (size_t)o * o * o * v);
    TView Q(q.p, {o, o, o, v});
    einsum(e, "ie,mjeb->imjb", 1.0, V(t1), V(v_oovv), 0.0, Q);
    einsum(e, "imjb,ma->ijab", -1.0, Q, V(t1), 1.0, V(X));
    TView R(q.p, {o, o, v, o});
    einsum(e, "ie,maje->imaj", 1.0, V(t1), V(v_ovov), 0.0, R);
    einsum(e, "imaj,mb->ijab", -1.0, R, V(t1), 1.0, V(X));
  }
  E("ma,ijmb->ijab", -1.0, t1, I_ooov_p, 1.0, X);         // :1705-1715
  {
    // X <- X + X(j,i,b,a) + v_oovv  (:1721-1722), then the denominators (:1727-1728)
    Scratch tmp(e.pool, (size_t)X.size());
    TView Xt(tmp.p, X.dims);
    transpose(e, "ijab->jiba", 1.0, V(X), 0.0, Xt);
    axpby(st, X.size(), 1.0, tmp.p, 1.0, X.p());
    axpby(st, X.size(), 1.0, v_oovv.p(), 1.0, X.p());
  }
  divide_d2(st, X.p(), X.p(), s.eo.p(), s.ev.p(), o, v);
  divide_d1(st, r1.p(), r1.p(), s.eo.p(), s.ev.p(), o, v);
  std::swap(s.t1.buf, s.t1n.buf);
  std::swap(s.t2.buf, s.t2n.buf);
  s.iterations += 1;
}

// build_cr_ccsd_t_intermediates (src/ccsd.f90:2338-2551): I_vovv_pp(c,i,a,b), I_ooov_pp(j,k,i,a).
// Q3b: I_vo and asym_t2 are the ones left by the last iteration (built from its *input* amplitudes) unless the
// option is cleared, in which case they are rebuilt from the converged amplitudes.  Q3a: see the `es` slices.
void ccsd_spatial_cr_intermediates(CCState& s) {
  Engine& e = s.eng;
  cudaStream_t st = e.stream;
  const int o = s.o, v = s.v;
  Tensor &t1 = s.t1, &t2 = s.t2;
  Tensor &v_oovv = s.get("v_oovv"), &v_ovov = s.get("v_ovov"), &v_vvov = s.get("v_vvov"), &v_oovo = s.get("v_oovo"),
         &v_oooo = s.get("v_oooo");
  // The CR intermediates need <ec|ba> t1(i,e) once (:2515).  The dense v^4 slice (134 GB at nbf=400) is never formed:
  // the term is accumulated below from slabs over the last virtual index, gathered from the packed MO integrals.
  AFESP_REQUIRE(s.eri_mo.p != nullptr, "CR intermediates need the packed MO integrals on the device");
  s.drop("V_plus"); s.drop("V_minus");   // the iterations are over: make room (67 GB at nbf=400)
  Tensor &I_vo = s.get("I_vo"), &asym = s.get("asym_t2");
  if (!s.opt.q3b_stale_intermediates) {
    transpose(e, "ijab->jiab", -1.0, V(t2), 0.0, V(asym));
    axpby(st, asym.size(), 2.0, t2.p(), 1.0, asym.p());
    einsum(e, "imae,me->ai", 1.0, V(s.get("A_oovv")), V(t1), 0.0, V(I_vo));
  }
  auto E = [&](const char* spec, double alpha, const TView& a, const TView& b, double beta, const TView& cc) {
    einsum(e, spec, alpha, a, b, beta, cc);
  };
  // free what the reference frees (:2364-2365) to make room
  for (const char* nm : {"I_oooo", "I_ovov", "I_voov", "I_ooov_p", "x_voov", "c_oovv"}) s.drop(nm);
  Tensor x_vvvo_p({v, v, v, o}), x_vvvo({v, v, v, o}), x_ovov_p({o, v, o, v}), x_voov_p({v, o, o, v}),
      x_ovoo({o, v, o, o}), x_ovov_pp({o, v, o, v}), x_voov_pp({v, o, o, v});
  // x_vvvo_p(b,c,a,i) = v_vvov(c,b,i,a) - 1/2 t1(m,a) v_oovv(m,i,b,c)                     (:2425-2435)
  transpose(e, "cbia->bcai", 1.0, V(v_vvov), 0.0, V(x_vvvo_p));
  E("ma,mibc->bcai", -0.5, V(t1), V(v_oovv), 1.0, V(x_vvvo_p));
  // x_vvvo = x_vvvo_p - 1/2 t1(m,a) v_oovv(m,i,b,c)                                        (:2461-2471)
  AFESP_CUDA_CHECK(cudaMemcpyAsync(x_vvvo.p(), x_vvvo_p.p(), x_vvvo.size() * 8, cudaMemcpyDeviceToDevice, st));
  E("ma,mibc->bcai", -0.5, V(t1), V(v_oovv), 1.0, V(x_vvvo));
  // x_ovov_p(j,b,i,a) = v_ovov - 1/2 v_oovo(m,i,b,j) t1(m,a) + t1(j,e) x_vvvo_p(b,e,a,i)   (:2437-2447)
  AFESP_CUDA_CHECK(cudaMemcpyAsync(x_ovov_p.p(), v_ovov.p(), v_ovov.size() * 8, cudaMemcpyDeviceToDevice, st));
  E("mibj,ma->jbia", -0.5, V(v_oovo), V(t1), 1.0, V(x_ovov_p));
  E("je,beai->jbia", 1.0, V(t1), V(x_vvvo_p), 1.0, V(x_ovov_p));
  // x_voov_p(b,j,i,a) = v_oovv(i,j,b,a) - 1/2 v_oovo(i,m,b,j) t1(m,a) + x_vvvo_p(e,b,a,i) t1(j,e)   (:2449-2459)
  transpose(e, "ijba->bjia", 1.0, V(v_oovv), 0.0, V(x_voov_p));
  E("imbj,ma->bjia", -0.5, V(v_oovo), V(t1), 1.0, V(x_voov_p));
  E("ebai,je->bjia", 1.0, V(x_vvvo_p), V(t1), 1.0, V(x_voov_p));
  x_vvvo_p.free();
  // x_ovoo(k,a,i,j) = v_oovo(j,i,a,k) + t1(k,e) v_oovv(i,j,e,a)                            (:2473-2483)
  transpose(e, "jiak->kaij", 1.0, V(v_oovo), 0.0, V(x_ovoo));
  E("ke,ijea->kaij", 1.0, V(t1), V(v_oovv), 1.0, V(x_ovoo));
  // x_ovov_pp / x_voov_pp                                                                  (:2485-2507)
  AFESP_CUDA_CHECK(cudaMemcpyAsync(x_ovov_pp.p(), v_ovov.p(), v_ovov.size() * 8, cudaMemcpyDeviceToDevice, st));
  E("mibj,ma->jbia", -1.0, V(v_oovo), V(t1), 1.0, V(x_ovov_pp));
  E("je,beai->jbia", 0.5, V(t1), V(x_vvvo), 1.0, V(x_ovov_pp));
  transpose(e, "ijba->bjia", 1.0, V(v_oovv), 0.0, V(x_voov_pp));
  E("imbj,ma->bjia", -1.0, V(v_oovo), V(t1), 1.0, V(x_voov_pp));
  E("ebai,je->bjia", 0.5, V(x_vvvo), V(t1), 1.0, V(x_voov_pp));
  // I_vovv_pp(c,i,a,b)                                                                     (:2509-2525)
  Tensor& Ivv = s.make("I_vovv_pp", {v, o, v, v});
  transpose(e, "baic->ciab", 1.0, V(v_vvov), 0.0, V(Ivv));
  {
    // Ivv(c,i,a,b) += sum_e <ec|ba> t1(i,e), slab by slab over a:  Y(i; c,b,a') = t1(i,e) <ec|b a0+a'>  (one GEMM on
    // the gathered slab in place), then a strided permute-add into Ivv(c,i,a0+a',b).
    const long long v3 = (long long)v * v * v;
    const int nb = (int)std::max<long long>(1, std::min<long long>(v, (4LL << 30) / (v3 * 8)));
    const int nocc = s.nocc_spatial;   // first virtual orbital in the packed MO integrals
    Scratch slab(e.pool, (size_t)(v3 * nb)), y(e.pool, (size_t)((long long)o * v * v * nb));
    const long long ostr[4] = {1, v, (long long)v * o * v, (long long)v * o};   // out axes (c, i, b, a') inside Ivv
    for (int a0 = 0; a0 < v; a0 += nb) {
      const int cb = std::min(nb, v - a0);
      const int lo4[4] = {nocc, nocc, nocc, nocc + a0}, cnt4[4] = {v, v, v, cb};
      slice_phys(e, slab.p, s.eri_mo.p, lo4, cnt4);                       // slab(e,c,b,a')
      TView SL(slab.p, {v, v, v, cb}), Y(y.p, {o, v, v, cb});
      einsum(e, "ie,ecba->icba", 1.0, V(t1), SL, 0.0, Y);
      const int dims[4] = {o, v, v, cb}, perm[4] = {1, 0, 2, 3};           // Y(i,c,b,a') -> (c,i,b,a')
      permute_strided(st, 4, dims, perm, 1.0, y.p, 1.0, Ivv.p() + (long long)a0 * v * o, ostr);
    }
  }
  E("icma,mb->ciab", -1.0, V(x_ovov_p), V(t1), 1.0, V(Ivv));
  E("ma,cimb->ciab", -1.0, V(t1), V(x_voov_p), 1.0, V(Ivv));
  E("cm,miab->ciab", -1.0, V(I_vo), V(t2), 1.0, V(Ivv));
  E("mnba,icmn->ciab", 1.0, V(t2), V(x_ovoo), 1.0, V(Ivv));
  E("ceam,imbe->ciab", 1.0, V(x_vvvo), V(asym), 1.0, V(Ivv));
  E("ecam,mieb->ciab", -1.0, V(x_vvvo), V(t2), 1.0, V(Ivv));
  E("miae,ecbm->ciab", -1.0, V(t2), V(x_vvvo), 1.0, V(Ivv));
  // I_ooov_pp(j,k,i,a)                                                                     (:2527-2544)
  Tensor& Ioo = s.make("I_ooov_pp", {o, o, o, v});
  transpose(e, "kjai->jkia", 1.0, V(v_oovo), 0.0, V(Ioo));
  E("mikj,ma->jkia", -1.0, V(v_oooo), V(t1), 1.0, V(Ioo));
  E("jeia,ke->jkia", 1.0, V(x_ovov_pp), V(t1), 1.0, V(Ioo));
  E("je,ekia->jkia", 1.0, V(t1), V(x_voov_pp), 1.0, V(Ioo));
  E("kjef,efai->jkia", 1.0, V(t2), V(x_vvvo), 1.0, V(Ioo));
  {
    // Q3a: the reference's `do e = 1, nocc` runs the virtual index e only over its first nocc values (:2535).
    const int ne = s.opt.q3a_truncated_e ? std::min(o, v) : v;
    // gather the e-slices so the contractions stay plain GEMMs
    Tensor xo({o, ne, o, o}), ase({o, o, ne, v}), t2e({o, o, ne, v}), t2ae({o, o, v, ne});
    // x_ovoo(j,e,i,m), e < ne
    {
      int dims[4] = {o, v, o, o};
      // strided copy via permute on a view is not available; use einsum with an identity selector instead:
      // build selector P(e', e) = delta(e', e) for e' < ne and contract.  Cheap (o^3 v ne).
      Tensor P({ne, v});
      fill(st, P.size(), 0.0, P.p());
      std::vector<double> hp((size_t)ne * v, 0.0);
      for (int k = 0; k < ne; ++k) hp[k + (size_t)ne * k] = 1.0;
      AFESP_CUDA_CHECK(cudaMemcpyAsync(P.p(), hp.data(), hp.size() * 8, cudaMemcpyHostToDevice, st));
      AFESP_CUDA_CHECK(cudaStreamSynchronize(st));
      (void)dims;
      E("xe,jeim->jxim", 1.0, V(P), V(x_ovoo), 0.0, V(xo));
      E("xe,mkea->mkxa", 1.0, V(P), V(asym), 0.0, V(ase));
      E("xe,mkea->mkxa", 1.0, V(P), V(t2), 0.0, V(t2e));
      E("mjae,xe->mjax", 1.0, V(t2), V(P), 0.0, V(t2ae));
    }
    E("jeim,mkea->jkia", 1.0, V(xo), V(ase), 1.0, V(Ioo));
    E("jemi,mkea->jkia", -1.0, V(xo), V(t2e), 1.0, V(Ioo));
    E("mjae,kemi->jkia", -1.0, V(t2ae), V(xo), 1.0, V(Ioo));
  }
  s.have_cr = true;
}

}  // namespace afesp
