// Spin-orbital CCSD on the device: Stanton, Gauss, Watts, Bartlett, JCP 94, 4334 (1991) as coded by the reference in
// src/ccsd.f90:71-277 (do_ccsd_spinorb), 678-715 (build_tau), 717-797 (build_F), 799-905 (build_W) and 907-1038
// (update_amplitudes).  RHF orbitals are spin-blocked: spin-orbital 2p is alpha, 2p+1 beta of spatial orbital p.
//
// The reference's bottleneck, the 6-deep o^3 v^3 loop nest at :980-992, and its other naive loops (:748-783,
// :947-961) are DMMA GEMMs here.  Q1 (SURVEY.md App. B): the 1/2 tau~ <mn||ef> term of F_mi is added transposed,
// exactly as the dgemm at :793-795 does, unless Options::q1_transposed_foo is cleared.
#include "ccsd.cuh"

namespace afesp {

namespace {
inline TView V(Tensor& t) { return t.view(); }
}  // namespace

void ccsd_spinorb_init(CCState& s, int diis_n) {
  const int n = s.n;
  // active occupied spin-orbitals start at 2 nfrozen (frozen core), virtual ones at 2 nocc
  const int olo = 2 * s.nfrozen, vlo = 2 * s.nocc_spatial;
  const int o = vlo - olo, v = 2 * n - vlo;
  s.restricted = false;
  s.o = o; s.v = v;
  AFESP_REQUIRE(o > 0 && v > 0, "ccsd init: need at least one occupied and one virtual orbital");
  Engine& e = s.eng;
  // canon_levels_spinorb (src/ccsd.f90:460-463)
  std::vector<double> es(2 * n);
  for (int p = 0; p < n; ++p) es[2 * p] = es[2 * p + 1] = s.eps_host[p];
  s.eo.init({o}); s.ev.init({v});
  AFESP_CUDA_CHECK(cudaMemcpyAsync(s.eo.p(), es.data() + olo, o * 8, cudaMemcpyHostToDevice, e.stream));
  AFESP_CUDA_CHECK(cudaMemcpyAsync(s.ev.p(), es.data() + vlo, v * 8, cudaMemcpyHostToDevice, e.stream));
  AFESP_CUDA_CHECK(cudaStreamSynchronize(e.stream));
  // nine slices of <pq||rs> (src/ccsd.f90:182-194), gathered straight from the packed MO integrals: the (2n)^4
  // tensor of :108 is never formed.
  cudaEvent_t ev[3];
  for (auto& x : ev) AFESP_CUDA_CHECK(cudaEventCreate(&x));
  AFESP_CUDA_CHECK(cudaEventRecord(ev[0], e.stream));
  for (const char* nm : {"oooo", "ooov", "ovoo", "oovo", "oovv", "ovvo", "ovvv", "vovv", "vvvv"}) {
    int lo[4], cnt[4];
    std::vector<int> dims;
    for (int d = 0; d < 4; ++d) {
      lo[d] = nm[d] == 'o' ? olo : vlo;
      cnt[d] = nm[d] == 'o' ? o : v;
      dims.push_back(cnt[d]);
    }
    Tensor& t = s.make(nm, dims);
    slice_spinorb(e, t.p(), s.eri_mo.p, lo, cnt);
  }
  AFESP_CUDA_CHECK(cudaEventRecord(ev[1], e.stream));
  // the reference's run-time assertion on <pq||rs> (src/ccsd.f90:150-167): same index set, same four identities, same
  // threshold (depsilon), over the active spin-orbitals; a violation aborts the calculation with the reference's message
  if (s.red_out.n < 16) s.red_out.alloc(16);
  spinorb_symmetry_error(e, n, olo, s.eri_mo.p, s.red_out.p);
  AFESP_CUDA_CHECK(cudaEventRecord(ev[2], e.stream));
  AFESP_CUDA_CHECK(cudaMemcpyAsync(&s.sym_err, s.red_out.p, 8, cudaMemcpyDeviceToHost, e.stream));
  AFESP_CUDA_CHECK(cudaStreamSynchronize(e.stream));
  float ms01 = 0.f, ms12 = 0.f;
  cudaEventElapsedTime(&ms01, ev[0], ev[1]);
  cudaEventElapsedTime(&ms12, ev[1], ev[2]);
  for (auto& x : ev) cudaEventDestroy(x);
  s.ms_slices = ms01; s.ms_symcheck = ms12;
  if (!(s.sym_err <= s.opt.spinorb_symmetry_tol))
    throw Error(5, "Permutational symmetry of antisymmetrised integrals does not hold");
  s.t1.init({o, v}); s.t1n.init({o, v});
  s.t2.init({o, o, v, v}); s.t2n.init({o, o, v, v}); s.t2_old.init({o, o, v, v});
  fill(e.stream, s.t1.size(), 0.0, s.t1.p());
  fill(e.stream, s.t2_old.size(), 0.0, s.t2_old.p());
  divide_d2(e.stream, s.t2.p(), s.get("oovv").p(), s.eo.p(), s.ev.p(), o, v);  // MP1 guess (:523)
  s.make("F_vv", {v, v}); s.make("F_oo", {o, o}); s.make("F_ov", {o, v});
  s.make("W_ijmn", {o, o, o, o}); s.make("W_efab", {v, v, v, v}); s.make("W_ovvo", {o, v, v, o});
  s.make("tau", {o, o, v, v}); s.make("tau_tilde", {o, o, v, v});
  s.diis.init(diis_n, o, v);
  s.energy = s.energy_old = 0.0;
  s.iterations = 0;
  s.finalized = false;
}

void ccsd_spinorb_iterate(CCState& s) {
  Engine& e = s.eng;
  cudaStream_t st = e.stream;
  const int o = s.o, v = s.v;
  Tensor &t1 = s.t1, &t2 = s.t2;
  Tensor &oooo = s.get("oooo"), &ooov = s.get("ooov"), &oovo = s.get("oovo"), &oovv = s.get("oovv"),
         &ovvo = s.get("ovvo"), &ovvv = s.get("ovvv"), &vovv = s.get("vovv"), &vvvv = s.get("vvvv");
  Tensor &F_vv = s.get("F_vv"), &F_oo = s.get("F_oo"), &F_ov = s.get("F_ov"), &W_ijmn = s.get("W_ijmn"),
         &W_efab = s.get("W_efab"), &W_ovvo = s.get("W_ovvo"), &tau = s.get("tau"), &tau_t = s.get("tau_tilde");
  auto E = [&](const char* spec, double alpha, const TView& a, const TView& b, double beta, const TView& cc) {
    einsum(e, spec, alpha, a, b, beta, cc);
  };
  const long long n2 = t2.size();

  // build_tau (:678-715)
  t2_plus_t1t1(st, tau_t.p(), t2.p(), t1.p(), o, v, 0.5, -0.5);
  t2_plus_t1t1(st, tau.p(), t2.p(), t1.p(), o, v, 1.0, -1.0);
  // build_F (:717-797)
  E("mf,mafe->ae", 1.0, V(t1), V(ovvv), 0.0, V(F_vv));               // :748-757
  E("mnaf,mnfe->ae", 0.5, V(tau_t), V(oovv), 1.0, V(F_vv));          // :787-790
  E("ne,nmie->mi", -1.0, V(t1), V(ooov), 0.0, V(F_oo));              // :760-770
  if (s.opt.q1_transposed_foo) E("rnef,cnef->rc", 0.5, V(tau_t), V(oovv), 1.0, V(F_oo));  // as coded (:793-795)
  else E("rnef,cnef->cr", 0.5, V(tau_t), V(oovv), 1.0, V(F_oo));                           // Stanton Eq. 4
  E("nf,mnef->me", 1.0, V(t1), V(oovv), 0.0, V(F_ov));               // :773-783
  // build_W (:799-905)
  {
    Scratch w(e.pool, (size_t)oooo.size()), sc(e.pool, (size_t)oooo.size());
    TView Wm(w.p, {o, o, o, o}), S(sc.p, {o, o, o, o});
    AFESP_CUDA_CHECK(cudaMemcpyAsync(w.p, oooo.p(), oooo.size() * 8, cudaMemcpyDeviceToDevice, st));
    E("mnie,je->mnij", 1.0, V(ooov), V(t1), 0.0, S);                 // :828
    axpby(st, oooo.size(), 1.0, sc.p, 1.0, w.p);
    transpose(e, "mnij->mnji", -1.0, S, 1.0, Wm);                    // :829-830
    E("mnef,ijef->mnij", 0.5, V(oovv), V(tau), 1.0, Wm);             // :835-836
    transpose(e, "mnij->ijmn", 1.0, Wm, 0.0, V(W_ijmn));             // :841-842
  }
  {
    Scratch sc(e.pool, (size_t)vvvv.size());
    TView S(sc.p, {v, v, v, v});
    E("mb,maef->baef", 1.0, V(t1), V(ovvv), 0.0, S);                 // :850  scratch(b,a,e,f)
    transpose(e, "abef->efab", 1.0, V(vvvv), 0.0, V(W_efab));        // :854-857
    transpose(e, "baef->efab", 1.0, S, 1.0, V(W_efab));
    transpose(e, "abef->efab", -1.0, S, 1.0, V(W_efab));
  }
  {
    AFESP_CUDA_CHECK(cudaMemcpyAsync(W_ovvo.p(), ovvo.p(), ovvo.size() * 8, cudaMemcpyDeviceToDevice, st));
    E("mbef,jf->mbej", 1.0, V(ovvv), V(t1), 1.0, V(W_ovvo));         // :864-865
    E("nb,nmej->mbej", 1.0, V(t1), V(oovo), 1.0, V(W_ovvo));         // :870-873
    Scratch sc(e.pool, (size_t)n2);
    TView S(sc.p, {o, v, o, v});                                     // scratch(n,f,j,b) :885-893
    E("jf,nb->nfjb", 1.0, V(t1), V(t1), 0.0, S);
    transpose(e, "jnfb->nfjb", 0.5, V(t2), 1.0, S);
    E("mnef,nfjb->mbej", -1.0, V(oovv), S, 1.0, V(W_ovvo));          // :897-901
  }
  // update_amplitudes (:907-1038)
  Tensor &r1 = s.t1n, &r2 = s.t2n;
  E("ie,ae->ia", 1.0, V(t1), V(F_vv), 0.0, V(r1));                   // :939
  E("mi,ma->ia", -1.0, V(F_oo), V(t1), 1.0, V(r1));                  // :941
  E("me,maei->ia", 1.0, V(t1), V(ovvo), 1.0, V(r1));                 // :947-961
  E("miea,me->ia", 1.0, V(t2), V(F_ov), 1.0, V(r1));
  E("mife,mafe->ia", 0.5, V(t2), V(ovvv), 1.0, V(r1));
  E("mnea,mnei->ia", -0.5, V(t2), V(oovo), 1.0, V(r1));
  divide_d1(st, r1.p(), r1.p(), s.eo.p(), s.ev.p(), o, v);           // :963

  Scratch sbuf(e.pool, (size_t)n2);
  TView S(sbuf.p, {o, o, v, v});
  auto acc = [&](double c_id, double c_ji, double c_ba, double c_jiba) {  // r2 += sum of permuted copies of S
    if (c_id != 0.0) axpby(st, n2, c_id, sbuf.p, 1.0, r2.p());
    if (c_ji != 0.0) transpose(e, "ijab->jiab", c_ji, S, 1.0, V(r2));
    if (c_ba != 0.0) transpose(e, "ijab->ijba", c_ba, S, 1.0, V(r2));
    if (c_jiba != 0.0) transpose(e, "ijab->jiba", c_jiba, S, 1.0, V(r2));
  };
  AFESP_CUDA_CHECK(cudaMemcpyAsync(r2.p(), oovv.p(), n2 * 8, cudaMemcpyDeviceToDevice, st));  // <ij||ab> :975
  {
    // P(ij)P(ab)[t2(m,i,e,a) W_ovvo(m,b,e,j) - t1(i,e) t1(m,a) ovvo(m,b,e,j)]        (:980-1000)
    Scratch u(e.pool, (size_t)o * o * v * o);
    TView U(u.p, {o, o, v, o});
    E("ie,mbej->imbj", 1.0, V(t1), V(ovvo), 0.0, U);
    E("imbj,ma->ijab", -1.0, U, V(t1), 0.0, S);
    E("miea,mbej->ijab", 1.0, V(t2), V(W_ovvo), 1.0, S);
    acc(1.0, -1.0, -1.0, 1.0);
  }
  E("ijae,be->ijab", 1.0, V(t2), V(F_vv), 0.0, S);                   // :1003-1005
  acc(1.0, 0.0, -1.0, 0.0);
  {
    Tensor M({v, v}), Nn({o, o});
    E("mb,me->be", 1.0, V(t1), V(F_ov), 0.0, V(M));                  // matmul(transpose(t1),F_ov) :1007
    E("ijae,be->ijab", 1.0, V(t2), V(M), 0.0, S);
    acc(-0.5, 0.0, 0.5, 0.0);
    E("ie,me->im", 1.0, V(t1), V(F_ov), 0.0, V(Nn));                 // matmul(t1,transpose(F_ov)) :1011
    E("im,mjab->ijab", 1.0, V(Nn), V(t2), 0.0, S);
    acc(-0.5, 0.5, 0.0, 0.0);
    AFESP_CUDA_CHECK(cudaStreamSynchronize(st));  // M, Nn are freed at scope exit
  }
  E("ie,ejab->ijab", 1.0, V(t1), V(vovv), 0.0, S);                   // :1015-1017
  acc(1.0, -1.0, 0.0, 0.0);
  E("ijam,mb->ijab", 1.0, V(oovo), V(t1), 0.0, S);                   // :1019-1022
  acc(-1.0, 0.0, 1.0, 0.0);
  E("mi,mjab->ijab", 1.0, V(F_oo), V(t2), 0.0, S);                   // :1024-1026
  acc(-1.0, 1.0, 0.0, 0.0);
  E("ijmn,mnab->ijab", 0.5, V(W_ijmn), V(tau), 1.0, V(r2));          // :1028
  E("ijef,efab->ijab", 0.5, V(tau), V(W_efab), 1.0, V(r2));          // :1030  particle-particle ladder
  divide_d2(st, r2.p(), r2.p(), s.eo.p(), s.ev.p(), o, v);           // :1034
  std::swap(s.t1.buf, s.t1n.buf);
  std::swap(s.t2.buf, s.t2n.buf);
  s.iterations += 1;
}

}  // namespace afesp
