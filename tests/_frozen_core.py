"""Frozen core on top of the NumPy oracle (test infrastructure; the product never imports it).

With canonical RHF orbitals the frozen-core Fock operator is diagonal with unchanged orbital energies, so a calculation
with k frozen orbitals is, by definition, the same calculation on the active-orbital integrals: orbitals k..n-1 repacked,
eps[k:], nocc-k doubly occupied.  `active_space` states that once; `run` is oracle/afesp_oracle.py's whole program with
the correlated stages on the active space; `FrozenCoreEngine` is the oracle engine of the host tests with the
library's option "frozen_core".
"""
import numpy as np

from oracle import afesp_oracle as orc
from tests._double import bridge
from tests._oracle_engine import OracleEngine


def active_space(eri_mo_packed, eps, nocc, k):
    """(packed MO integrals over orbitals k..n-1, eps[k:], nocc - k); k = 0 returns the inputs unchanged."""
    if k == 0:
        return eri_mo_packed, eps, nocc
    n = len(eps)
    p, q = np.tril_indices(n - k)  # active pairs in packed order (see orc.pack_eri)
    full = orc.tri(p + k, q + k)   # the same pairs in the full orbital range
    a, b = np.tril_indices(full.size)
    return np.ascontiguousarray(np.asarray(eri_mo_packed)[orc.tri(full[a], full[b])]), np.asarray(eps)[k:], nocc - k


def run(sysm, k, q1=True, q3a=True, q3b=True):
    """orc.run (src/main.F90) with MP2, CCSD and the triples on the active space of k frozen orbitals."""
    level, restricted, paren, renorm, comp_renorm = orc.CALC_TYPES[sysm.calc_type]
    orc.do_rhf(sysm)
    res = {"e_hf": sysm.e_hf, "e_nuc": sysm.e_nuc, "scf": sysm.log["scf"]}
    if level == "HF":
        return res
    sysm.eri_mo = orc.ao2mo_packed(sysm.eri, sysm.coeff)
    eri_mo, eps, nocc = active_space(sysm.eri_mo, sysm.eps, sysm.nel // 2, k)
    res["e_mp2"] = orc.mp2_energy(eri_mo, eps, nocc)
    if level == "MP2":
        return res
    if restricted:
        cc = orc.ccsd_spatial(eri_mo, eps, nocc, sysm.ccsd_e_tol, sysm.ccsd_t_tol, sysm.ccsd_diis_n_errmat,
                              sysm.ccsd_maxiter, want_cr=comp_renorm, q3a=q3a, q3b=q3b)
        res.update(ccsd=cc["table"], e_ccsd=cc["e_ccsd"], t1_diag=cc["t1_diag"])
        if level == "CCSD(T)":
            en, sums = orc.triples_spatial(cc, eps, paren, renorm, comp_renorm)
            res.update(en)
            res["triples_sums"] = sums
    else:
        cc = orc.ccsd_spinorb(eri_mo, eps, sysm.nel - 2 * k, sysm.ccsd_e_tol, sysm.ccsd_t_tol,
                              sysm.ccsd_diis_n_errmat, sysm.ccsd_maxiter, q1=q1)
        res.update(ccsd=cc["table"], e_ccsd=cc["e_ccsd"])
        if level == "CCSD(T)":
            G = cc["G"]
            res["e_ccsd_t"] = cc["e_ccsd"] + orc.triples_spinorb(cc["t1"], cc["t2"], G["oovv"], G["vovv"], G["ovoo"],
                                                                 cc["eps_so"])
    res["cc"] = cc
    return res


class FrozenCoreEngine(OracleEngine):
    """OracleEngine plus option "frozen_core": mp2_energy and ccsd_init see the active space, and the CC state keeps it
    (t1 / t2 / eps / nocc of the state are the active ones, as in the library)."""

    def __init__(self, **kw):
        super().__init__(**kw)
        self.frozen_core = 0

    def set_option(self, key, value):
        super().set_option(key, value)
        if key == "frozen_core":
            self.frozen_core = int(value)

    def mp2_energy(self, nocc, eps):
        self._log("mp2_energy")
        return orc.mp2_energy(*active_space(self.eri_mo, np.asarray(eps), int(nocc), self.frozen_core))

    def ccsd_init(self, nocc, restricted, eps, diis_n=8):
        k = self.frozen_core
        eri_full, n_full = self.eri_mo, self.n
        self.eri_mo, eps, nocc = active_space(eri_full, np.asarray(eps, dtype=float), int(nocc), k)
        self.n = n_full - k
        try:
            return super().ccsd_init(nocc, restricted, eps, diis_n)
        finally:
            self.eri_mo, self.n = eri_full, n_full


class Bridge(bridge.Bridge):
    """The C test double's bridge (tests/_double/bridge.py) over FrozenCoreEngine; loaded by tests/_frozen_core_double.c."""

    def __init__(self):
        super().__init__()
        self.eng = FrozenCoreEngine()
