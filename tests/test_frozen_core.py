"""Frozen-core MP2 / CCSD / triples on the CPU: the active-space definition (tests/_frozen_core.py) against pinned values,
and the `frozen_core` namelist key through both host programs (afesp_b200/host.py over the oracle engine with the option,
host/els_host.cpp over the C test double built on it, tests/_frozen_core_double.c).

A frozen-core calculation with k frozen orbitals is, by definition, the same calculation on the active-orbital integrals
(orbitals k..n-1, eps[k:], nocc-k doubly occupied): with canonical RHF orbitals the frozen-core Fock operator is diagonal
with unchanged orbital energies.  The pinned values below are that recipe (RHF, AO->MO, restrict and repack, then
ccsd_spatial with the CR intermediates and triples_spatial) on the shipped N2 / F2 inputs with k = 2.
"""
import os
import re
import subprocess
import sysconfig

import numpy as np
import pytest

from oracle import afesp_oracle as orc
from tests import _frozen_core as fc
from tests._fixtures import compare_els_out, els_host_binary, load_system, write_sample_dir

E_TOL = 1e-9

# k = 2, calc_type CRCCSD(T)_spatial: correlation energies (Eh), CCSD iteration count, T1 diagnostic, D[T] / D(T)
PINNED = {
    "n2": {"e_mp2": -0.8424179352, "e_ccsd": -0.5789372271, "iterations": 22, "t1_diag": 0.0383269295,
           "e_ccsd_t": -0.6968571526, "e_ccsd_tt": -0.6822998871, "e_rccsd_t": -0.6403002041, "e_rccsd_tt": -0.6325945884,
           "e_crccsd_t": -0.6256657973, "e_crccsd_tt": -0.6209014028, "D_T": 1.9216786933, "D_TT": 1.9263463103},
    "f2": {"e_mp2": -0.4333018929, "e_ccsd": -0.4468334864, "iterations": 15, "t1_diag": 0.0156110231,
           "e_ccsd_t": -0.4673498250, "e_ccsd_tt": -0.4663606352, "e_rccsd_t": -0.4638786519, "e_rccsd_tt": -0.4630533587,
           "e_crccsd_t": -0.4623683882, "e_crccsd_tt": -0.4615948145, "D_T": 1.2036456059, "D_TT": 1.2039027448},
}
# labels of the final energy block (src/main.F90:123-175) -> keys above
FINAL_LABELS = {"MP2 correlation energy:": "e_mp2", "CCSD correlation energy:": "e_ccsd",
                "CCSD[T] correlation energy:": "e_ccsd_t", "CCSD(T) correlation energy:": "e_ccsd_tt",
                "R-CCSD[T] correlation energy:": "e_rccsd_t", "R-CCSD(T) correlation energy:": "e_rccsd_tt",
                "CR-CCSD[T] correlation energy:": "e_crccsd_t", "CR-CCSD(T) correlation energy:": "e_crccsd_tt",
                "T1 diagnostic:": "t1_diag", "D[T]:": "D_T", "D(T):": "D_TT"}


ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def fc_double_env(double_env, tmp_path_factory):
    """double_env with the C double whose engine honours "frozen_core" LD_PRELOADed instead (built like double_env)."""
    out = tmp_path_factory.mktemp("fc_double") / "afesp_gpu_fc_double.so"
    cmd = ["gcc", "-O1", "-shared", "-fPIC", "-I", sysconfig.get_config_var("INCLUDEPY"),
           os.path.join(ROOT, "tests", "_frozen_core_double.c"), "-o", str(out), "-L", sysconfig.get_config_var("LIBDIR"),
           "-lpython" + sysconfig.get_config_var("LDVERSION"), "-Wl,-rpath," + sysconfig.get_config_var("LIBDIR")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    return dict(double_env, LD_PRELOAD=str(out))


def _with_frozen_core(text, k):
    """els.in with `frozen_core = k` added before the closing `/` of the namelist group."""
    head, sep, tail = text.rpartition("/")
    assert sep
    return head.rstrip("\n") + ",\nfrozen_core = %d\n/" % k + tail


def _final_block(stdout):
    out = {}
    for line in stdout.splitlines():
        for label, key in FINAL_LABELS.items():
            if line.startswith(" " + label):
                out[key] = float(line[len(label) + 1:])
    return out


@pytest.mark.parametrize("name", ["n2", "f2"])
def test_oracle_frozen_core_reproduces_the_pinned_values(name):
    r = fc.run(load_system(name, "CRCCSD(T)_spatial"), 2)
    want = PINNED[name]
    assert r["cc"]["iterations"] == want["iterations"]
    got = {k: r[k] for k in want if k != "iterations"}
    for k, v in got.items():
        assert abs(v - want[k]) < E_TOL, (k, v, want[k])


def test_active_space_is_the_restricted_and_repacked_integral_array():
    s = load_system("n2", "MP2_spatial")
    orc.do_rhf(s)
    mo = orc.ao2mo_packed(s.eri, s.coeff)
    for k in [1, 2, 3]:
        act, eps, nocc = fc.active_space(mo, s.eps, s.nocc, k)
        want = orc.pack_eri(orc.unpack_eri(mo, s.nbasis)[k:, k:, k:, k:])
        assert np.array_equal(act, want) and np.array_equal(eps, s.eps[k:]) and nocc == s.nocc - k
    same = fc.active_space(mo, s.eps, s.nocc, 0)
    assert same[0] is mo and same[1] is s.eps and same[2] == s.nocc


@pytest.mark.parametrize("name,calc", [("n2", None), ("f2", None), ("h2o", "CCSD(T)_spinorb")])
def test_frozen_core_zero_is_the_all_electron_oracle_run(name, calc, oracle_runs):
    _, ref = oracle_runs(name, calc)
    r = fc.run(load_system(name, calc), 0)
    for k in ["e_mp2", "e_ccsd", "t1_diag", "e_ccsd_t", "e_crccsd_tt", "D_TT"]:
        assert (k in r) == (k in ref) and r.get(k) == ref.get(k), k
    assert r["ccsd"] == ref["ccsd"]
    if "triples_sums" in ref:
        assert np.array_equal(r["triples_sums"], ref["triples_sums"])


def test_both_hosts_run_n2_with_frozen_core_and_print_the_same_text(fc_double_env, tmp_path):
    """N2 CRCCSD(T)_spatial with frozen_core = 2: the Python host over the oracle engine and els_host over the C double
    print the pinned energies, set the option before the MP2 stage and print identical text (times masked)."""
    from afesp_b200 import host

    text = _with_frozen_core(write_sample_dir("n2", str(tmp_path)), 2)
    (tmp_path / "els.in").write_text(text)
    log = tmp_path / "calls.log"
    r = subprocess.run([els_host_binary(), str(tmp_path)], capture_output=True, text=True, timeout=900,
                       env=dict(fc_double_env, AFESP_DOUBLE_CALL_LOG=str(log)))
    assert r.returncode == 0, r.stderr[-3000:]
    calls = log.read_text().split()
    assert calls.index("set_option") < calls.index("mp2_energy")

    inp = host.read_inputs(str(tmp_path))
    assert inp.frozen_core == 2
    eng = fc.FrozenCoreEngine()
    res = host.run(inp, gpu=eng)
    assert eng.calls.index("set_option:frozen_core") < eng.calls.index("mp2_energy")
    assert len(res.ccsd_table) - 1 == PINNED["n2"]["iterations"]

    for stdout in (res.stdout, r.stdout):
        lines = stdout.splitlines()
        k = lines.index(" Number of virtual orbitals: 21")
        assert lines[k + 1] == " Number of frozen core orbitals: 2"
        got = _final_block(stdout)
        assert set(got) == set(FINAL_LABELS.values())
        for key, v in got.items():
            assert abs(v - PINNED["n2"][key]) < E_TOL, (key, v)
    diffs = compare_els_out(r.stdout, res.stdout, ulps=1.0, abs_tol=1e-10)
    assert diffs == [], "\n".join(diffs[:20])


def test_namelist_key_is_parsed():
    from afesp_b200 import host

    assert host.parse_namelist("&elsinput calc_type='MP2_spatial', frozen_core = 3 /") == {
        "calc_type": "MP2_spatial", "frozen_core": 3}
    assert host.ElsInput().frozen_core == 0


@pytest.mark.parametrize("k", [-1, 7])
def test_out_of_range_frozen_core_is_rejected_with_the_same_message_by_both_hosts(fc_double_env, k, tmp_path):
    """N2 has nocc = 7: frozen_core must lie in 0..6."""
    from afesp_b200 import host

    text = _with_frozen_core(write_sample_dir("n2", str(tmp_path), calc_type="MP2_spatial"), k)
    (tmp_path / "els.in").write_text(text)
    inp = host.read_inputs(str(tmp_path))
    eng = fc.FrozenCoreEngine()
    with pytest.raises(ValueError) as ei:
        host.run(inp, gpu=eng)
    assert eng.calls == []
    where, msg = str(ei.value).split(": ", 1)
    assert where == "system::read_system_in" and msg == "frozen_core = %d is outside 0..6 (nocc - 1)!" % k
    r = subprocess.run([els_host_binary(), str(tmp_path)], capture_output=True, text=True, timeout=300, env=fc_double_env)
    assert r.returncode != 0
    assert "Programme stops in procedure: %s." % where in r.stderr and "Reason: %s." % msg in r.stderr
    assert "System information" not in r.stdout
