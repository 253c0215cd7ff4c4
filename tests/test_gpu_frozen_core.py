"""Frozen core on the device (option "frozen_core"): against the oracle on the sample molecules, and against the same
library fed the active-orbital integrals at a multi-tile synthetic shape.

k = 3 at nbf = 120 / nocc = 12 leaves o = 9 active occupied orbitals next to v = 108 virtual ones: the (T) GEMM depth
K = v + o is odd there and is padded with one zero column / row (triples.cu); k = 2 is the even case.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import _frozen_core as fc
from tests._fixtures import load_els_input, load_system

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
E_TOL = 1e-9
REL = 1e-12
N, NOCC = 120, 12


@pytest.fixture(scope="module")
def gpu():
    from afesp_b200 import AfespGpu

    g = AfespGpu(0)
    yield g
    g.close()


@pytest.fixture
def fresh(gpu):
    """The module's handle with frozen_core back at 0 after the test."""
    yield gpu
    gpu.set_option("frozen_core", 0)


@pytest.fixture(scope="module")
def synth():
    from afesp_b200 import synthetic

    return synthetic.make(N, NOCC, seed=5)


def _chain(g, nbasis, nocc, eps, mo_packed=None, ao=None, iters=3):
    """ao2mo (or set_eri_mo), MP2, ccsd_init, `iters` plain iterations, finalize with CR intermediates, six (T) sums."""
    if ao is not None:
        mo = g.ao2mo(nbasis, ao[0], ao[1], want_result=True)
    else:
        g.set_eri_mo(nbasis, mo_packed)
        mo = None
    e_mp2 = g.mp2_energy(nocc, eps)
    rows = [g.ccsd_init(nocc, True, eps, 8)]
    for _ in range(iters):
        rows.append(g.ccsd_iterate())
    t1_diag, t1, t2 = g.ccsd_finalize(want_cr=True, want_amplitudes=True)
    sums, const = g.ccsd_t_spatial(True, False, True)
    return {"mo": mo, "e_mp2": e_mp2, "rows": np.array(rows), "t1_diag": t1_diag, "t1": t1, "t2": t2,
            "sums": np.array(sums), "const": const}


def _close(a, b, rel=REL):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    assert a.shape == b.shape
    scale = max(float(np.max(np.abs(b))), 1e-300)
    return float(np.max(np.abs(a - b))) <= rel * scale


def test_frozen_core_zero_is_bit_identical_to_not_setting_it(gpu, synth):
    """First in the module: the handle has never seen the option."""
    eri, C, eps = synth
    ref = _chain(gpu, N, NOCC, eps, ao=(eri, C))
    gpu.set_option("frozen_core", 0)
    got = _chain(gpu, N, NOCC, eps, ao=(eri, C))
    for k in ["mo", "e_mp2", "rows", "t1_diag", "t1", "t2", "sums", "const"]:
        assert np.array_equal(np.asarray(got[k]), np.asarray(ref[k])), k


def test_guards(fresh, synth):
    from afesp_b200.capi import AfespError

    eri, C, eps = synth
    for bad in [-1, 1.5]:
        with pytest.raises(AfespError) as ei:
            fresh.set_option("frozen_core", bad)
        assert ei.value.code == 1 and "frozen_core" in str(ei.value)
    fresh.ao2mo(N, eri, C, want_result=False)
    fresh.set_option("frozen_core", NOCC)
    for call in (lambda: fresh.mp2_energy(NOCC, eps), lambda: fresh.ccsd_init(NOCC, True, eps, 8)):
        with pytest.raises(AfespError) as ei:
            call()
        assert ei.value.code == 1 and "frozen_core" in str(ei.value)


@pytest.mark.parametrize("k", [3, 2])
def test_frozen_core_equals_the_active_space_integrals_at_a_multi_tile_shape(fresh, synth, k):
    eri, C, eps = synth
    fresh.set_option("frozen_core", k)
    frz = _chain(fresh, N, NOCC, eps, ao=(eri, C))
    assert fresh.o == NOCC - k and frz["t2"].shape == (NOCC - k, NOCC - k, N - NOCC, N - NOCC)
    fresh.set_option("frozen_core", 0)
    act, eps_a, nocc_a = fc.active_space(frz["mo"], eps, NOCC, k)
    ref = _chain(fresh, N - k, nocc_a, eps_a, mo_packed=act)
    assert _close(frz["e_mp2"], ref["e_mp2"])
    assert _close(frz["rows"][:, 0], ref["rows"][:, 0]) and _close(frz["rows"][:, 1], ref["rows"][:, 1])
    assert _close(frz["t1_diag"], ref["t1_diag"]) and _close(frz["t1"], ref["t1"]) and _close(frz["t2"], ref["t2"])
    assert _close(frz["sums"], ref["sums"]) and _close(frz["const"], ref["const"])


def test_padded_triples_at_odd_o_agree_between_the_tma_and_cpasync_kernels(fresh, synth):
    eri, C, eps = synth
    fresh.set_option("frozen_core", 3)
    frz = _chain(fresh, N, NOCC, eps, ao=(eri, C))
    fresh.set_option("gemm_use_tma", 0)
    try:
        cp, _ = fresh.ccsd_t_spatial(True, False, True)
    finally:
        fresh.set_option("gemm_use_tma", 2)
    tma, _ = fresh.ccsd_t_spatial(True, False, True)
    assert _close(tma, frz["sums"]) and _close(cp, frz["sums"])
    # the work dealt to 3 ranks adds up to the whole
    parts = []
    for rank in range(3):
        fresh.set_partition(rank, 3)
        parts.append(fresh.ccsd_t_spatial(True, False, True)[0])
    fresh.set_partition(0, 1)
    assert _close(np.sum(parts, axis=0), frz["sums"])


SPATIAL = ["MP2_spatial", "CCSD_spatial", "CCSD(T)_spatial", "CCSD[T]_spatial", "RCCSD(T)_spatial", "RCCSD[T]_spatial",
           "CRCCSD(T)_spatial", "CRCCSD[T]_spatial"]
KEYS = ["e_ccsd_t", "e_ccsd_tt", "e_rccsd_t", "e_rccsd_tt", "e_crccsd_t", "e_crccsd_tt", "D_T", "D_TT"]


@pytest.mark.parametrize("calc", SPATIAL)
@pytest.mark.parametrize("k", [2, 1])
@pytest.mark.parametrize("name", ["n2", "f2"])
def test_spatial_calc_types_with_frozen_core_match_the_oracle(fresh, name, k, calc):
    from afesp_b200 import host

    r = fc.run(load_system(name, calc), k)
    inp = load_els_input(name, calc)
    inp.frozen_core = k
    res = host.run(inp, gpu=fresh)
    assert abs(res.e_mp2 - r["e_mp2"]) < E_TOL
    if "ccsd" not in r:
        return
    assert len(res.ccsd_table) == len(r["ccsd"])
    for (it, e, _, rms), (oit, oe, _, orms) in zip(res.ccsd_table, r["ccsd"]):
        assert it == oit and abs(e - oe) < E_TOL and abs(rms - orms) < 1e-9, (it, e, oe)
    assert abs(res.t1_diagnostic - r["t1_diag"]) < E_TOL
    for key in KEYS:
        assert (key in r) == (key in res.energies), key
        if key in r:
            assert abs(res.energies[key] - r[key]) < E_TOL, (key, res.energies[key], r[key])


def test_h2o_cc_pvtz_spinorbital_ccsd_t_with_one_frozen_orbital_matches_the_oracle(fresh):
    from afesp_b200 import host

    r = fc.run(load_system("h2o_tz", "CCSD(T)_spinorb"), 1)
    inp = load_els_input("h2o_tz", "CCSD(T)_spinorb")
    inp.frozen_core = 1
    res = host.run(inp, gpu=fresh)
    assert abs(res.e_mp2 - r["e_mp2"]) < E_TOL
    assert len(res.ccsd_table) == len(r["ccsd"])
    for (it, e, _, rms), (oit, oe, _, orms) in zip(res.ccsd_table, r["ccsd"]):
        assert it == oit and abs(e - oe) < E_TOL and abs(rms - orms) < 1e-9, (it, e, oe)
    assert abs(res.energies["e_ccsd_t"] - r["e_ccsd_t"]) < E_TOL


def test_sharded_chain_with_frozen_core_matches_replicated_on_two_gpus():
    import torch

    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    port = 29600 + (os.getpid() % 300) + 13
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "dist_check.py"), "--frozen-core", "3"]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["pass"] and line["ranks_bit_identical"] and line["frozen_core"] == 3, line
