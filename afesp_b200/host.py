"""Host side of the drop-in: a Python mirror of the reference's program flow (src/main.F90:36-175).

The reference's Fortran main program reads `els.in` and the `*.dat` files, runs RHF on the host, and then enters
the hot path.  This module plays that role above the C ABI so the path can be exercised without a Fortran compiler
(none exists in this image): same inputs, same calc_type strings, same convergence logic, same printed lines.
Everything from the AO->MO transform onwards runs on the GPU through include/afesp_gpu.h; the SCF (outside the
north-star path, SURVEY.md §2.1) is a small NumPy routine that follows src/hf.f90 step by step because CC energies
are first order in the residual SCF error.  Nothing here imports the test oracle.
"""
from __future__ import annotations

import io
import os
import re
import time
from dataclasses import dataclass, field

import numpy as np

from .capi import AfespError, AfespGpu

# calc_type -> (level, restricted, paren, renorm, comp_renorm)  (src/system.f90:116-165)
CALC_TYPES = {
    "RHF": (0, True, False, False, False),
    "UHF": (0, False, False, False, False),
    "MP2_spinorb": (1, False, False, False, False),
    "MP2_spatial": (1, True, False, False, False),
    "CCSD_spinorb": (2, False, False, False, False),
    "CCSD_spatial": (2, True, False, False, False),
    "CCSD(T)_spinorb": (3, False, False, False, False),
    "CCSD(T)_spatial": (3, True, True, False, False),
    "CCSD[T]_spatial": (3, True, False, False, False),
    "RCCSD(T)_spatial": (3, True, True, True, False),
    "RCCSD[T]_spatial": (3, True, False, True, False),
    "CRCCSD(T)_spatial": (3, True, True, False, True),
    "CRCCSD[T]_spatial": (3, True, False, False, True),
}


@dataclass
class ElsInput:
    """The &elsinput namelist (src/system.f90:96-97) plus the integral files."""

    calc_type: str = "CCSD(T)_spatial"
    scf_e_tol: float = 1e-6
    scf_d_tol: float = 1e-6
    scf_diis_n_errmat: int = 6
    ccsd_e_tol: float = 1e-6
    ccsd_t_tol: float = 1e-6
    ccsd_diis_n_errmat: int = 8
    scf_maxiter: int = 50
    ccsd_maxiter: int = 50
    write_fcidump: bool = False
    scf_read_guess: bool = False
    scf_write_guess: bool = False
    frozen_core: int = 0               # frozen doubly occupied orbitals (extension of the namelist; 0 = all-electron)
    nbasis: int = 0
    nel: int = 0
    e_nuc: float = 0.0
    ovlp: np.ndarray | None = None
    core_hamil: np.ndarray | None = None
    eri: np.ndarray | None = None      # packed AO ERIs, canonical order (src/integrals.f90:196-210)
    guess: np.ndarray | None = None    # guess_in.dat Fock matrix
    fock_final: np.ndarray | None = None  # AO Fock matrix of the converged SCF (guess_out.dat)
    els_in_text: str = ""              # els.in as read (echoed into the output, src/integrals.f90:240-249)


@dataclass
class ElsResult:
    e_hf: float = 0.0
    e_nuc: float = 0.0
    e_mp2: float = 0.0
    e_ccsd: float = 0.0
    energies: dict = field(default_factory=dict)
    scf_table: list = field(default_factory=list)
    ccsd_table: list = field(default_factory=list)
    ccsd_converged: bool = False
    t1_diagnostic: float = 0.0
    coeff: np.ndarray | None = None
    eps: np.ndarray | None = None
    timings: dict = field(default_factory=dict)
    stdout: str = ""


def pair_index(i, j):
    i = np.asarray(i, dtype=np.int64)
    j = np.asarray(j, dtype=np.int64)
    hi, lo = np.maximum(i, j), np.minimum(i, j)
    return hi * (hi + 1) // 2 + lo


NAMELIST_KEYS = {"calc_type": str, "scf_e_tol": float, "scf_d_tol": float, "ccsd_e_tol": float, "ccsd_t_tol": float,
                 "scf_diis_n_errmat": int, "ccsd_diis_n_errmat": int, "scf_maxiter": int, "ccsd_maxiter": int,
                 "write_fcidump": bool, "scf_read_guess": bool, "scf_write_guess": bool,   # src/system.f90:96-97
                 "frozen_core": int}


def parse_namelist(text):
    """`read(unit=ir, nml=elsinput)` of src/system.f90:105 with Fortran namelist rules: the group starts at `&elsinput` (any
    case) and ends at the first `/` outside a string; `!` starts a comment; assignments are separated by commas, blanks or
    line ends (several may share a line); names are case-insensitive; logicals are .true./.t./t... ; reals may carry a `d`
    exponent.  Anything the compiler's runtime would refuse (no group, unknown name, malformed value) raises the
    reference's error text (:107)."""
    def bad():
        return ValueError("system::read_system_in: invalid input file format!")

    # strip comments (outside quotes) and find the group
    body, quote = [], None
    for raw in text.splitlines():
        line = []
        for ch in raw:
            if quote:
                if ch == quote:
                    quote = None
            elif ch in "\"'":
                quote = ch
            elif ch == "!":
                break
            line.append(ch)
        body.append("".join(line))
    flat = "\n".join(body)
    m = re.search(r"&elsinput\b", flat, flags=re.I)
    if not m:
        raise bad()
    rest, out, pos = flat[m.end():], {}, 0
    tok = re.compile(r"\s*(?:,\s*)?(?:(/|&end\b)|([A-Za-z_]\w*)\s*=\s*(\"[^\"]*\"|'[^']*'|[^,\s/!]+))", flags=re.I)
    while True:
        t = tok.match(rest, pos)
        if not t:
            if rest[pos:].strip(" \t\r\n,") == "":
                raise bad()   # group never closed
            raise bad()
        pos = t.end()
        if t.group(1):
            break
        k, v = t.group(2).lower(), t.group(3)
        kind = NAMELIST_KEYS.get(k)
        if kind is None:
            raise bad()
        try:
            if kind is str:
                out[k] = v[1:-1] if v[:1] in "\"'" else v
                out[k] = out[k].strip()
            elif kind is bool:
                w = v.lower().lstrip(".")
                if w[:1] not in "tf":
                    raise bad()
                out[k] = w[0] == "t"
            elif kind is int:
                out[k] = int(v)
            else:
                out[k] = float(v.lower().replace("d", "e"))
        except ValueError:
            raise bad() from None
    return out


def _sym_from_triples(d, n):
    m = np.zeros((n, n))
    i, j = d[:, 0].astype(int) - 1, d[:, 1].astype(int) - 1
    m[i, j] = d[:, 2]
    m[j, i] = d[:, 2]
    return m


def read_inputs(dirpath) -> ElsInput:
    """read_system_in, read_integrals_in, read_geometry_in (src/system.f90:81, integrals.f90:48, geometry.f90:8)."""
    inp = ElsInput()
    with open(os.path.join(dirpath, "els.in")) as f:
        inp.els_in_text = f.read()
    for k, v in parse_namelist(inp.els_in_text).items():
        if hasattr(inp, k):
            setattr(inp, k, v)
    if inp.calc_type not in CALC_TYPES:
        raise ValueError("system::read_system_in: Unrecognised calculation type!")
    s = np.loadtxt(os.path.join(dirpath, "s.dat"), ndmin=2)
    n = int(max(s[:, 0].max(), s[:, 1].max()))
    inp.nbasis = n
    inp.ovlp = _sym_from_triples(s, n)
    inp.core_hamil = _sym_from_triples(np.loadtxt(os.path.join(dirpath, "t.dat"), ndmin=2), n) + \
        _sym_from_triples(np.loadtxt(os.path.join(dirpath, "v.dat"), ndmin=2), n)
    npair = n * (n + 1) // 2
    bin_path = os.path.join(dirpath, "eri.bin")
    if os.path.exists(bin_path):
        # extension for large basis sets (SURVEY.md section 8f-3): the packed array itself, little-endian float64
        inp.eri = np.fromfile(bin_path, dtype="<f8")
        if inp.eri.size != npair * (npair + 1) // 2:
            raise ValueError("integrals::read_integrals_in: eri.bin does not hold npair(npair+1)/2 doubles for this basis")
    elif os.path.exists(os.path.join(dirpath, "eri.dat")):
        d = np.loadtxt(os.path.join(dirpath, "eri.dat"), ndmin=2)
        idx = d[:, :4].astype(np.int64) - 1
        eri = np.zeros(npair * (npair + 1) // 2)
        eri[pair_index(pair_index(idx[:, 0], idx[:, 1]), pair_index(idx[:, 2], idx[:, 3]))] = d[:, 4]
        inp.eri = eri
    with open(os.path.join(dirpath, "geom.dat")) as f:
        toks = f.read().split()
    nat = int(toks[0])
    g = np.array(toks[1:1 + 4 * nat], dtype=float).reshape(nat, 4)
    if inp.eri is None:
        # extension (SURVEY.md section 8f-4): no eri.dat (the reference checkout ships none for sample_data/h2o-cc-pvtz).  With
        # the basis set named -- one-line file basis.dat, or AFESP_BASIS -- the integrals are generated from geom.dat
        # (afesp_b200/gint.py, Psi4 conventions) and must reproduce the overlap matrix of s.dat.
        basis = None
        if os.path.exists(os.path.join(dirpath, "basis.dat")):
            basis = open(os.path.join(dirpath, "basis.dat")).read().split()[0]
        basis = basis or os.environ.get("AFESP_BASIS")
        if not basis:
            raise FileNotFoundError("integrals::read_integrals_in: cannot open eri.dat")
        from . import gint

        res = gint.compute(g[:, 0], g[:, 1:], basis)
        if res["nbf"] != n or np.max(np.abs(res["s"] - inp.ovlp)) > 1e-10:
            raise ValueError(f"integrals::read_integrals_in: generated overlap matrix differs from s.dat (basis set {basis}?)")
        inp.eri = res["eri"]
    set_geometry(inp, g[:, 0], g[:, 1:])
    if inp.scf_read_guess:
        inp.guess = read_scf_guess(os.path.join(dirpath, "guess_in.dat"), n)
    return inp


def set_geometry(inp: ElsInput, charges, xyz):
    z = np.asarray(charges).astype(int)  # charges(i) = int(charge)  (src/geometry.f90:33)
    xyz = np.asarray(xyz, dtype=float)
    inp.nel = int(z.sum())
    e = 0.0
    for j in range(1, len(z)):
        for i in range(j):
            e += z[i] * z[j] / np.linalg.norm(xyz[i] - xyz[j])
    inp.e_nuc = e


def check_frozen_core(inp: ElsInput):
    """frozen_core must leave at least one doubly occupied orbital active (same text as host/els_host.cpp)."""
    nocc = inp.nel // 2
    if not 0 <= inp.frozen_core < nocc:
        raise ValueError("system::read_system_in: frozen_core = %d is outside 0..%d (nocc - 1)!" % (inp.frozen_core, nocc - 1))


def _unpack(packed, n):
    r = np.arange(n)
    ij = pair_index(r[:, None], r[None, :])
    return packed[pair_index(ij[:, :, None, None], ij[None, None, :, :])]


def rhf(inp: ElsInput, out=None):
    """do_rhf (src/hf.f90:21-151) with Pulay DIIS (:197-242); returns (e_elec, C[mo,ao], eps, table, converged).
    The AO Fock matrix of the last diagonalisation (what write_out_scf_guess stores, :131-134) is left in
    inp.fock_final."""
    n, nocc = inp.nbasis, inp.nel // 2
    S, h = inp.ovlp, inp.core_hamil
    g = _unpack(inp.eri, n)
    J_src = g                      # (ij|kl)
    K_src = g.transpose(0, 2, 1, 3)  # (ik|jl) viewed as [i,j,k,l]
    w, U = np.linalg.eigh(S)
    X = U @ np.diag(1.0 / np.sqrt(w)) @ U.T
    F = inp.guess.copy() if (inp.scf_read_guess and inp.guess is not None) else h.copy()
    nerr = inp.scf_diis_n_errmat
    use_diis = nerr >= 2
    Fs = np.zeros((max(nerr, 1), n, n))
    Es = np.zeros((max(nerr, 1), n, n))
    slot = n_active = 0
    energy, D_old = 0.0, np.zeros((n, n))
    table, conv = [], False
    C_mo = eps = None
    if out is not None:
        if inp.scf_read_guess and inp.guess is not None:
            out.write(" Reading previous AO Fock matrix as guess...\n")
        out.write("-" * 75 + "\n Iteration        Energy           deltaE           delta RMS D      Time  \n" + "-" * 75 + "\n")
    t0 = time.perf_counter()
    for it in range(1, inp.scf_maxiter + 1):
        eps, Cp = np.linalg.eigh(X.T @ F @ X)
        inp.fock_final = F.copy()
        C_mo = (X @ Cp).T
        D = C_mo[:nocc].T @ C_mo[:nocc]
        e_old, energy = energy, float(np.sum(D * (h + F)))
        rms = float(np.sqrt(np.sum((D - D_old) ** 2)))
        conv = rms < inp.scf_d_tol and abs(energy - e_old) < inp.scf_e_tol
        D_old = D
        t1 = time.perf_counter()
        table.append((it, energy, energy - e_old, rms))
        if out is not None:
            out.write(" %9d   %15.10f   %15.10f   %15.10f   %8.6f\n" % (it, energy, energy - e_old, rms, t1 - t0))
        t0 = t1
        if conv:
            if out is not None:   # src/hf.f90:115-122
                out.write("-" * 75 + "\n Convergence reached within tolerance.\n")
                out.write(" Final SCF Energy (Hartree): %15.8f\n" % energy)
                out.write(" Orbital energies (Hartree):\n")
                for i in range(n, 0, -1):
                    out.write(" %3d %15.8f\n" % (i, eps[i - 1]))
            break
        F = h + 2.0 * np.einsum("ijkl,kl->ij", J_src, D) - np.einsum("ijkl,kl->ij", K_src, D)
        if use_diis:
            slot = slot + 1 if slot < nerr else 1
            n_active = min(n_active + 1, nerr)
            Fs[slot - 1] = F
            Es[slot - 1] = F @ D @ S - S @ D @ F
            na = n_active
            if na > 1:
                B = np.zeros((na + 1, na + 1))
                for i in range(na):
                    for j in range(i + 1):
                        B[i, j] = B[j, i] = np.sum(Es[i] * Es[j])
                B[na, :na] = B[:na, na] = -1.0
                rhs = np.zeros(na + 1)
                rhs[na] = -1.0
                c = np.linalg.solve(B, rhs)
                F = np.tensordot(c[:na], Fs[:na], axes=(0, 0))
    return energy, C_mo, eps, table, conv


def _es(x, width, digits):
    """Fortran ESw.d edit descriptor (one non-zero digit before the point, two-digit exponent)."""
    return ("%" + str(width) + "." + str(digits) + "E") % x


def write_scf_guess(path, fock):
    """write_out_scf_guess (src/hf.f90:172-191): every (i, j, F_ij), format (I0, 1X, I0, 1X, ES16.9)."""
    n = fock.shape[0]
    with open(path, "w") as f:
        for i in range(n):
            for j in range(n):
                f.write("%d %d %s\n" % (i + 1, j + 1, _es(fock[i, j], 16, 9)))


def read_scf_guess(path, n):
    """read_in_scf_guess (src/hf.f90:153-170): free-format (i, j, value) triples."""
    gd = np.loadtxt(path, ndmin=2)
    g = np.zeros((n, n))
    g[gd[:, 0].astype(int) - 1, gd[:, 1].astype(int) - 1] = gd[:, 2]
    return g


def fcidump_indices(n):
    """(p, q, r, s), 1-based, of every packed MO integral in the reference's canonical loop order
    (src/mp2.f90:466-479: p, q<=p, r<=p, s<=(q if r==p else r)) -- the same order as the packed array."""
    P, Q, R, S = [], [], [], []
    for p in range(1, n + 1):
        for q in range(1, p + 1):
            for r in range(1, p + 1):
                s_up = q if r == p else r
                cnt = s_up
                P.append(np.full(cnt, p)); Q.append(np.full(cnt, q)); R.append(np.full(cnt, r))
                S.append(np.arange(1, s_up + 1))
    return tuple(np.concatenate(a) for a in (P, Q, R, S))


def write_fcidump(path, eri_mo_packed, n):
    """write_fcidump (src/mp2.f90:451-487): one line per packed MO integral with |v| > 1e-7,
    format (I3,I3,I3,I3,ES17.9), canonical order, no header (as the reference writes it)."""
    p, q, r, s = fcidump_indices(n)
    v = np.asarray(eri_mo_packed)
    assert v.size == p.size, (v.size, p.size)
    keep = np.abs(v) > np.float32(1e-7)   # the reference compares against a default-real literal
    with open(path, "w") as f:
        for a, b, c, d, x in zip(p[keep], q[keep], r[keep], s[keep], v[keep]):
            f.write("%3d%3d%3d%3d%s\n" % (a, b, c, d, _es(x, 17, 9)))
    return int(keep.sum())


def assemble_triples(e_ccsd, sums, const, paren, renorm, comp_renorm):
    """Energy assembly of do_ccsd_t_spatial (src/ccsd.f90:2239-2276)."""
    e_T, e_TT, D_T, D_TT, e_CR, e_CRT = [float(x) for x in sums]
    en = {}
    if renorm or comp_renorm:
        D_T += const
        if paren:
            D_TT += const
    en["e_ccsd_t"] = e_ccsd + e_T
    if paren:
        en["e_ccsd_tt"] = e_ccsd + e_TT
    if renorm or comp_renorm:
        en["e_rccsd_t"] = e_ccsd + e_T / D_T
        en["D_T"] = D_T
        if paren:
            en["e_rccsd_tt"] = e_ccsd + e_TT / D_TT
        if comp_renorm:
            en["e_crccsd_t"] = e_ccsd + e_CR / D_T
            en["D_TT"] = D_TT
            if paren:
                en["e_crccsd_tt"] = e_ccsd + e_CRT / D_TT
    return en


def ccsd_loop(gpu: AfespGpu, nocc, restricted, eps, e_tol, t_tol, diis_n, maxiter, out=None):
    """The iteration loop of do_ccsd_spatial / do_ccsd_spinorb (src/ccsd.f90:339-396 / 229-271) on the host side:
    the GPU does one iteration per call, the host keeps the table, the convergence test (:1805) and the DIIS call."""
    t_init = time.perf_counter()
    try:
        e, rms = gpu.ccsd_init(nocc, restricted, eps, diis_n)
    except AfespError as ex:
        if ex.code == 5 and out is not None:   # the reference's assertion on <pq||rs> fired (src/ccsd.f90:161-164)
            info = gpu.ccsd_init_info()
            out.write(" Forming antisymmetrised spinorbital ERIs...\n Time taken: %8.6f s\n\n" % info["slices_s"])
            out.write(" Checking that the permuational symmetry of the antisymmetrised integrals hold...\n")
            out.write(" Permutational symmetry error: %s\n" % _e_f(info["symmetry_error"], 15, 6))   # E15.6, :165
        raise
    table = [("MP1", e, e - 0.0, rms)]
    if out is not None:
        if restricted:   # src/ccsd.f90:312-324 with the prints of init_cc (:427-526)
            out.write(" Initialise CC intermediate tensors and DIIS auxilliary arrays...\n"
                      " Forming energy denominator matrices...\n Allocating amplitude tensors...\n"
                      " Forming ERI slices...\n Forming initial amplitude guesses...\n"
                      " Allocating stored intermediate tensors...\n")
        else:            # src/ccsd.f90:106-220.  The (2n)^4 tensor is never formed here: the nine slices are gathered
            # straight from the packed MO integrals (first timer), the reference's symmetry assertion runs on the device
            # over the same index set (second timer), and nothing is left to do for the third banner.
            info = gpu.ccsd_init_info()
            out.write(" Forming antisymmetrised spinorbital ERIs...\n Time taken: %8.6f s\n\n" % info["slices_s"])
            out.write(" Checking that the permuational symmetry of the antisymmetrised integrals hold...\n"
                      " Time taken: %8.6f s\n\n" % info["check_s"])
            out.write(" Forming slices of antisymmetrised spinorbital ERIs\n Time taken: %8.6f s\n\n" % 0.0)
            out.write(" Initialise CC intermediate tensors and DIIS auxilliary arrays...\n"
                      " Forming energy denominator matrices...\n Allocating amplitude tensors...\n"
                      " Forming ERI slices...\n Forming initial amplitude guesses...\n"
                      " Allocating stored intermediate tensors...\n")
        out.write(" Time taken: %8.6f s\n\n" % (time.perf_counter() - t_init))
        out.write(" Initialisation done, now entering iterative CC solver...\n")
        out.write("-" * 75 + "\n Iteration        Energy           deltaE          delta RMS T2      Time  \n" + "-" * 75 + "\n")
        out.write(" %9s   %15.12f   %15.12f   %15.12f\n" % ("MP1", e, e, rms))
    conv = False
    e_old = e
    ms = []
    for it in range(1, maxiter + 1):
        t0 = time.perf_counter()
        e, rms = gpu.ccsd_iterate()
        ms.append(gpu.last_stage_ms())
        table.append((it, e, e - e_old, rms))
        if out is not None:
            out.write(" %9d   %15.12f   %15.12f   %15.12f   %8.6f\n" % (it, e, e - e_old, rms, time.perf_counter() - t0))
        if np.sqrt(rms) < t_tol and abs(e - e_old) < e_tol:
            conv = True
            break
        e_old = e
        gpu.ccsd_diis()
    return table, conv, e, ms


def run(inp: ElsInput, gpu: AfespGpu | None = None, device: int = 0, verbose: bool = False,
        workdir: str | None = None) -> ElsResult:
    """Whole program (src/main.F90): RHF on the host, everything from do_mp2_spatial onwards on the GPU.
    With `workdir` the files the reference writes into its run directory are written there too: guess_out.dat
    (scf_write_guess) and FCIDUMP (write_fcidump)."""
    level, restricted, paren, renorm, comp_renorm = CALC_TYPES[inp.calc_type]
    check_frozen_core(inp)
    out = io.StringIO()
    res = ElsResult(e_nuc=inp.e_nuc)
    t_glob = time.perf_counter()
    out.write(header_block(inp))
    out.write(_taken("system initialisation", time.perf_counter() - t_glob))
    t0 = time.perf_counter()
    out.write(" " + "-" * 23 + "\n Restricted Hartree-Fock\n " + "-" * 23 + "\n")
    res.e_hf, C_mo, eps, res.scf_table, conv = rhf(inp, out)
    res.coeff, res.eps = C_mo, eps
    res.timings["rhf_s"] = time.perf_counter() - t0
    if not conv:
        out.write(" Convergence not reached, please increase maxiter.\n")
    elif inp.scf_write_guess:
        out.write(" Writing AO Fock matrix for future use...\n")
        if workdir is not None:
            write_scf_guess(os.path.join(workdir, "guess_out.dat"), inp.fock_final)
    out.write(_taken("restricted Hartree-Fock", res.timings["rhf_s"]))
    if level >= 1:
        own = gpu is None
        gpu = gpu or AfespGpu(device)
        try:
            nocc = inp.nel // 2
            if inp.frozen_core > 0:   # MP2, CCSD and the triples correlate orbitals frozen_core.. only
                gpu.set_option("frozen_core", inp.frozen_core)
            t0 = time.perf_counter()
            out.write(" ----------\n MP2\n ----------\n Performing AO to MO ERI transformation...\n")
            gpu.ao2mo(inp.nbasis, inp.eri, C_mo, want_result=False)
            res.timings["ao2mo_device_ms"] = gpu.last_stage_ms()
            out.write(" Calculating MP2 energy...\n")
            res.e_mp2 = gpu.mp2_energy(nocc, eps)
            out.write(" MP2 correlation energy (Hartree): %15.8f\n" % res.e_mp2)
            if inp.write_fcidump:
                out.write(" Writing FCIDUMP file...\n")
                if workdir is not None:
                    write_fcidump(os.path.join(workdir, "FCIDUMP"), gpu.get_eri_mo(), inp.nbasis)
                out.write(" Done writing FCIDUMP file!\n")
            res.timings["mp2_s"] = time.perf_counter() - t0
            out.write(_taken("restricted MP2", res.timings["mp2_s"]))
            if level >= 2:
                t0 = time.perf_counter()
                out.write(" ----------\n CCSD\n ----------\n")
                res.ccsd_table, res.ccsd_converged, res.e_ccsd, ms = ccsd_loop(
                    gpu, nocc, restricted, eps, inp.ccsd_e_tol, inp.ccsd_t_tol, inp.ccsd_diis_n_errmat,
                    inp.ccsd_maxiter, out)
                res.timings["ccsd_iter_device_ms"] = ms
                if res.ccsd_converged:
                    out.write("-" * 75 + "\n Convergence reached within tolerance.\n")
                    out.write(" Final CCSD Energy (Hartree): %15.12f\n" % res.e_ccsd)
                res.t1_diagnostic, _, _ = gpu.ccsd_finalize(want_cr=comp_renorm)
                res.timings["ccsd_s"] = time.perf_counter() - t0
                if restricted and res.ccsd_converged:
                    out.write(" T1 diagnostic: %8.5f\n" % res.t1_diagnostic)
                    if res.t1_diagnostic > 0.02:   # src/ccsd.f90:374-376
                        out.write(" Significant multireference character detected, CCSD result might be unreliable!\n")
                out.write(_taken("restricted CCSD" if restricted else "unrestricted CCSD", res.timings["ccsd_s"]))
                if level >= 3 and res.ccsd_converged:
                    t0 = time.perf_counter()
                    out.write(" ----------\n CCSD(T)\n ----------\n")
                    if restricted:
                        sums, const = gpu.ccsd_t_spatial(paren, renorm, comp_renorm)
                        res.energies = assemble_triples(res.e_ccsd, sums, const, paren, renorm, comp_renorm)
                        res.energies["triples_sums"] = sums
                        name = triples_calcname(paren, renorm, comp_renorm)
                        out.write(" Restricted %s correlation energy (Hartree): %15.9f\n" % (
                            name, highest_energy(res.energies, paren, renorm, comp_renorm)))
                    else:
                        res.energies = {"e_ccsd_t": res.e_ccsd + gpu.ccsd_t_spinorb()}
                        name = "CCSD(T)"
                        out.write(" Unrestricted CCSD(T) correlation energy (Hartree): %15.9f\n" % res.energies["e_ccsd_t"])
                    res.timings["triples_device_ms"] = gpu.last_stage_ms()
                    res.timings["triples_s"] = time.perf_counter() - t0
                    out.write(_taken(("restricted " if restricted else "unrestricted ") + name, res.timings["triples_s"]))
        except AfespError as ex:
            ex.stdout = out.getvalue()   # what els.out held when the reference would have stopped (error -> stop 999)
            raise
        finally:
            if own:
                gpu.close()
    out.write(final_table(inp, res))
    now = time.localtime()
    out.write(" " + "=" * 64 + "\n Finished running on %02d/%02d/%04d at %02d:%02d:%02d\n" % (
        now.tm_mday, now.tm_mon, now.tm_year, now.tm_hour, now.tm_min, now.tm_sec))
    out.write(" Total execution time: %16.8f\n" % (time.perf_counter() - t_glob))   # src/main.F90:185
    res.stdout = out.getvalue()
    if verbose:
        print(res.stdout)
    return res


def highest_energy(en, paren, renorm, comp_renorm):
    """sys%e_highest after do_ccsd_t_spatial (src/ccsd.f90:2252-2276): the last energy assigned."""
    key = "e_ccsd_tt" if paren else "e_ccsd_t"
    if renorm or comp_renorm:
        key = "e_rccsd_tt" if paren else "e_rccsd_t"
        if comp_renorm:
            key = "e_crccsd_tt" if paren else "e_crccsd_t"
    return en[key]


def _e_f(x, width, digits):
    """Fortran Ew.d: mantissa in [0.1, 1), e.g. E15.6 of 3.5e-7 is '   0.350000E-06' (C's %E would print 3.500000E-07)."""
    if x == 0.0 or not np.isfinite(x):
        mant, ex = (0.0 if x == 0.0 else x), 0
    else:
        ex = int(np.floor(np.log10(abs(x)))) + 1
        mant = x / 10.0 ** ex
        if abs(float("%.*f" % (digits, mant))) >= 1.0:   # rounding carried into the leading digit
            ex += 1
            mant = x / 10.0 ** ex
    return ("%.*fE%+03d" % (digits, mant, ex)).rjust(width)


def _es_f(x, width, digits):
    """Fortran ESw.d for the system-information block (two-digit exponent)."""
    return ("%" + str(width) + "." + str(digits) + "E") % x


def header_block(inp: ElsInput, when=None) -> str:
    """Program banner, integral read-in log, system information and the echo of els.in
    (src/main.F90:26-32, src/integrals.f90:75-163, 223-249), byte for byte apart from the date."""
    when = when or time.localtime()
    if CALC_TYPES[inp.calc_type][1]:   # src/geometry.f90:40-46: spatial orbitals when restricted, spin-orbitals otherwise
        nocc_print, nvirt_print = inp.nel // 2, inp.nbasis - inp.nel // 2
    else:
        nocc_print, nvirt_print = inp.nel, (inp.nbasis - inp.nel // 2) * 2
    L = [" " + "=" * 64, " A Fortran Electronic Structure Programme (AFESP)", " " + "=" * 64,
         " Started running on %02d/%02d/%04d at %02d:%02d:%02d" % (when.tm_mday, when.tm_mon, when.tm_year, when.tm_hour,
                                                                    when.tm_min, when.tm_sec),
         " " + "-" * 16, " Integral read-in", " " + "-" * 16,
         " Getting number of basis functions...", " Allocating integral store...", " Reading overlap matrix...",
         " Reading kinetic integrals...", " Reading nuclear-electron integrals...", " Constructing core Hamiltonian...",
         " Reading two-body integrals...", " Done reading integrals!",
         " " + "-" * 20, " System information", " " + "-" * 20,
         " Number of electrons: %d" % inp.nel, " Number of basis functions: %d" % inp.nbasis,
         " Number of occupied orbitals: %d" % nocc_print, " Number of virtual orbitals: %d" % nvirt_print]
    if inp.frozen_core > 0:
        L.append(" Number of frozen core orbitals: %d" % inp.frozen_core)
    L += [" E_nuc: " + _es_f(inp.e_nuc, 15, 8),
         " scf_e_tol: " + _es_f(inp.scf_e_tol, 8, 2), " scf_d_tol: " + _es_f(inp.scf_d_tol, 8, 2),
         " ccsd_e_tol: " + _es_f(inp.ccsd_e_tol, 8, 2), " ccsd_t_tol: " + _es_f(inp.ccsd_t_tol, 8, 2),
         " Number of SCF DIIS error matrices: %d" % inp.scf_diis_n_errmat,
         " Number of CCSD DIIS error matrices: %d" % inp.ccsd_diis_n_errmat,
         " Maximum number of SCF iterations: %d" % inp.scf_maxiter,
         " Maximum number of CCSD iterations: %d" % inp.ccsd_maxiter,
         " Printing out the input file...", "-" * 30]
    L += [ln.rstrip() for ln in inp.els_in_text.splitlines()]
    L.append("-" * 30)
    return "\n".join(L) + "\n"


def _taken(label, seconds):
    """'(1X, A, 1X, F16.8, A)' of src/main.F90:43-115 (the shipped N2/F2 logs predate it and print F7.4)."""
    return " Time taken for %s: %16.8fs\n" % (label, seconds)


def triples_calcname(paren, renorm, comp_renorm):
    """calcname of src/ccsd.f90:2278-2287."""
    name = "CCSD(T)" if paren else "CCSD[T]"
    if renorm:
        name = "renormalised " + name
    if comp_renorm:
        name = "completely renormalised " + name
    return name


def final_table(inp: ElsInput, r: ElsResult) -> str:
    """The 'Final energy breakdown' block, labels byte-identical to src/main.F90:123-175 (parsed by els_wrapper.py)."""
    level, restricted, paren, renorm, comp_renorm = CALC_TYPES[inp.calc_type]
    base = r.e_hf + r.e_nuc
    L = [" " + "=" * 64, " Final energy breakdown", " %-31s %15.10f" % ("RHF energy:", base)]

    def two(label, corr):
        L.append(" %-31s %15.10f" % (label + " correlation energy:", corr))
        L.append(" %-31s %15.10f" % (label + " energy:", corr + base))

    highest = 0.0
    if level >= 1:
        two("MP2", r.e_mp2)
        highest = r.e_mp2
    if level >= 2:
        two("CCSD", r.e_ccsd)
        highest = r.e_ccsd
    en = r.energies
    if level >= 3 and en:
        if restricted:
            two("CCSD[T]", en["e_ccsd_t"]); highest = en["e_ccsd_t"]
            if paren:
                two("CCSD(T)", en["e_ccsd_tt"]); highest = en["e_ccsd_tt"]
            if renorm or comp_renorm:
                two("R-CCSD[T]", en["e_rccsd_t"]); highest = en["e_rccsd_t"]
                if paren:
                    two("R-CCSD(T)", en["e_rccsd_tt"]); highest = en["e_rccsd_tt"]
                if comp_renorm:
                    two("CR-CCSD[T]", en["e_crccsd_t"]); highest = en["e_crccsd_t"]
                    if paren:
                        two("CR-CCSD(T)", en["e_crccsd_tt"]); highest = en["e_crccsd_tt"]
        else:
            two("CCSD(T)", en["e_ccsd_t"]); highest = en["e_ccsd_t"]
    if level >= 2 and restricted:
        L.append(" " + "-" * 47)
        L.append(" %-31s %15.10f" % ("T1 diagnostic:", r.t1_diagnostic))
    if (renorm or comp_renorm) and en:
        L.append(" %-31s %15.10f" % ("D[T]:", en["D_T"]))
        if paren:  # sys%D_TT is only set for the CR methods and prints as zero otherwise (src/ccsd.f90:2262-2266)
            L.append(" %-31s %15.10f" % ("D(T):", en.get("D_TT", 0.0)))
    L.append(" " + "-" * 47)
    L.append(" %-31s %15.10f" % ("Total electronic energy:", r.e_hf + highest))
    L.append(" %-31s %15.10f" % ("Nuclear repulsion:", r.e_nuc))
    L.append(" %-31s %15.10f" % ("Total energy:", r.e_hf + highest + r.e_nuc))
    return "\n".join(L) + "\n"
