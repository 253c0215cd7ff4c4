"""ctypes bindings of include/afesp_gpu.h (one class method per exported function)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libafesp_gpu.so")

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_H = C.c_void_p

# name -> (argtypes) ; every function returns int except last_error
SIGNATURES = {
    "afesp_gpu_open": [C.c_int, C.POINTER(_H)],
    "afesp_gpu_close": [_H],
    "afesp_gpu_set_option": [_H, C.c_char_p, C.c_double],
    "afesp_gpu_counters": [_H, C.POINTER(C.c_longlong), _dp],
    "afesp_gpu_ao2mo": [_H, C.c_int, _dp, _dp, _dp],
    "afesp_gpu_set_eri_mo": [_H, C.c_int, _dp],
    "afesp_gpu_synth_eri_ao": [_H, C.c_int, C.c_int, _dp, _dp],
    "afesp_gpu_get_eri_mo": [_H, _dp],
    "afesp_gpu_release": [_H, C.c_char_p],
    "afesp_gpu_mp2_energy": [_H, C.c_int, _dp, _dp],
    "afesp_gpu_ccsd_init": [_H, C.c_int, C.c_int, _dp, C.c_int, _dp, _dp],
    "afesp_gpu_ccsd_init_info": [_H, _dp],
    "afesp_gpu_ccsd_iterate": [_H, _dp, _dp],
    "afesp_gpu_ccsd_diis": [_H],
    "afesp_gpu_ccsd_finalize": [_H, C.c_int, _dp, _dp, _dp],
    "afesp_gpu_ccsd_t_spatial": [_H, C.c_int, C.c_int, C.c_int, _dp, _dp],
    "afesp_gpu_ccsd_t_spinorb": [_H, _dp],
    "afesp_gpu_comm_unique_id": [C.c_char_p],
    "afesp_gpu_comm_init": [_H, C.c_int, C.c_int, C.c_char_p],
    "afesp_gpu_set_partition": [_H, C.c_int, C.c_int],
    "afesp_gpu_host_register": [C.c_void_p, C.c_longlong],
    "afesp_gpu_host_unregister": [C.c_void_p],
    "afesp_gpu_triples_partition": [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_longlong)],
    "afesp_gpu_column_partition": [C.c_longlong, C.c_int, C.c_int, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)],
    "afesp_gpu_dgemm_wrapper": [_H, C.c_char, C.c_char, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, C.c_double, C.c_double],
    "afesp_gpu_omp_reshape": [_H, _dp, _dp, _ip, C.c_char_p, C.c_int, C.c_double],
    "afesp_gpu_bench_dgemm": [_H, C.c_char, C.c_char, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, _dp],
    "afesp_gpu_dmma_peak": [_H, _dp],
    "afesp_gpu_last_stage_ms": [_H, _dp],
    "afesp_gpu_timer": [_H, C.c_int, _dp],
    "afesp_gpu_tma_status": [_H, C.POINTER(C.c_int), C.POINTER(C.c_int)],
    "afesp_gpu_bench_hbm": [_H, C.c_char_p, C.c_int, C.c_int, C.c_int, _dp, _dp],
    "afesp_gpu_gemm_time": [_H, _dp, _dp],
    "afesp_gpu_gemm_stats": [_H, _dp, _dp, C.POINTER(C.c_longlong)],
    "afesp_gpu_gemm_crosscheck": [_H, C.c_char, C.c_char, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int,
                                  C.POINTER(C.c_longlong), _dp, _dp],
}

_lib = None


class AfespError(RuntimeError):
    def __init__(self, fn, code, msg):
        super().__init__(f"afesp_gpu::{fn} failed (status {code}): {msg}")
        self.code = code


def load_library(path: str | None = None):
    """dlopen the engine.  Raises if the library has not been built -- there is no fallback."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise FileNotFoundError(f"{p} not built; run `python -c 'import __graft_entry__ as g; g.build()'` or make -C afesp_b200/csrc")
    lib = C.CDLL(p, mode=C.RTLD_GLOBAL)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    lib.afesp_gpu_last_error.argtypes = [_H]
    lib.afesp_gpu_last_error.restype = C.c_char_p
    if path is None:
        _lib = lib
    return lib


def _f64(a, writable=False):
    a = np.asarray(a, dtype=np.float64)
    if not a.flags.f_contiguous and not a.flags.c_contiguous:
        a = np.asfortranarray(a)
    return a


def _ptr(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def fortran_flat(a):
    """Column-major flattening of an array given in the reference's index order."""
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64).ravel(order="F"))


class AfespGpu:
    """One handle = one CUDA device (include/afesp_gpu.h)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        self.h = _H()
        rc = self.lib.afesp_gpu_open(int(device), C.byref(self.h))
        if rc != 0:
            raise AfespError("open", rc, self.lib.afesp_gpu_last_error(None).decode())
        self.n = 0
        self.o = 0
        self.v = 0
        self.frozen_core = 0   # option "frozen_core" as last set; ccsd_init sizes the amplitudes from it

    # -- plumbing
    def _check(self, fn, rc):
        if rc != 0:
            raise AfespError(fn, rc, self.lib.afesp_gpu_last_error(self.h).decode())

    def close(self):
        if self.h:
            self.lib.afesp_gpu_close(self.h)
            self.h = _H()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, key, value):
        self._check("set_option", self.lib.afesp_gpu_set_option(self.h, key.encode(), float(value)))
        if key == "frozen_core":
            self.frozen_core = int(value)

    def counters(self):
        n = C.c_longlong(0)
        f = C.c_double(0)
        self._check("counters", self.lib.afesp_gpu_counters(self.h, C.byref(n), C.byref(f)))
        return n.value, f.value

    def last_stage_ms(self):
        ms = C.c_double(0)
        self._check("last_stage_ms", self.lib.afesp_gpu_last_stage_ms(self.h, C.byref(ms)))
        return ms.value

    # -- AO->MO + MP2
    def ao2mo(self, nbasis, eri_ao=None, coeff=None, want_result=True):
        """coeff is C[mo, ao] in index order; it is passed column-major as the Fortran host would."""
        nbasis = int(nbasis)
        npk = (nbasis * (nbasis + 1) // 2) * (nbasis * (nbasis + 1) // 2 + 1) // 2
        out = np.empty(npk) if want_result else None
        if eri_ao is None:
            rc = self.lib.afesp_gpu_ao2mo(self.h, nbasis, None, None, _ptr(out))
        else:
            e = np.ascontiguousarray(eri_ao, dtype=np.float64)
            assert e.size == npk, (e.size, npk)
            c = fortran_flat(coeff)
            rc = self.lib.afesp_gpu_ao2mo(self.h, nbasis, _ptr(e), _ptr(c), _ptr(out))
        self._check("ao2mo", rc)
        self.n = nbasis
        return out

    def synth_eri_ao(self, nbasis, factors, coeff):
        """factors: (npair, naux) array in pair order; the packed AO integrals are built on the device."""
        f = fortran_flat(factors)
        c = fortran_flat(coeff)
        self._check("synth_eri_ao", self.lib.afesp_gpu_synth_eri_ao(self.h, int(nbasis), int(factors.shape[1]),
                                                                    _ptr(f), _ptr(c)))
        self.n = int(nbasis)

    def get_eri_mo(self, out=None):
        npair = self.n * (self.n + 1) // 2
        if out is None:
            out = np.empty(npair * (npair + 1) // 2)
        self._check("get_eri_mo", self.lib.afesp_gpu_get_eri_mo(self.h, _ptr(out)))
        return out

    def release(self, what):
        self._check("release", self.lib.afesp_gpu_release(self.h, what.encode()))

    def set_eri_mo(self, nbasis, eri_mo):
        """eri_mo may be None on ranks > 0 of a communicator: they receive rank 0's copy over NVLink."""
        e = None if eri_mo is None else np.ascontiguousarray(eri_mo, dtype=np.float64)
        self._check("set_eri_mo", self.lib.afesp_gpu_set_eri_mo(self.h, int(nbasis), _ptr(e)))
        self.n = int(nbasis)

    def mp2_energy(self, nocc, eps):
        e = np.ascontiguousarray(eps, dtype=np.float64)
        out = C.c_double(0)
        self._check("mp2_energy", self.lib.afesp_gpu_mp2_energy(self.h, int(nocc), _ptr(e), C.byref(out)))
        return out.value

    # -- CCSD
    def ccsd_init(self, nocc, restricted, eps, diis_n=8):
        e = np.ascontiguousarray(eps, dtype=np.float64)
        e1, r = C.c_double(0), C.c_double(0)
        self._check("ccsd_init", self.lib.afesp_gpu_ccsd_init(self.h, int(nocc), int(bool(restricted)), _ptr(e),
                                                              int(diis_n), C.byref(e1), C.byref(r)))
        nact = int(nocc) - self.frozen_core   # t1 / t2 cover the active occupied orbitals only
        if restricted:
            self.o, self.v = nact, self.n - int(nocc)
        else:
            self.o, self.v = 2 * nact, 2 * (self.n - int(nocc))
        return e1.value, r.value

    def ccsd_init_info(self):
        """Spin-orbital integral preparation of the last ccsd_init (src/ccsd.f90:106-202): dict with the error of the
        permutational-symmetry self-check and the device seconds of the slice gather and of the check."""
        info = (C.c_double * 4)()
        self._check("ccsd_init_info", self.lib.afesp_gpu_ccsd_init_info(self.h, info))
        return {"symmetry_error": info[0], "slices_s": info[1], "check_s": info[2]}

    def ccsd_iterate(self):
        e, r = C.c_double(0), C.c_double(0)
        self._check("ccsd_iterate", self.lib.afesp_gpu_ccsd_iterate(self.h, C.byref(e), C.byref(r)))
        return e.value, r.value

    def ccsd_diis(self):
        self._check("ccsd_diis", self.lib.afesp_gpu_ccsd_diis(self.h))

    def ccsd_finalize(self, want_cr=False, want_amplitudes=False, out=None):
        """out = (t1_buffer, t2_buffer): caller-provided flat float64 arrays (e.g. pinned host memory) for the amplitudes."""
        d = C.c_double(0)
        t1 = t2 = None
        if out is not None:
            t1, t2 = out
            want_amplitudes = True
            assert t1.size == self.o * self.v and t2.size == self.o * self.o * self.v * self.v
        elif want_amplitudes:
            t1 = np.empty(self.o * self.v)
            t2 = np.empty(self.o * self.o * self.v * self.v)
        self._check("ccsd_finalize", self.lib.afesp_gpu_ccsd_finalize(self.h, int(bool(want_cr)), C.byref(d),
                                                                      _ptr(t1), _ptr(t2)))
        if want_amplitudes:
            t1 = t1.reshape((self.o, self.v), order="F")
            t2 = t2.reshape((self.o, self.o, self.v, self.v), order="F")
        return d.value, t1, t2

    # -- triples
    def ccsd_t_spatial(self, paren, renorm, comp_renorm):
        sums = np.zeros(6)
        c = C.c_double(0)
        self._check("ccsd_t_spatial", self.lib.afesp_gpu_ccsd_t_spatial(self.h, int(bool(paren)), int(bool(renorm)),
                                                                        int(bool(comp_renorm)), _ptr(sums), C.byref(c)))
        return sums, c.value

    def ccsd_t_spinorb(self):
        e = C.c_double(0)
        self._check("ccsd_t_spinorb", self.lib.afesp_gpu_ccsd_t_spinorb(self.h, C.byref(e)))
        return e.value

    # -- multi-GPU
    @staticmethod
    def comm_unique_id():
        lib = load_library()
        buf = C.create_string_buffer(128)
        rc = lib.afesp_gpu_comm_unique_id(buf)
        if rc != 0:
            raise AfespError("comm_unique_id", rc, lib.afesp_gpu_last_error(None).decode())
        return buf.raw

    def comm_init(self, rank, nranks, uid: bytes):
        assert len(uid) == 128
        self._check("comm_init", self.lib.afesp_gpu_comm_init(self.h, int(rank), int(nranks), uid))

    @staticmethod
    def host_register(arr) -> bool:
        """Page-lock a NumPy array in place (cudaHostRegister); False when the driver refuses."""
        return load_library().afesp_gpu_host_register(C.c_void_p(arr.ctypes.data), int(arr.nbytes)) == 0

    @staticmethod
    def host_unregister(arr) -> bool:
        return load_library().afesp_gpu_host_unregister(C.c_void_p(arr.ctypes.data)) == 0

    def set_partition(self, rank, nranks):
        self._check("set_partition", self.lib.afesp_gpu_set_partition(self.h, int(rank), int(nranks)))

    @staticmethod
    def triples_partition(nocc_active, nranks, symmetric=True, strict=False):
        lib = load_library()
        counts = (C.c_longlong * nranks)()
        rc = lib.afesp_gpu_triples_partition(int(nocc_active), int(symmetric), int(strict), int(nranks), counts)
        if rc != 0:
            raise AfespError("triples_partition", rc, "bad arguments")
        return list(counts)

    @staticmethod
    def column_partition(ncols, nranks, granularity=64):
        """[(lo, hi)] per rank: the column split of the sharded GEMMs (64) and of the AO->MO pair blocks (16)."""
        lib = load_library()
        lo, hi = (C.c_longlong * nranks)(), (C.c_longlong * nranks)()
        rc = lib.afesp_gpu_column_partition(int(ncols), int(nranks), int(granularity), lo, hi)
        if rc != 0:
            raise AfespError("column_partition", rc, "bad arguments")
        return list(zip(lo, hi))

    # -- linalg.fpp operators
    def dgemm_wrapper(self, transA, transB, M, N, K, A, B, Cmat=None, alpha=1.0, beta=0.0):
        """Same contract as dgemm_wrapper (src/linalg.fpp:58-89); A, B, C are flat column-major buffers."""
        a = np.ascontiguousarray(A, dtype=np.float64).ravel()
        b = np.ascontiguousarray(B, dtype=np.float64).ravel()
        c = np.zeros(M * N) if Cmat is None else np.ascontiguousarray(Cmat, dtype=np.float64).ravel().copy()
        self._check("dgemm_wrapper", self.lib.afesp_gpu_dgemm_wrapper(
            self.h, transA.encode(), transB.encode(), int(M), int(N), int(K), _ptr(a), _ptr(b), _ptr(c),
            float(alpha), float(beta)))
        return c

    def omp_reshape(self, in_arr, arr_order, out_arr=None, beta=None):
        """omp_reshape (src/linalg.fpp:99-156): in_arr is a 4-index array in index order; returns out in index order."""
        x = np.asarray(in_arr, dtype=np.float64)
        dims = (C.c_int * 4)(*x.shape)
        perm = [int(ch) - 1 for ch in arr_order]
        oshape = tuple(x.shape[p] for p in perm)
        xin = fortran_flat(x)
        out = np.zeros(x.size) if out_arr is None else fortran_flat(out_arr).copy()
        self._check("omp_reshape", self.lib.afesp_gpu_omp_reshape(
            self.h, _ptr(out), _ptr(xin), dims, arr_order.encode(), int(beta is not None),
            float(beta if beta is not None else 0.0)))
        return out.reshape(oshape, order="F")

    def bench_dgemm(self, transA, transB, M, N, K, reps=5, beta=0.0):
        ms = C.c_double(0)
        self._check("bench_dgemm", self.lib.afesp_gpu_bench_dgemm(self.h, transA.encode(), transB.encode(), int(M),
                                                                  int(N), int(K), float(beta), int(reps), C.byref(ms)))
        return ms.value

    def gemm_crosscheck(self, transA, transB, M, N, K, nbatch=1, beta=0.0, reps=10):
        """TMA-staged kernel vs cp.async kernel on one problem: (mismatching elements, ms TMA, ms cp.async)."""
        bad, a, b = C.c_longlong(0), C.c_double(0), C.c_double(0)
        self._check("gemm_crosscheck", self.lib.afesp_gpu_gemm_crosscheck(
            self.h, transA.encode(), transB.encode(), int(M), int(N), int(K), int(nbatch), float(beta), int(reps),
            C.byref(bad), C.byref(a), C.byref(b)))
        return bad.value, a.value, b.value

    def gemm_time(self):
        """(milliseconds, executed flop) of all DMMA GEMM launches since option gemm_timing was set / last call."""
        ms, fl = C.c_double(0), C.c_double(0)
        self._check("gemm_time", self.lib.afesp_gpu_gemm_time(self.h, C.byref(ms), C.byref(fl)))
        return ms.value, fl.value

    def bench_hbm(self, what, nocc, nvirt, reps=10):
        """(ms per launch, algorithmic bytes per launch) of an HBM-bound kernel at the (o,o,v,v) shape."""
        ms, by = C.c_double(0), C.c_double(0)
        self._check("bench_hbm", self.lib.afesp_gpu_bench_hbm(self.h, what.encode(), int(nocc), int(nvirt), int(reps),
                                                              C.byref(ms), C.byref(by)))
        return ms.value, by.value

    def tma_status(self):
        """(scope in force, self-test state): see afesp_gpu_tma_status."""
        a, b = C.c_int(0), C.c_int(0)
        self._check("tma_status", self.lib.afesp_gpu_tma_status(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def timer_start(self):
        self._check("timer", self.lib.afesp_gpu_timer(self.h, 0, None))

    def timer_stop(self):
        """Device milliseconds on the engine's stream since timer_start()."""
        ms = C.c_double(0)
        self._check("timer", self.lib.afesp_gpu_timer(self.h, 1, C.byref(ms)))
        return ms.value

    def gemm_stats(self):
        """(milliseconds, executed flop, launches) of the DMMA GEMM launches since gemm_timing was set / last call."""
        ms, fl, nl = C.c_double(0), C.c_double(0), C.c_longlong(0)
        self._check("gemm_stats", self.lib.afesp_gpu_gemm_stats(self.h, C.byref(ms), C.byref(fl), C.byref(nl)))
        return ms.value, fl.value, nl.value

    def dmma_peak(self):
        t = C.c_double(0)
        self._check("dmma_peak", self.lib.afesp_gpu_dmma_peak(self.h, C.byref(t)))
        return t.value
