#!/usr/bin/env python
"""Benchmark of the coupled-cluster hot path (BASELINE.json metric: CCSD s/iter & (T) wall-s; % FP64 tensor peak; vs CPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--nbf 200 --nocc 20] [--dump-outputs DIR]
    python bench.py --workload n2|f2|h2o|h2o-spinorb      (sample_data molecules, whole converged run; see below)

One "step" = one pass of the hot path over the synthetic (nbf, nocc) system: one spin-free CCSD iteration
(intermediates + amplitude equations + energy + DIIS extrapolation) followed by the full (T) correction
(calc_type CCSD(T)_spatial).  `value` = seconds per step, device-resident inputs, max over ranks; the breakdown
(ccsd_s_per_iter, t_wall_s, ao2mo_s) is carried in extra keys.  Under torchrun every rank runs its column share of the
CCSD GEMMs and its round-robin share of the (i<=j<=k) triples; the six (T) sums are combined by one NCCL allreduce inside
the library ("scaling": "strong": total work fixed).

After the timed loop at the headline shape (nbf=200/nocc=20, BASELINE.json configs[3]) the same hot path runs ONCE at
the north-star target shape nbf=400/nocc=40 (configs[4]; one e2e pass, then one device-timed pass) and is attached as
`target_config` -- its ~85 s step cannot be the K-step default of a bench that has to end in minutes.

`--impl reference` times the CPU port of the reference's own code path (oracle/cpu_ccsd.c, oracle/cpu_kernels.c: the same
dgemm calls through the image's OpenBLAS, the same omp_reshape passes and naive OpenMP loop nests as src/ccsd.f90) on all
host cores; the Fortran reference cannot be compiled here (no Fortran compiler).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ccsd_iter_plus_T_seconds"
UNIT = "s"
PINNED = os.environ.get("AFESP_BENCH_PINS") or os.path.join(ROOT, "tests", "golden", "bench_pinned.json")   # (env: tests)


# Keep stdout clean for the single JSON line: libraries loaded later (NCCL prints its version banner on stdout) write
# to fd 1, so fd 1 is pointed at stderr for the whole run and the JSON goes to the saved original descriptor.
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line: dict):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def config_of(nbf, nocc):
    """`config` of BOTH arms (the driver compares them): the workload and nothing else."""
    return {"workload": f"synthetic integrals nbf={nbf} nocc={nocc} CCSD(T)_spatial", "nbf": nbf, "nocc": nocc,
            "calc_type": "CCSD(T)_spatial"}


# ------------------------------------------------------------------------------------------------ CPU reference arm
def run_reference(args, rank):
    """The reference's CPU path (oracle/cpu_reference.py, a subprocess with its own thread environment: every host core
    for the OpenMP loops and the OpenBLAS dgemms).  One sample per step; see CpuReference for what a sample is."""
    if rank != 0:
        return
    from oracle import cpu_reference

    total = args.warmup + args.steps
    # CPU seconds per sample.  A sample with both naive o^3v^3 loop nests IN FULL costs ~17.5 s on 16 cores at nbf=200
    # (11.3 s CCSD iteration + 6.1 s for one complete triple per thread): 480 s over the driver's K + W = 25 samples leaves
    # room for that (19 s each, ~8 min in all); smaller budgets fall back to slabs of the nests' outer index, stated in `sample`
    budget = max(8.0, min(60.0, 480.0 / max(1, total)))
    res = cpu_reference.run_subprocess(args.nbf, args.nocc, total, budget)
    samples = res["samples"][args.warmup:]
    vals = [s["value"] for s in samples]
    ao = res["ao2mo"]
    v = float(np.mean(vals))
    last = samples[-1]
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": v * 1e3, "higher_is_better": False, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_of(args.nbf, args.nocc),
        "ccsd_s_per_iter": float(np.median([s["ccsd_s_per_iter"] for s in samples])),
        "t_wall_s": float(np.median([s["t_wall_s"] for s in samples])),
        "ao2mo_s": ao["ao2mo_s"] if ao else None, "ao2mo_slab": ao["slab"] if ao else None,
        "samples": {"n": len(vals), "min": float(np.min(vals)), "median": float(np.median(vals)), "max": float(np.max(vals)),
                    "cpu_seconds_per_sample": last["parts"]["ccsd_sample_s"] + last["parts"]["triples_sample_s"]},
        "parts_last_sample": last["parts"],
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": res["threads"], "kind": "port", "sample": last["describe"]},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "thread_env": res["env"],
        "note": "value is the full-workload time each bounded sample extrapolates to (factors in cpu_baseline.sample); "
                "the timed region itself is samples.cpu_seconds_per_sample per step",
    }
    emit(line)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ parity
def load_pins():
    try:
        return json.load(open(PINNED))
    except Exception:
        return {}


def parity_block(n, o, e_mp2, e_mp1, traj):
    """Energies of this run against the pinned values for the same shape.  CPU-computed pins: MP2 (NumPy oracle), E_CCSD
    after the first iteration (CPU port of the reference) and the (T) sum e_T of the first step (oracle, BLAS orbit form).
    Pins from the single-GPU (replicated) run: MP1 and, step by step, E_CCSD and e_T (sharded vs replicated at N > 1).
    Tolerance 1e-9 Eh (BASELINE.json north_star)."""
    pins = load_pins().get(f"nbf{n}_nocc{o}")
    if not pins:
        return {"pinned": False, "note": f"no pinned values for nbf={n} nocc={o} in tests/golden/bench_pinned.json"}
    tol = 1e-9
    out = {"pinned": True, "tolerance_Eh": tol, "source": pins.get("source")}
    diffs = {}
    if "e_mp2" in pins:
        diffs.update({"e_mp2": abs(e_mp2 - pins["e_mp2"]), "e_mp1": abs(e_mp1 - pins["e_mp1"])})
    if "e_mp2_oracle" in pins:
        diffs["e_mp2_vs_cpu_oracle"] = abs(e_mp2 - pins["e_mp2_oracle"])
    if "e_ccsd_iter1_cpu_port" in pins and traj:
        diffs["e_ccsd_iter1_vs_cpu_port"] = abs(traj[0][0] - pins["e_ccsd_iter1_cpu_port"])
    if "e_T_step1_cpu_oracle" in pins and traj:   # the (T) sum of the first step, computed on the CPU (make_bench_pins.py cpu_T)
        diffs["e_T_step1_vs_cpu_oracle"] = abs(traj[0][1] - pins["e_T_step1_cpu_oracle"])
    steps = pins.get("steps", [])
    k = min(len(traj), len(steps))
    if k:
        diffs["e_ccsd_max_over_steps"] = max(abs(traj[i][0] - steps[i][0]) for i in range(k))
        diffs["e_T_max_over_steps"] = max(abs(traj[i][1] - steps[i][1]) for i in range(k))
    cpu_steps = pins.get("steps_cpu", [])   # the first steps computed entirely on the CPU (make_bench_pins.py cpu_traj)
    kc = min(len(traj), len(cpu_steps))
    if kc:
        diffs["e_ccsd_vs_cpu_first_steps"] = max(abs(traj[i][0] - cpu_steps[i][0]) for i in range(kc))
        diffs["e_T_vs_cpu_first_steps"] = max(abs(traj[i][1] - cpu_steps[i][1]) for i in range(kc))
        out["steps_compared_with_cpu"] = kc
    out["steps_compared"] = k
    out["abs_diff"] = diffs
    out["ok"] = bool(diffs and all(d < tol for d in diffs.values()))
    return out


def mp1_triples_check(gpu, n, o, eps, src, big, chk):
    """(T) contributions of single unique triples, GPU against CPU, at a shape where no CPU CCSD iteration is affordable (the
    target shape nbf=400): the state right after afesp_gpu_ccsd_init holds the MP1 amplitudes, afesp_gpu_set_partition(r, T)
    makes the handle own exactly triple number r of the T unique (i <= j <= k) triples, and the CPU value of that orbit's [T]
    accumulator comes from the factored form of the synthetic integrals (tests/golden/make_bench_pins.py cpu_mp1_triples).
    Runs after all measurements (it re-initialises the CCSD state).  Relative tolerance 1e-9 (absolute floor 1e-15 Eh: the
    i = j = k orbits vanish identically)."""
    gpu.set_option("finalize_keep_ccsd", 0)
    gpu.ccsd_finalize()          # drop what the device-timed loop kept (DIIS history, ladder integrals, intermediates)
    gpu.release("scratch")
    gpu.set_eri_mo(n, src)       # from here on the sequence of the e2e leg without the iteration
    gpu.ccsd_init(o, True, eps, 8)
    if big:
        gpu.release("eri_mo")
    gpu.ccsd_finalize()
    got = []
    try:
        for r in chk["ranks"]:
            gpu.set_partition(int(r), int(chk["ntriples"]))
            sums, _ = gpu.ccsd_t_spatial(True, False, False)
            got.append(float(sums[0]))
    finally:
        gpu.set_partition(0, 1)
    diffs = [abs(a - b) for a, b in zip(got, chk["e_T"])]
    ok = all(d <= max(1e-9 * abs(c), 1e-15) for d, c in zip(diffs, chk["e_T"]))
    return {"what": "e_T of single (i<=j<=k) orbits on the MP1 amplitudes: GPU (set_partition(r, ntriples) + ccsd_t_spatial) "
                    "against NumPy from the factored integrals", "ijk": chk["ijk"], "e_T_gpu": got, "e_T_cpu": chk["e_T"],
            "abs_diff": diffs, "tolerance": "relative 1e-9, absolute floor 1e-15 Eh", "ok": bool(ok)}


# ------------------------------------------------------------------------------------------------ outputs
DUMP_T2_SAMPLE = 1 << 20   # T2 positions kept by --dump-outputs (8 MB; all of T2 is 104 MB at nbf=200/nocc=20)


def dump_outputs(gpu, out_dir, last):
    """--dump-outputs: what a caller of the timed path receives from its last step, as float64 .npy files, so that two
    builds run with the same arguments (hence the same seeded inputs) can be compared output by output:
      ccsd_iterate.npy   [E_CCSD, rms of the T2 update] (afesp_gpu_ccsd_iterate)
      t1_diagnostic.npy  [T1 diagnostic] (afesp_gpu_ccsd_finalize)
      ccsd_t_sums.npy    the six (T) sums (afesp_gpu_ccsd_t_spatial)
      t1.npy             T1 (nocc, nvirt)
      t2_sample.npy      T2 at DUMP_T2_SAMPLE distinct positions of its column-major (nocc, nocc, nvirt, nvirt) storage,
                         drawn with a fixed seed and kept in ascending order (all of T2 when it is not larger)
    The amplitudes are read with afesp_gpu_ccsd_finalize, which under finalize_keep_ccsd=1 copies them and changes no state."""
    _, t1, t2 = gpu.ccsd_finalize(want_amplitudes=True)
    t2 = t2.ravel(order="F")
    if t2.size > DUMP_T2_SAMPLE:
        t2 = t2[np.sort(np.random.default_rng(0).choice(t2.size, DUMP_T2_SAMPLE, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("ccsd_iterate", [last["e_ccsd"], last["rms"]]), ("t1_diagnostic", [last["t1_diagnostic"]]),
                    ("ccsd_t_sums", last["sums"]), ("t1", t1), ("t2_sample", t2)):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))
    log(f"outputs of the last timed step written to {out_dir}")


# ------------------------------------------------------------------------------------------------ GPU arm
def attach_comm(gpu, rank, world):
    import torch
    import torch.distributed as dist

    from afesp_b200 import AfespGpu

    uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        uid = torch.tensor(list(AfespGpu.comm_unique_id()), dtype=torch.uint8, device="cuda")
    dist.broadcast(uid, 0)
    gpu.comm_init(rank, world, bytes(uid.cpu().tolist()))


def run_shape(args, rank, world, local, n, o, steps, warmup, e2e_first=False, want_hbm=True, dump_dir=None):
    """The hot path at one (nbf, nocc) shape: device-resident timed loop + e2e leg.  Returns the measurement dict
    (rank 0) or None.  dump_dir: see dump_outputs."""
    import torch
    import torch.distributed as dist

    from afesp_b200 import AfespGpu, synthetic

    v = n - o
    big = n > 240   # host-side expansion of the packed ERIs needs npair^2 doubles: expand on the device instead
    t0 = time.perf_counter()
    if big:
        Bfac, Cmo, eps = synthetic.make_factors(n, o)
        eri = None
    else:
        eri, Cmo, eps = synthetic.make(n, o)
    log(f"[rank {rank}] synthetic inputs nbf={n} nocc={o} generated in {time.perf_counter() - t0:.1f}s")
    gpu = AfespGpu(local)
    if world > 1:
        attach_comm(gpu, rank, world)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.tma >= 0:
        gpu.set_option("gemm_use_tma", args.tma)
    if args.dist_chunks > 0:
        gpu.set_option("dist_overlap_chunks", args.dist_chunks)
    if os.environ.get("AFESP_DIST_ALLGATHER") is not None:   # A/B aid: 0 = grouped broadcasts, 1 = one all-gather
        gpu.set_option("dist_allgather", float(os.environ["AFESP_DIST_ALLGATHER"]))
    tma_scope, tma_selftest = gpu.tma_status()
    peak = max(gpu.dmma_peak(), gpu.dmma_peak())
    npair = n * (n + 1) // 2
    npk = npair * (npair + 1) // 2
    # host copy of the packed MO integrals (input of the e2e leg): ONE copy per node.  Single GPU: a pinned buffer.  Several
    # ranks: a shared-memory file (/dev/shm) written by rank 0 and mapped + page-locked (cudaHostRegister) by every rank,
    # so that each rank uploads its 1/N share over its own PCIe link inside afesp_gpu_set_eri_mo.
    src, shm_path, shm_registered = None, None, False
    if world == 1:
        pinned = torch.empty(npk, dtype=torch.float64).pin_memory()
        src = pinned.numpy()
    else:
        ok = 0.0
        shm_path = "/dev/shm/afesp_bench_%s_%d.bin" % (os.environ.get("MASTER_PORT", "0"), n)
        try:
            st = os.statvfs("/dev/shm")
            # (arrays above 4 GB stay on the proven path -- one pinned copy on rank 0 + NVLink broadcast: page-locking a
            #  25.7 GB tmpfs mapping from 8 processes at once is where an nbf=400 run at N=8 stalled)
            if npk * 8 <= (4 << 30) and st.f_bavail * st.f_frsize > npk * 8 * 1.1:
                if rank == 0:
                    np.memmap(shm_path, dtype=np.float64, mode="w+", shape=(npk,)).flush()
                ok = 1.0
        except OSError:
            ok = 0.0
        flag = torch.tensor([ok if rank == 0 else 1.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if flag.item() > 0.5:
            src = np.memmap(shm_path, dtype=np.float64, mode="r+", shape=(npk,))
            shm_registered = AfespGpu.host_register(src)   # False: the driver refused (error cleared inside)
        flag = torch.tensor([1.0 if shm_registered else 0.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if flag.item() < 0.5:
            # no page-locked shared mapping on this box (small /dev/shm, registration refused): one pinned copy on rank 0,
            # the other ranks receive the integrals over NVLink inside afesp_gpu_set_eri_mo
            if shm_registered:
                AfespGpu.host_unregister(src)
            shm_registered = False
            src = None
            if rank == 0:
                try:
                    os.unlink(shm_path)
                except OSError:
                    pass
                src = torch.empty(npk, dtype=torch.float64).pin_memory().numpy()
            shm_path = None
    amp_out = None
    if rank == 0:   # pinned landing buffers for the D2H of T1/T2 (only rank 0 asks for the amplitudes)
        amp_out = (torch.empty(o * v, dtype=torch.float64).pin_memory().numpy(),
                   torch.empty(o * o * v * v, dtype=torch.float64).pin_memory().numpy())
    if big:
        gpu.synth_eri_ao(n, Bfac, Cmo)
        gpu.ao2mo(n, want_result=False)
    else:
        gpu.ao2mo(n, eri, Cmo, want_result=False)   # also leaves AO integrals + C resident
        gpu.ao2mo(n)                                # resident repeat, device-timed
    ao2mo_ms = gpu.last_stage_ms()
    if rank == 0:
        gpu.get_eri_mo(src)
    barrier()   # the shared host copy is complete before any rank reads its share
    gpu.release("eri_ao")
    e_mp2 = gpu.mp2_energy(o, eps)
    h2d = int(npk * 8 + n * 8)
    d2h = int((o * o * v * v + o * v) * 8 + 10 * 8)
    parts = {"h2d_set_eri_mo": 0.0, "ccsd_init": 0.0, "iterate+diis": 0.0, "finalize_d2h": 0.0, "ccsd_t": 0.0}

    def e2e_leg(ksteps):
        """End to end through the C ABI with host buffers (pinned): H2D of the step's MO integrals, D2H of amplitudes."""
        def lap(key, t_prev):
            t = time.perf_counter()
            parts[key] += t - t_prev
            return t

        gpu.set_option("finalize_keep_ccsd", 0)   # the product path: finalize frees the CCSD work arrays before (T)
        barrier()
        t0 = time.perf_counter()
        for _ in range(ksteps):
            t = time.perf_counter()
            gpu.set_eri_mo(n, src)
            t = lap("h2d_set_eri_mo", t)
            gpu.ccsd_init(o, True, eps, 8)
            if big:
                gpu.release("eri_mo")
            t = lap("ccsd_init", t)
            gpu.ccsd_iterate()
            gpu.ccsd_diis()
            t = lap("iterate+diis", t)
            gpu.ccsd_finalize(out=amp_out)   # D2H of T1/T2 into pinned memory on rank 0 (None elsewhere: no copy)
            t = lap("finalize_d2h", t)
            gpu.ccsd_t_spatial(True, False, False)
            t = lap("ccsd_t", t)
        barrier()
        el = time.perf_counter() - t0
        te = torch.tensor([el], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return float(te.item()) / ksteps

    e2e_value = None
    if e2e_first:   # target shape: the e2e pass doubles as the warm-up of the device-timed pass
        e2e_value = e2e_leg(1)
        gpu.set_eri_mo(n, src)
    # ---- device-resident leg
    gpu.set_option("finalize_keep_ccsd", 1)
    e_mp1, _ = gpu.ccsd_init(o, True, eps, 8)
    if big:
        gpu.release("eri_mo")
    comp = {"ccsd": [], "diis": [], "t": []}
    gstat = {"ccsd": [0.0, 0.0, 0], "t": [0.0, 0.0, 0]}   # DMMA GEMM (ms, flop, launches) per stage of the timed region
    traj = []
    last = {}

    def step(record):
        e, rms = gpu.ccsd_iterate()
        a = gpu.last_stage_ms()
        gpu.ccsd_diis()
        b = gpu.last_stage_ms()
        t1_diag, _, _ = gpu.ccsd_finalize()
        if record:
            ms, fl, nl = gpu.gemm_stats()
            gstat["ccsd"][0] += ms; gstat["ccsd"][1] += fl; gstat["ccsd"][2] += nl
        sums, _ = gpu.ccsd_t_spatial(True, False, False)
        c = gpu.last_stage_ms()
        if record:
            ms, fl, nl = gpu.gemm_stats()
            gstat["t"][0] += ms; gstat["t"][1] += fl; gstat["t"][2] += nl
        traj.append([e, float(sums[0]), rms])
        last.update(e_ccsd=e, rms=rms, t1_diagnostic=t1_diag, sums=sums)
        if record:
            comp["ccsd"].append(a); comp["diis"].append(b); comp["t"].append(c)

    for _ in range(warmup):
        step(False)
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    l0, f0 = gpu.counters()
    gpu.set_option("gemm_timing", 1)
    gpu.timer_start()                      # CUDA events on the stream the kernels are launched on
    t0 = time.perf_counter()
    for _ in range(steps):
        step(True)
    dev_ms = gpu.timer_stop()
    barrier()
    wall = time.perf_counter() - t0
    gpu.set_option("gemm_timing", 0)
    l1, f1 = gpu.counters()
    clocks = sampler.stop() if sampler else None
    tt = torch.tensor([dev_ms * 1e-3, wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    elapsed, wall = float(tt[0].item()), float(tt[1].item())
    value = elapsed / steps
    if dump_dir and rank == 0:   # before the e2e leg, which starts the CCSD state afresh
        dump_outputs(gpu, dump_dir, last)

    if not e2e_first:
        e2e_value = e2e_leg(steps)
    ksteps = 1 if e2e_first else steps

    # ---- HBM-bound kernels of the path (permute / denominators / energy), device resident, vs the measured copy peak
    hbm = None
    if rank == 0 and want_hbm:
        try:
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
            peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy)"
        except Exception:
            hbm_peak, peak_src = 6452.0, "fallback 6452 GB/s (B200_PROFILING.md measured copy)"
        hbm = {"peak_gbs": hbm_peak, "peak_source": peak_src, "kernels": {}}
        for (oo_, vv_) in sorted({(o, v), (40, 360)}):
            for what in ("permute:3412", "permute:2143", "permute_acc:2143", "divide", "energy", "axpby"):
                try:
                    ms, by = gpu.bench_hbm(what, oo_, vv_, reps=20)
                    hbm["kernels"][f"{what} o={oo_} v={vv_}"] = {
                        "ms": ms, "algorithmic_bytes": by, "gbs": by / ms / 1e6, "frac": by / ms / 1e6 / hbm_peak}
                except Exception as ex:
                    hbm["kernels"][f"{what} o={oo_} v={vv_}"] = {"error": str(ex)}
    # ---- per-triple (T) check against CPU values (shapes with such pins: the target shape), after every measurement
    mp1_check = None
    chk = (load_pins().get(f"nbf{n}_nocc{o}") or {}).get("mp1_triples")
    if chk and world == 1:
        try:
            mp1_check = mp1_triples_check(gpu, n, o, eps, src, big, chk)
        except Exception as ex:   # a check, never a reason to lose the measurements
            mp1_check = {"error": f"{type(ex).__name__}: {ex}"}
    out = None
    if rank == 0:
        traffic, traffic_source = None, None
        tpath = os.path.join(ROOT, "profiles", "ncu_gemm_traffic.json")
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                traffic = tj.get("dram_bytes_per_launch", {}).get(f"nbf{n}", {}).get("tma" if tma_scope >= 1 else "cpasync")
                traffic_source = ("static: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of "
                                  "this kernel at this shape, " + str(tj.get("sources", {}).get("tma" if tma_scope >= 1 else "cpasync"))
                                  + " (not measured in this run)") if traffic else None
            except Exception:
                traffic = None
        tot_ms = gstat["ccsd"][0] + gstat["t"][0]
        tot_fl = gstat["ccsd"][1] + gstat["t"][1]
        tf = lambda g: (g[1] / (g[0] * 1e-3) / 1e12) if g[0] > 0 else None
        # dominant kernel: the batched (T) GEMM, one launch per batch of triples: per block
        #   Y_s(x,(u,w)) = Acat(x,[d|l]; P0,P1) Bcat([d|l],(u,w); P2) + Acat(x,[d|l]; P0,P2) BcatT([d|l],(u,w); P1)
        t_ms, t_fl, t_nl = gstat["t"]
        achieved = tf(gstat["t"])
        out = {
            "value": value, "ms_per_step": value * 1e3, "wall_s_per_step": wall / steps, "steps": steps, "warmup": warmup,
            "ccsd_s_per_iter": (float(np.mean(comp["ccsd"])) + float(np.mean(comp["diis"]))) / 1e3,
            "t_wall_s": float(np.mean(comp["t"])) / 1e3, "ao2mo_s": ao2mo_ms / 1e3,
            "energies": {"e_mp2": e_mp2, "e_mp1": e_mp1, "e_ccsd": traj[-1][0], "rms": traj[-1][2], "e_T": traj[-1][1]},
            "trajectory": [[t[0], t[1]] for t in traj],
            "parity": parity_block(n, o, e_mp2, e_mp1, traj),
            "gemm_tflops_executed": {"all": (tot_fl / (tot_ms * 1e-3) / 1e12) if tot_ms > 0 else None,
                                     "ccsd": tf(gstat["ccsd"]), "t": tf(gstat["t"]),
                                     "gemm_share_of_step": tot_ms * 1e-3 / elapsed if elapsed > 0 else None},
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": traffic_source,
                         "kernel": ("gemm_f64_tma<N,N>" if tma_scope >= 1 else "gemm_f64_dmma<64,64,16> (cp.async ring)") +
                                   f" batched over (triple, first-label permutation) blocks: (T) contraction M={v} N={v * v} "
                                   f"K=2x{n} per block (two K segments: the permutations sharing their first label)",
                         "launches": t_nl, "flops_per_launch": (t_fl / t_nl) if t_nl else None,
                         "ms_per_launch": (t_ms / t_nl) if t_nl else None,
                         "share_of_step": t_ms * 1e-3 / elapsed if elapsed > 0 else None,
                         "all_gemms": {"achieved": (tot_fl / (tot_ms * 1e-3) / 1e12) if tot_ms > 0 else None,
                                       "flops_per_step": tot_fl / steps, "ms_per_step": tot_ms / steps},
                         "peak_source": "BUILDER-MEASURED: in-run register-resident DMMA.8x8x4 issue-rate probe "
                                        "(afesp_gpu_dmma_peak); MEASURED_PEAKS.json has no FP64 entry; vendor FP64 "
                                        "tensor figure 40 TFLOP/s"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "what": "set_eri_mo(H2D from pinned host memory" + ((", each rank its 1/N share over its own PCIe link, "
                            "shares exchanged over NVLink" if shm_path else ", rank 0 uploads, NVLink broadcast") if world > 1 else "") + ") + ccsd_init + iterate + diis + "
                            "finalize(D2H t1,t2 into pinned memory) + ccsd_t"
                            + ("; single pass that also served as warm-up of the device-timed pass" if e2e_first else ""),
                    "breakdown_s": {k: x / ksteps for k, x in parts.items()}},
            "gpu_launches": int(l1 - l0), "clocks": clocks,
            "tma": {"scope": tma_scope, "selftest": tma_selftest}, "hbm_kernels": hbm,
        }
    if out is not None and mp1_check is not None:
        out["parity"]["mp1_triples_vs_cpu"] = mp1_check
        if mp1_check.get("ok") is False:
            out["parity"]["ok"] = False
    gpu.close()
    if shm_path is not None:
        if shm_registered:
            AfespGpu.host_unregister(src)
        del src
        barrier()
        if rank == 0:
            try:
                os.unlink(shm_path)
            except OSError:
                pass
    return out


def run_ours(args, rank, world, local):
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n, o = args.nbf, args.nocc
    v = n - o
    m = run_shape(args, rank, world, local, n, o, args.steps, args.warmup, dump_dir=args.dump_outputs)
    line = None
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu:
            try:
                from oracle import cpu_reference

                res = cpu_reference.run_subprocess(n, o, 2, 25.0, ao2mo_budget=4.0)   # first sample calibrates the slabs
                smp, ao = res["samples"][-1], res["ao2mo"]
                cpu = {"value": smp["value"], "unit": UNIT, "cores": res["threads"], "kind": "port", "sample": smp["describe"],
                       "ccsd_s_per_iter": smp["ccsd_s_per_iter"], "t_wall_s": smp["t_wall_s"],
                       "ao2mo_s": ao["ao2mo_s"] if ao else None, "parts": smp["parts"]}
            except Exception as ex:  # the CPU leg must never take the GPU line down
                cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {ex}"}
        line = {
            "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": m["ms_per_step"], "higher_is_better": False, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_of(n, o),
            "parallelism": (f"(T) ijk round-robin x{world}; CCSD GEMMs column-sharded x{world} with NCCL slab exchange, "
                            f"V+/- ladder integrals sharded by column block") if world > 1 else "single GPU",
            "l2": "inputs larger than L2 (packed ladder integrals %.1f GB, (T) work buffers %.1f GB)" % (v ** 4 * 4 / 1e9, 6.0),
            "timing": "CUDA events on the engine's stream around the K steps, max over ranks",
        }
        for k in ("wall_s_per_step", "ccsd_s_per_iter", "t_wall_s", "ao2mo_s", "energies", "parity", "gemm_tflops_executed",
                  "roofline", "e2e", "gpu_launches", "clocks", "tma", "hbm_kernels"):
            line[k] = m[k]
        line["cpu_baseline"] = cpu
        line["target_config"] = None
        if args.trajectory:
            line["trajectory"] = m["trajectory"]
        if world > 1:
            line["exchange"] = "NCCL slab exchange of the column-sharded CCSD GEMMs; one allreduce of the six (T) sums"
    # ---- the north-star target shape, once, AFTER the headline measurements are complete.  A watchdog on every rank
    # guarantees that the headline line is printed even if this leg stalls (several ranks at this shape have had far
    # less GPU time than the headline shape): at the limit rank 0 prints the line with an error note and all ranks leave.
    tn, to = (int(x) for x in os.environ.get("AFESP_BENCH_TARGET_SHAPE", "400,40").split(","))   # (tests use a small one)
    run_target = (args.target == 2 or (args.target == 1 and world == 1)) and (n, o) != (tn, to)
    if args.target == 1 and world > 1 and line is not None:
        line["target_config"] = {"skipped": "the nbf=400 target leg runs by default on one GPU only; --target 2 runs it on "
                                            "every rank count (watchdog-limited)"}
    if run_target:
        import threading

        limit = float(os.environ.get("AFESP_BENCH_TARGET_LIMIT_S", "600" if world == 1 else "300"))
        done = threading.Event()

        def watchdog():
            if not done.wait(limit):
                if line is not None:
                    line["target_config"] = {"error": f"target leg did not finish within {limit:.0f} s: abandoned by the "
                                                      f"watchdog (headline measurements above are complete)"}
                    emit(line)
                os._exit(0)

        threading.Thread(target=watchdog, daemon=True).start()
        target = None
        try:
            target = run_shape(args, rank, world, local, tn, to, 1, 0, e2e_first=True, want_hbm=False)
            if target is not None:
                target.pop("hbm_kernels", None)
                if not args.trajectory:
                    target.pop("trajectory", None)
                target["config"] = config_of(tn, to)
                target["note"] = ("BASELINE.json configs[4], the north-star target shape: one e2e pass (which is also the "
                                  "warm-up), then ONE device-timed step (W=0 after that pass, K=1)")
        except Exception as ex:   # the target leg must never take the headline line down
            target = {"error": f"{type(ex).__name__}: {ex}"}
        done.set()
        if line is not None:
            line["target_config"] = target
    if line is not None:
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nbf", type=int, default=200)
    ap.add_argument("--nocc", type=int, default=20)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--target", type=int, default=int(os.environ.get("AFESP_BENCH_TARGET", "1")),
                    help="1 (default): on ONE GPU also run the nbf=400/nocc=40 target shape once and attach it as "
                         "target_config; 2: at every rank count; 0: never")
    ap.add_argument("--trajectory", action="store_true", help="print the per-step (E_CCSD, e_T) list (pinning runs)")
    ap.add_argument("--tma", type=int, default=-1, help="gemm_use_tma: -1 library default (2: TMA-staged kernel for every "
                                                        "aligned GEMM), 1 the (T) batches only, 0 cp.async kernels only")
    ap.add_argument("--dist-chunks", type=int, default=0, help="dist_overlap_chunks of the sharded CCSD GEMMs (0: library default)")
    ap.add_argument("--workload", default=None, help="sample_data molecule run: n2 | f2 | h2o | h2o-spinorb")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload or args.impl != "ours"):
        ap.error("--dump-outputs applies to the GPU arm at the synthetic shape only")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload:
        from tools import bench_samples

        bench_samples.run(args, rank, world, local, emit, log)
        return
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_ours(args, rank, world, local)


if __name__ == "__main__":
    main()
