"""Frozen-core cost on the device: one CCSD iteration and one CCSD(T) triples pass per number of frozen orbitals k.

    python tools/bench_frozen_core.py [--out profiles/frozen_core_b200.jsonl]

Synthetic inputs of afesp_b200.synthetic (the bench's seed) at nbf=400/nocc=40 (BASELINE.json configs[4]) with
k in {0, 8, 9}, and at nbf=200/nocc=20 with k in {0, 3, 4}.  One AO->MO per shape; then per k: ccsd_init, one
ccsd_iterate, ccsd_finalize and ccsd_t_spatial(paren) -- the stages bench.py times, the same (T) variant.  An odd k makes
the number of active occupied orbitals odd while v stays even: that is the case where the (T) GEMM depth K = v + o is
padded to keep the 16-byte-aligned (TMA) kernel, and where the CCSD GEMMs with a leading dimension o lose it.

One JSON line per (shape, k): device seconds of the iteration and of (T) (CUDA events on the engine's stream), the
DMMA GEMM TFLOP/s of both stages (gemm_stats: executed flop, padding included, over summed GEMM kernel time), the
energies, and the card's name and power limit read with nvidia-smi in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from afesp_b200 import AfespGpu, synthetic  # noqa: E402

SHAPES = [(400, 40, [0, 8, 9]), (200, 20, [0, 3, 4])]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=60)
    if q.returncode != 0:
        raise RuntimeError("nvidia-smi failed: " + q.stderr)
    name, power = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--shapes", default=None, help="e.g. 200:20:0,3,4 (default: the two shapes above)")
    args = ap.parse_args()
    shapes = SHAPES
    if args.shapes:
        shapes = []
        for spec in args.shapes.split(";"):
            n, o, ks = spec.split(":")
            shapes.append((int(n), int(o), [int(k) for k in ks.split(",")]))
    name, power = card()
    out = open(args.out, "a") if args.out else None
    gpu = AfespGpu(0)
    try:
        for n, o, ks in shapes:
            t0 = time.perf_counter()
            B, C, eps = synthetic.make_factors(n, o)   # the packed ERIs are expanded on the device
            gpu.synth_eri_ao(n, B, C)
            gpu.ao2mo(n, want_result=False)
            gpu.release("eri_ao")
            gen_s = time.perf_counter() - t0
            for k in ks:
                gpu.set_option("frozen_core", k)
                e_mp2 = gpu.mp2_energy(o, eps)
                e_mp1, _ = gpu.ccsd_init(o, True, eps, 8)
                gpu.set_option("gemm_timing", 1)
                gpu.gemm_stats()                       # reset the GEMM counters
                e_ccsd, rms = gpu.ccsd_iterate()
                it_ms = gpu.last_stage_ms()
                it_gemm = gpu.gemm_stats()
                t1_diag, _, _ = gpu.ccsd_finalize()
                gpu.gemm_stats()
                sums, _ = gpu.ccsd_t_spatial(True, False, False)
                t_ms = gpu.last_stage_ms()
                t_gemm = gpu.gemm_stats()
                gpu.set_option("gemm_timing", 0)
                oa, v = o - k, n - o
                line = {"what": "frozen-core CCSD iteration + CCSD(T), synthetic integrals", "nbf": n, "nocc": o,
                        "frozen_core": k, "o_active": oa, "v": v, "t_gemm_K": v + oa + (1 if v % 2 == 0 and oa % 2 else 0),
                        "ccsd_iter_s": it_ms * 1e-3, "triples_s": t_ms * 1e-3,
                        "ccsd_gemm_tflops": it_gemm[1] / (it_gemm[0] * 1e-3) / 1e12 if it_gemm[0] > 0 else None,
                        "ccsd_gemm_s": it_gemm[0] * 1e-3,
                        "triples_gemm_tflops": t_gemm[1] / (t_gemm[0] * 1e-3) / 1e12 if t_gemm[0] > 0 else None,
                        "triples_gemm_s": t_gemm[0] * 1e-3, "triples_gemm_launches": t_gemm[2],
                        "e_mp2": e_mp2, "e_mp1": e_mp1, "e_ccsd_iter1": e_ccsd, "rms_iter1": rms, "t1_diagnostic": t1_diag,
                        "e_T": float(sums[0]), "triples_sums": [float(x) for x in sums],
                        "tma_status": list(gpu.tma_status()), "inputs_s": gen_s, "gpu": name, "power_limit": power}
                print(json.dumps(line), flush=True)
                if out:
                    out.write(json.dumps(line) + "\n")
                    out.flush()
            gpu.set_option("frozen_core", 0)
            gpu.release("eri_mo")
            gpu.release("scratch")
    finally:
        gpu.close()
        if out:
            out.close()


if __name__ == "__main__":
    main()
