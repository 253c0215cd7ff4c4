"""Multi-GPU parity: the rank-sharded AO->MO / CCSD / (T) path against the replicated single-GPU path, same inputs.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 \
        tools/dist_check.py [--nbf 96 --nocc 10]

Every rank first runs the whole chain with the communicator's CCSD sharding switched off (option dist_ccsd = 0: only
(T) is partitioned), then again with it on (column-sharded GEMMs + NCCL slab exchange, V+/- slabs, AO->MO all-to-all),
and compares: packed MO integrals (1e-12), every CCSD iteration energy (1e-10 Eh), T1/T2 (1e-9), (T) sums (1e-10).
Also checks that all ranks hold bit-identical amplitudes after the sharded run.  Exit code 0 = pass.

The compared iterations run WITHOUT the DIIS extrapolation (plain fixed-point steps, which contract differences).
With DIIS the comparison would measure the conditioning of the DIIS linear system rather than the sharding: on a
single GPU, two runs that differ only in the summation order inside a k-tile (TMA kernel vs cp.async kernel) drift
apart by up to 2e-10 Eh within 6 extrapolated iterations of these fast-converging synthetic systems and meet
again at convergence
(tools/rounding_sensitivity.py, profiles/r01_rounding_sensitivity.json) -- and slab-width GEMMs select other tile
shapes than full-width ones.  `--diis` switches the extrapolation back on."""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
_REAL = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)

import torch
import torch.distributed as dist

from afesp_b200 import AfespGpu, synthetic


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nbf", type=int, default=96)
    ap.add_argument("--nocc", type=int, default=10)
    ap.add_argument("--iters", type=int, default=6)
    ap.add_argument("--spinorb", action="store_true")
    ap.add_argument("--diis", action="store_true", help="extrapolate between the compared iterations")
    ap.add_argument("--frozen-core", type=int, default=0, help="frozen doubly occupied orbitals (option frozen_core)")
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n, o = args.nbf, args.nocc
    eri, Cmo, eps = synthetic.make(n, o)
    gpu = AfespGpu(local)
    uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        uid = torch.tensor(list(AfespGpu.comm_unique_id()), dtype=torch.uint8, device="cuda")
    dist.broadcast(uid, 0)
    gpu.comm_init(rank, world, bytes(uid.cpu().tolist()))
    gpu.set_option("dist_min_flops", 0.0)   # shard every GEMM wide enough, also at this small shape
    if args.frozen_core:
        gpu.set_option("frozen_core", args.frozen_core)   # every rank sets it, like the other collective arguments

    def chain(sharded):
        gpu.set_option("dist_ccsd", 1.0 if sharded else 0.0)
        mo = gpu.ao2mo(n, eri, Cmo, want_result=True)
        e_mp2 = gpu.mp2_energy(o, eps)
        e0, _ = gpu.ccsd_init(o, not args.spinorb, eps, 8)
        es = [e0]
        for _ in range(args.iters):
            e, r = gpu.ccsd_iterate()
            if args.diis:
                gpu.ccsd_diis()
            es.append(e)
        _, t1, t2 = gpu.ccsd_finalize(want_amplitudes=True)
        if args.spinorb:
            sums = np.array([gpu.ccsd_t_spinorb()])
        else:
            sums, _ = gpu.ccsd_t_spatial(True, False, False)
        return mo, e_mp2, np.array(es), t1, t2, np.array(sums)

    ref = chain(False)
    got = chain(True)
    names = ["eri_mo", "e_mp2", "ccsd energies", "t1", "t2", "(T) sums"]
    tols = [1e-12, 1e-12, 1e-10, 1e-9, 1e-9, 1e-10]
    errs = [float(np.max(np.abs(np.asarray(a) - np.asarray(b)))) for a, b in zip(ref, got)]
    # worst rank: every rank compares its own two runs
    et = torch.tensor(errs, dtype=torch.float64, device="cuda")
    dist.all_reduce(et, op=dist.ReduceOp.MAX)
    errs = [float(x) for x in et.tolist()]
    ok = all(e <= t for e, t in zip(errs, tols))
    per_iter = [float(x) for x in np.abs(ref[2] - got[2])]
    # replicated state must be bit-identical on every rank
    t2 = torch.from_numpy(np.ascontiguousarray(got[4]).ravel()).cuda()
    lo, hi = t2.clone(), t2.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    identical = bool(torch.equal(lo, hi))
    flag = torch.tensor([1.0 if (ok and identical) else 0.0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        _REAL.write(json.dumps({"world": world, "nbf": n, "nocc": o, "spinorb": args.spinorb, "diis": args.diis,
                                "frozen_core": args.frozen_core,
                                "max_abs_err": dict(zip(names, errs)), "tol": dict(zip(names, tols)),
                                "ranks_bit_identical": identical, "e_ccsd": float(got[2][-1]),
                                "abs_err_energy_per_iteration_rank0": per_iter,
                                "pass": bool(flag.item() == 1.0)}) + "\n")
        _REAL.flush()
    gpu.close()
    dist.destroy_process_group()
    sys.exit(0 if flag.item() == 1.0 else 1)


if __name__ == "__main__":
    main()
