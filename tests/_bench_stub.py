"""Stand-ins that let bench.py's GPU arm run on a CPU-only machine (tests/test_bench_flow.py): a fake engine behind the
AfespGpu interface, torch.cuda calls turned into no-ops, the NCCL process group replaced by gloo.  Only the CONTROL FLOW of
bench.py is exercised (argument handling, the shared-memory host copy, the target leg and its watchdog, the JSON line);
no number it prints means anything."""
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

_real_tensor, _real_zeros, _real_init = torch.tensor, torch.zeros, dist.init_process_group


def _strip(kw):
    kw.pop("device", None)
    return kw


torch.tensor = lambda *a, **k: _real_tensor(*a, **_strip(k))
torch.zeros = lambda *a, **k: _real_zeros(*a, **_strip(k))
torch.Tensor.pin_memory = lambda self: self
torch.Tensor.cuda = lambda self, *a, **k: self
torch.cuda.set_device = lambda *a, **k: None
torch.cuda.synchronize = lambda *a, **k: None
dist.init_process_group = lambda backend=None, **k: _real_init("gloo")

import afesp_b200  # noqa: E402


class FakeGpu:
    stall_target = os.environ.get("AFESP_STUB_STALL") == "1"
    registered = []

    def __init__(self, device=0):
        self.n = 0
        self.iter = 0
        self.launches = 0

    # context
    def close(self): pass
    def set_option(self, key, value): pass
    def tma_status(self): return 2, 1
    def dmma_peak(self): return 37.0
    def counters(self): self.launches += 100; return self.launches, 1e12
    def last_stage_ms(self): return 1.0
    def timer_start(self): self.t0 = time.perf_counter()
    def timer_stop(self): return (time.perf_counter() - self.t0) * 1e3 + 1.0
    def gemm_stats(self): return 0.5, 1e10, 3
    def bench_hbm(self, what, o, v, reps=10): return 0.1, 16.0 * o * o * v * v
    @staticmethod
    def comm_unique_id(): return bytes(range(128))
    def comm_init(self, rank, nranks, uid): assert len(uid) == 128
    @staticmethod
    def host_register(arr): FakeGpu.registered.append(arr.ctypes.data); return True
    @staticmethod
    def host_unregister(arr): FakeGpu.registered.remove(arr.ctypes.data); return True

    # stages
    def synth_eri_ao(self, n, B, C): self.n = n
    def ao2mo(self, n, eri=None, C=None, want_result=True): self.n = n
    def get_eri_mo(self, out=None):
        if self.stall_target and self.n == int(os.environ.get("AFESP_BENCH_TARGET_SHAPE", "400,40").split(",")[0]):
            time.sleep(3600)   # a stalled target leg: the watchdog has to get the headline line out
        out[:8] = 1.0
        return out
    def release(self, what): pass
    def mp2_energy(self, o, eps): return -0.1
    def set_eri_mo(self, n, eri):
        world = int(os.environ.get("WORLD_SIZE", "1"))
        assert eri is not None or (world > 1 and int(os.environ.get("RANK", "0")) != 0)
    def ccsd_init(self, o, restricted, eps, diis): self.iter = 0; self.o, self.v = o, self.n - o; return -0.1, 0.5
    def ccsd_iterate(self): self.iter += 1; return -0.1 - 0.01 / self.iter, 10.0 ** (-self.iter)
    def ccsd_diis(self): pass
    def ccsd_finalize(self, want_cr=False, want_amplitudes=False, out=None):
        if out is not None:
            assert out[0].size == self.o * self.v and out[1].size == self.o * self.o * self.v * self.v
        if want_amplitudes:
            t2 = np.linspace(-1e-3, 1e-3, (self.o * self.v) ** 2).reshape((self.o, self.o, self.v, self.v), order="F")
            return 0.01 * self.iter, np.full((self.o, self.v), 1e-4 * self.iter), t2
        return 0.01 * self.iter, None, None
    def ccsd_t_spatial(self, paren, renorm, cr): return np.array([-1e-3, -1e-3, 0, 0, 0, 0.0]), 0.0
    def set_partition(self, rank, nranks): self.partition = (rank, nranks)


afesp_b200.AfespGpu = FakeGpu

if __name__ == "__main__":
    import runpy

    sys.argv = [os.path.join(ROOT, "bench.py")] + sys.argv[1:]
    runpy.run_path(os.path.join(ROOT, "bench.py"), run_name="__main__")
