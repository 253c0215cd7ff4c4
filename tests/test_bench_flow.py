"""Control flow of bench.py's GPU arm on a CPU-only machine, through tests/_bench_stub.py (a fake engine behind the
AfespGpu interface): one rank and two ranks (gloo), the shared-memory host copy of the e2e leg, the target leg, and the
watchdog that must get the headline line out when the target leg stalls.  The numbers mean nothing here; the contract
keys, the single JSON line and the exit status do."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STUB = os.path.join(ROOT, "tests", "_bench_stub.py")
KEYS = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
        "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks", "parity", "target_config"]


def _run(cmd, env_extra, timeout=300):
    env = dict(os.environ, AFESP_BENCH_TARGET_SHAPE="40,4", **env_extra)
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


def test_single_rank_line_with_target_leg():
    d = _run([sys.executable, STUB, "--gpus", "1", "--steps", "2", "--warmup", "1", "--nbf", "36", "--nocc", "4", "--no-cpu"], {})
    for k in KEYS:
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["config"]["nbf"] == 36 and d["higher_is_better"] is False
    assert set(d["config"]) == {"workload", "nbf", "nocc", "calc_type"}       # identical in both arms
    t = d["target_config"]
    assert t["config"]["nbf"] == 40 and t["steps"] == 1 and "e2e" in t and "roofline" in t and "parity" in t
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["roofline"]["traffic_source"] is None or "static" in d["roofline"]["traffic_source"]


def test_watchdog_emits_the_headline_line_when_the_target_leg_stalls():
    d = _run([sys.executable, STUB, "--gpus", "1", "--steps", "1", "--warmup", "1", "--nbf", "36", "--nocc", "4", "--no-cpu"],
             {"AFESP_STUB_STALL": "1", "AFESP_BENCH_TARGET_LIMIT_S": "3"}, timeout=120)
    assert d["value"] > 0 and "did not finish" in d["target_config"]["error"]


def test_two_ranks_gloo_shared_host_copy_and_skipped_target():
    port = 32500 + (os.getpid() % 2000)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), STUB, "--gpus", "2", "--steps", "2", "--warmup", "1", "--nbf", "36", "--nocc", "4",
           "--no-cpu"]
    d = _run(cmd, {})
    assert d["n_gpus"] == 2 and "own PCIe link" in d["e2e"]["what"]       # the shared-memory + sliced-upload mode was taken
    assert "skipped" in d["target_config"] and "exchange" in d
    d = _run(cmd + ["--target", "2"], {})
    assert d["target_config"]["config"]["nbf"] == 40 and d["target_config"]["e2e"]["value"] > 0


def test_parity_block_uses_the_cpu_pins_and_the_pin_file_is_self_consistent():
    """tests/golden/bench_pinned.json at the headline shape: the CPU-computed pins (MP2 by the NumPy oracle; E_CCSD after the
    first iteration by the CPU port; the (T) sum of the first step and the first steps of the trajectory by the CPU port +
    the oracle's BLAS orbit form, tests/golden/make_bench_pins.py) agree with the trajectory a single B200 produced to far
    below the 1e-9 Eh tolerance -- so every bench line's `parity` block ties the GPU numbers at nbf=200 to CPU computations
    of the reference algorithm, not only to an earlier GPU run -- and bench.parity_block reports them."""
    pins = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_pinned.json")))["nbf200_nocc20"]
    steps = pins["steps"]
    assert len(steps) >= 25
    assert abs(pins["e_mp2"] - pins["e_mp2_oracle"]) < 1e-12
    assert abs(steps[0][0] - pins["e_ccsd_iter1_cpu_port"]) < 1e-12
    assert abs(steps[0][1] - pins["e_T_step1_cpu_oracle"]) < 1e-12
    assert len(pins["steps_cpu"]) >= 25
    for cpu, gpu in zip(pins["steps_cpu"], steps):
        assert abs(cpu[0] - gpu[0]) < 1e-11 and abs(cpu[1] - gpu[1]) < 1e-11
    # the target shape: MP2, the first CCSD iteration, the (T) sum of the first step (100 CPU-minutes) and sixteen single-orbit values
    t = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_pinned.json")))["nbf400_nocc40"]
    assert abs(t["e_mp2"] - t["e_mp2_oracle"]) < 1e-12 and abs(t["steps"][0][0] - t["e_ccsd_iter1_cpu_port"]) < 1e-12
    assert abs(t["steps"][0][1] - t["e_T_step1_cpu_oracle"]) < 1e-12          # the full (T) sum over all 11480 orbits
    m = t["mp1_triples"]
    assert m["ntriples"] == 40 * 41 * 42 // 6 and len(m["ranks"]) == len(m["e_T"]) == len(m["ijk"]) >= 5
    assert all(abs(x) < 1e-20 for x, ijk in zip(m["e_T"], m["ijk"]) if ijk[0] == ijk[2]) and min(m["e_T"]) < -1e-7
    # the function the bench uses, fed with the pinned trajectory itself and with a perturbed one
    code = ("import json, sys; sys.argv=['bench.py']; import bench; "
            "p=bench.load_pins()['nbf200_nocc20']; "
            "ok=bench.parity_block(200, 20, p['e_mp2'], p['e_mp1'], [s + [0.0] for s in p['steps']]); "
            "bad=bench.parity_block(200, 20, p['e_mp2'], p['e_mp1'], [[s[0], s[1] + 2e-9, 0.0] for s in p['steps']]); "
            "bench.emit({'ok': ok, 'bad': bad})")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["ok"]["ok"] is True and d["ok"]["steps_compared_with_cpu"] == len(pins["steps_cpu"])
    for key in ("e_mp2_vs_cpu_oracle", "e_ccsd_iter1_vs_cpu_port", "e_T_step1_vs_cpu_oracle", "e_ccsd_vs_cpu_first_steps",
                "e_T_vs_cpu_first_steps", "e_ccsd_max_over_steps", "e_T_max_over_steps"):
        assert key in d["ok"]["abs_diff"], key
    assert d["bad"]["ok"] is False and d["bad"]["abs_diff"]["e_T_step1_vs_cpu_oracle"] > 1e-9


def test_dump_outputs_writes_the_last_timed_step_and_steps_sets_the_step_count(tmp_path):
    """--dump-outputs DIR: float64 .npy files of what the last timed step returned, identical from run to run; the fake
    engine's energy and T1 diagnostic count the iterations since ccsd_init, so they show that exactly W + K steps ran
    before the dump.  At nbf=100/nocc=12 T2 (1115136 elements) is larger than the sample: the fake engine's T2 holds
    ascending values in column-major order, so the sample must be DUMP_T2_SAMPLE of them, distinct and ascending."""
    names = {"ccsd_iterate.npy", "t1_diagnostic.npy", "ccsd_t_sums.npy", "t1.npy", "t2_sample.npy"}
    runs = {}
    for tag, steps, n, o in (("a", 2, 36, 4), ("b", 2, 36, 4), ("c", 5, 36, 4), ("d", 1, 100, 12), ("e", 1, 100, 12)):
        out = tmp_path / tag
        d = _run([sys.executable, STUB, "--gpus", "1", "--steps", str(steps), "--warmup", "1", "--nbf", str(n), "--nocc",
                  str(o), "--no-cpu", "--target", "0", "--dump-outputs", str(out)], {})
        assert d["steps"] == steps and set(os.listdir(out)) == names
        arrs = {nm: np.load(out / nm) for nm in names}
        assert all(a.dtype == np.float64 for a in arrs.values())
        assert sum(a.nbytes for a in arrs.values()) <= 64 << 20
        assert arrs["ccsd_t_sums.npy"].shape == (6,) and arrs["t1.npy"].shape == (o, n - o)
        e, rms = arrs["ccsd_iterate.npy"]
        assert e == d["energies"]["e_ccsd"] and rms == d["energies"]["rms"]
        assert e == -0.1 - 0.01 / (1 + steps)                      # warm-up + timed iterations
        assert arrs["t1_diagnostic.npy"].tolist() == [0.01 * (1 + steps)]
        size = (o * (n - o)) ** 2
        t2 = arrs["t2_sample.npy"]
        if n == 36:
            assert t2.size == size                                 # smaller than the sample: kept whole
        else:
            assert size > 1 << 20 and t2.size == 1 << 20            # bench.DUMP_T2_SAMPLE
            full = np.linspace(-1e-3, 1e-3, size)
            pos = np.rint((t2 + 1e-3) / 2e-3 * (size - 1)).astype(np.int64)
            assert np.all(np.diff(pos) > 0) and np.array_equal(full[pos], t2)
        runs[tag] = arrs
    for a, b in (("a", "b"), ("d", "e")):
        for nm in names:
            assert np.array_equal(runs[a][nm], runs[b][nm]), (a, b, nm)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], cwd=ROOT, capture_output=True,
                       text=True, timeout=120)
    assert r.returncode != 0 and "--steps" in r.stderr


def test_per_triple_check_of_the_target_leg_is_attached_and_cannot_take_the_line_down(tmp_path):
    """bench.mp1_triples_check in the control flow (fake engine, so the numbers disagree): the target leg's parity block
    carries the per-triple comparison and turns false; when the check itself fails the measurements are kept."""
    pins = {"nbf40_nocc4": {"mp1_triples": {"ntriples": 20, "ijk": [[0, 1, 2], [1, 1, 3]], "ranks": [5, 11], "e_T": [-1e-6, -2e-6]}}}
    path = tmp_path / "pins.json"
    path.write_text(json.dumps(pins))
    cmd = [sys.executable, STUB, "--gpus", "1", "--steps", "1", "--warmup", "1", "--nbf", "36", "--nocc", "4", "--no-cpu"]
    d = _run(cmd, {"AFESP_BENCH_PINS": str(path)})
    chk = d["target_config"]["parity"]["mp1_triples_vs_cpu"]
    assert chk["ijk"] == [[0, 1, 2], [1, 1, 3]] and len(chk["e_T_gpu"]) == 2 and chk["ok"] is False
    assert d["target_config"]["parity"]["ok"] is False and d["target_config"]["value"] > 0
    pins["nbf40_nocc4"]["mp1_triples"]["ranks"] = ["not a number"]
    path.write_text(json.dumps(pins))
    d = _run(cmd, {"AFESP_BENCH_PINS": str(path)})
    assert "error" in d["target_config"]["parity"]["mp1_triples_vs_cpu"] and d["target_config"]["value"] > 0
