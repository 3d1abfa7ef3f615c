"""Host-side pieces of bench.py that run without a GPU: workload arithmetic, CPU thread selection, the N > 1 watchdog."""
import json
import os
import subprocess
import sys
import textwrap

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import bench  # noqa: E402


def test_code_bytes_match_survey_8d():
    # SURVEY §8d: one matvec moves out * (in / g) * K * ceil(nbits / 8) bytes of codes; Llama-3-8B 1x16 = 1.625 GiB per token
    assert bench.code_bytes(4096, 14336, 1, 16) == 14336 * 512 * 2
    assert bench.code_bytes(4096, 11008, 2, 8) == 11008 * 512 * 2
    assert bench.code_bytes(4096, 11008, 8, 8) == 11008 * 512 * 8
    assert bench.model_code_bytes("llama3-8b", 1, 16, 32) == 1744830464
    per_layer = sum(bench.code_bytes(fin, fout, 1, 16) for _, fin, fout in bench.layer_linears("llama3-70b"))
    assert bench.model_code_bytes("llama3-70b", 1, 16, 80) == 80 * per_layer


def test_host_threads_ignores_torchrun_omp_default(monkeypatch):
    monkeypatch.setenv("OMP_NUM_THREADS", "1")  # what torchrun exports to its workers
    n = bench.host_threads()
    assert 1 <= n <= (os.cpu_count() or 1)
    monkeypatch.setenv("AQLM_BENCH_CPU_THREADS", "3")
    assert bench.host_threads() == 3


def test_watchdog_ends_a_stuck_phase_and_respects_cancel():
    code = textwrap.dedent("""
        import sys, time
        sys.path.insert(0, %r)
        import bench
        w = bench.Watchdog(0, 0.4); w.phase("a"); w.phase("b"); w.cancel(); time.sleep(0.7); print("survived", flush=True)
        off = bench.Watchdog(0, 0.1, enabled=False); off.phase("single GPU"); time.sleep(0.3); print("disabled ok", flush=True)
        w = bench.Watchdog(0, 0.3); w.phase("stuck exchange"); time.sleep(5); print("NOT REACHED", flush=True)
    """ % REPO)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=60)
    assert r.returncode == 5, (r.returncode, r.stderr[-400:])
    lines = r.stdout.strip().splitlines()
    assert lines[:2] == ["survived", "disabled ok"] and "NOT REACHED" not in r.stdout
    err = json.loads(lines[-1])
    assert "stuck exchange" in err["error"] and err["rank"] == 0


def test_dump_outputs_one_float32_file_per_linear(tmp_path):
    import numpy as np
    import torch

    lins = bench.layer_linears("llama3-8b")
    ys = [torch.full((1, fout), float(layer), dtype=torch.float16) for layer in range(3) for _, _, fout in lins]
    bench.dump_outputs(str(tmp_path / "out"), "llama3-8b", ys)
    assert sorted(os.listdir(tmp_path / "out")) == sorted(f"{name}.npy" for name, _, _ in lins)
    for name, _, fout in lins:
        a = np.load(tmp_path / "out" / f"{name}.npy")
        assert a.dtype == np.float32 and a.shape == (3, 1, fout)
        assert a[:, 0, 0].tolist() == [0.0, 1.0, 2.0]


def test_dump_outputs_keeps_a_fixed_layer_subset_under_the_limit(tmp_path, monkeypatch):
    import numpy as np
    import torch

    lins = bench.layer_linears("llama3-8b")
    layer_bytes = 4 * sum(fout for _, _, fout in lins)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 3 * layer_bytes)
    ys = [torch.full((1, fout), float(layer), dtype=torch.float16) for layer in range(9) for _, _, fout in lins]
    bench.dump_outputs(str(tmp_path), "llama3-8b", ys)
    total = sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path))
    assert total <= 3 * layer_bytes + 128 * len(lins)  # + the .npy headers
    for name, _, _ in lins:
        assert np.load(tmp_path / f"{name}.npy")[:, 0, 0].tolist() == [0.0, 4.0, 8.0]


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr
