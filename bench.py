#!/usr/bin/env python
"""bench.py -- AQLM quantized-linear hot path on B200: matvec GB/s (code bytes) & tok/s vs the HBM roofline.

Contract (see DESIGN.md §Measurement):
  python bench.py --gpus N --steps K --warmup W        one JSON line on stdout (rank 0)
  python bench.py ... --dump-outputs DIR               also every linear's output of the last timed step, DIR/<linear>.npy
  python bench.py --impl reference ...                 the reference's OWN CPU code (baseline/_ref, unmodified) on host cores

A "step" is ONE decode-token pass over every quantized linear of the model named in `config.workload`
(q,k,v,o,gate,up,down x n_layers; batch 1; linears only), each linear with its own codes/codebooks/scales so a step
streams the whole model's codes from HBM (1.6 GiB for Llama-3-8B >> 126 MB L2: inputs larger than L2, no flush needed).
  N == 1 : workload = BASELINE.json configs[1], Llama-3-8B 1x16 g8 (override with --workload/--scheme)
  N  > 1 : workload = BASELINE.json configs[4], Llama-3-70B 1x16, every linear sharded along in_features across the N
           ranks, fp32 partials, ONE NCCL all-reduce per linear, scale+bias after the reduce ("strong" scaling).
`value`   = code bytes of the whole model / step time, inputs resident in HBM, step replayed as one CUDA graph.
`e2e`     = same metric through the public module API with the activations coming from pinned HOST memory every
            step (H2D) and the last linear's output read back (D2H), both inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

MODELS = {
    # hidden, intermediate, kv_dim, layers
    "llama3-8b": dict(hidden=4096, inter=14336, kv=1024, layers=32),
    "llama3-70b": dict(hidden=8192, inter=28672, kv=1024, layers=80),
    "llama2-7b": dict(hidden=4096, inter=11008, kv=4096, layers=32),
}


def layer_linears(model: str):
    m = MODELS[model]
    h, i, kv = m["hidden"], m["inter"], m["kv"]
    return [("q_proj", h, h), ("k_proj", h, kv), ("v_proj", h, kv), ("o_proj", h, h), ("gate_proj", h, i),
            ("up_proj", h, i), ("down_proj", i, h)]


def code_bytes(fin, fout, K, nbits, g=8):
    return fout * (fin // g) * K * ((nbits + 7) // 8)


def model_code_bytes(model, K, nbits, n_layers):
    return n_layers * sum(code_bytes(fin, fout, K, nbits) for _, fin, fout in layer_linears(model))


def measured_peaks():
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class Watchdog:
    """N > 1 only: the fused exchange makes kernels of one rank wait for kernels of the others; if a rank never arrives (a bug,
    a dead peer), that wait would spin until the driver's own limit.  The watchdog ends the process instead: it prints which
    phase was stuck (rank 0: as a JSON line on stdout) and leaves through os._exit, which tears the CUDA context down and
    with it the spinning kernel.  Armed per phase; `phase()` re-arms it."""

    def __init__(self, rank, seconds, enabled=True):
        self.rank, self.seconds, self.enabled = rank, float(seconds), enabled and seconds > 0
        self.name, self.timer = "start", None

    def _fire(self):
        msg = {"error": f"watchdog: phase '{self.name}' did not finish within {self.seconds:.0f} s", "rank": self.rank}
        print(f"[bench] {json.dumps(msg)}", file=sys.stderr, flush=True)
        if self.rank == 0:
            print(json.dumps(msg), flush=True)
        os._exit(5)

    def phase(self, name):
        self.cancel()
        self.name = name
        if self.enabled:
            self.timer = threading.Timer(self.seconds, self._fire)
            self.timer.daemon = True
            self.timer.start()

    def cancel(self):
        if self.timer is not None:
            self.timer.cancel()
            self.timer = None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.thread = [], None, None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------------------
# CPU side: the reference's CPU path (oracle C port), used for cpu_baseline and --impl reference
# ------------------------------------------------------------------------------------------------------------
def cpu_layer_sample(model, K, nbits, target_seconds, nthreads=0):
    """Time the oracle's C port of `dequantize_gemm` (reference inference_kernels/dequantization.py:9-21 -- the path
    QuantizedLinear.forward takes on CPU for 1x16, kernel_selector.py:99-102) or, for 256-entry codebooks, of the Numba
    LUT kernel (numba_kernel.py:37-48, kernel_selector.py:95-98) on ONE decoder layer's 7 linears, bs=1, fp32."""
    import numpy as np

    from oracle import c_oracle

    threads = nthreads or c_oracle.num_threads()  # the library build() made: no rebuild here, the tree may be read-only
    rng = np.random.default_rng(0)
    lins = []
    for _, fin, fout in layer_linears(model):
        codes = rng.integers(-(2 ** (nbits - 1)), 2 ** (nbits - 1), size=(fout, fin // 8, K)).astype(
            np.int8 if nbits <= 8 else np.int16)
        cb = rng.standard_normal((K, 2**nbits, 1, 8), dtype=np.float32)
        sc = rng.standard_normal((fout, 1, 1, 1), dtype=np.float32)
        x = rng.standard_normal((1, fin), dtype=np.float32)
        if 2**nbits == 256:  # the reference permutes codes to [in_g, out, K] for its LUT kernel (inference.py:78-83)
            alt = np.ascontiguousarray(np.transpose(codes, (1, 0, 2))).view(np.uint8)
            lins.append(("lut", x, alt, cb, sc))
        else:
            lins.append(("dq", x, codes, cb, sc))
    nbytes = sum(code_bytes(fin, fout, K, nbits) for _, fin, fout in layer_linears(model))

    def one_pass():
        for kind, x, codes, cb, sc in lins:
            if kind == "lut":
                c_oracle.lut_gemv(x[0], codes, cb, sc, threads)
            else:
                c_oracle.dequantize_gemm(x, codes, cb, sc, None, threads)

    one_pass()  # warm-up
    t0 = time.perf_counter()
    one_pass()
    t1 = time.perf_counter() - t0
    reps = max(1, min(50, int(target_seconds / max(t1, 1e-6))))
    t0 = time.perf_counter()
    for _ in range(reps):
        one_pass()
    dt = (time.perf_counter() - t0) / reps
    kernel = "numba_gemm_lut port (oracle/aqlm_oracle.c: aqlm_oracle_lut_gemv)" if 2**nbits == 256 else \
        "dequantize_gemm port (oracle/aqlm_oracle.c: aqlm_oracle_dequantize_gemm)"
    return dict(value=nbytes / dt / 1e9, unit="GB/s", cores=threads, kind="port", seconds_per_layer=dt,
                sample=f"one decoder layer (7 linears, {nbytes / 2**20:.1f} MiB of codes) of {model} {K}x{nbits}, bs=1, fp32, "
                       f"{reps} reps, {kernel}", tok_s=1.0 / (dt * MODELS[model]["layers"]))


REF_DIR = os.path.join(REPO, "baseline", "_ref")


def import_reference_aqlm():
    """The UNMODIFIED reference package, pip-installed into the git-ignored baseline/_ref (it travels to the GPU box).
    Only its CPU path is used here (QuantizedLinear.forward -> dequantize_gemm / numba_gemm_lut); its CUDA extension is
    never imported in this process."""
    if not os.path.isdir(os.path.join(REF_DIR, "aqlm")):
        return None
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import aqlm

    if os.path.abspath(REF_DIR) not in os.path.abspath(aqlm.__file__):
        raise RuntimeError(f"`aqlm` resolved to {aqlm.__file__}, not the reference in {REF_DIR}")
    return aqlm


def host_threads():
    """Threads for the CPU legs: the physical cores this process may run on (torch's own default when OMP_NUM_THREADS is
    unset).  torchrun exports OMP_NUM_THREADS=1 to its workers, which would silently turn the N > 1 reference arm into a
    single-thread run; the reference arm is meant to use the host cores it can (AQLM_BENCH_CPU_THREADS overrides)."""
    forced = int(os.environ.get("AQLM_BENCH_CPU_THREADS", "0") or 0)
    if forced > 0:
        return forced
    try:
        logical = len(os.sched_getaffinity(0))
    except AttributeError:
        logical = os.cpu_count() or 1
    physical = set()
    try:
        phys = "0"
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("physical id"):
                    phys = ln.split(":", 1)[1].strip()
                elif ln.startswith("core id"):
                    physical.add((phys, ln.split(":", 1)[1].strip()))
    except OSError:
        pass
    return max(1, min(logical, len(physical) or logical))


def cpu_reference_layer_sample(model, K, nbits, target_seconds, numba_threads=1):
    """Time the reference's own `QuantizedLinear.forward` on CPU (inference_lib/src/aqlm/inference.py:68-75) on ONE decoder
    layer's 7 linears, bs=1, fp32 (the dtype of benchmark/matmul_benchmark_cpu.py:114-123).  1x16 resolves to
    `dequantize_gemm` (kernel_selector.py:99-102; torch intra-op threads = all cores); 256-entry codebooks resolve to the
    Numba LUT kernel (kernel_selector.py:95-98, numba_kernel.py:10-65) with NUMBA_NUM_THREADS=1, the reference benchmark's
    default (`--nthreads 1`) and the only race-free setting.  Returns None when baseline/_ref is absent."""
    lut = 2**nbits == 256
    if lut:
        os.environ.setdefault("NUMBA_NUM_THREADS", str(numba_threads))
    try:
        aqlm = import_reference_aqlm()
    except Exception as e:
        print(f"[bench] reference package unusable ({type(e).__name__}: {e}); falling back to the oracle port", file=sys.stderr)
        return None
    if aqlm is None:
        return None
    import torch

    if not lut and torch.get_num_threads() < host_threads():
        torch.set_num_threads(host_threads())  # e.g. under torchrun, which sets OMP_NUM_THREADS=1 for its workers
    torch.manual_seed(0)
    lo, hi = (-128, 128) if nbits <= 8 else (-(2 ** (nbits - 1)), 2 ** (nbits - 1))
    mods = []
    for _, fin, fout in layer_linears(model):
        m = aqlm.QuantizedLinear(fin, fout, 8, 1, K, nbits, bias=False, dtype=torch.float32)
        m.codes.data = torch.randint(lo, hi, m.codes.shape, dtype=m.codes.dtype)
        m.codebooks.data = torch.randn(m.codebooks.shape)
        m.scales.data = torch.randn(m.scales.shape)
        mods.append((m, torch.randn(1, fin)))
    nbytes = sum(code_bytes(fin, fout, K, nbits) for _, fin, fout in layer_linears(model))

    def one_pass():
        with torch.no_grad():
            for m, x in mods:
                m(x)

    one_pass()  # warm-up: TorchScript / Numba JIT, the reference's lazy code permutation (inference.py:78-83)
    t0 = time.perf_counter()
    one_pass()
    t1 = time.perf_counter() - t0
    reps = max(1, min(50, int(target_seconds / max(t1, 1e-6))))
    t0 = time.perf_counter()
    for _ in range(reps):
        one_pass()
    dt = (time.perf_counter() - t0) / reps
    cores = numba_threads if lut else torch.get_num_threads()
    kernel = ("aqlm.inference_kernels.numba_kernel.numba_gemm_lut (baseline/_ref, NUMBA_NUM_THREADS=%d)" % numba_threads) if lut \
        else "aqlm.inference_kernels.dequantization.dequantize_gemm (baseline/_ref, torch CPU ops)"
    return dict(value=nbytes / dt / 1e9, unit="GB/s", cores=cores, kind="reference", seconds_per_layer=dt,
                sample=f"one decoder layer (7 linears, {nbytes / 2**20:.1f} MiB of codes) of {model} {K}x{nbits}, bs=1, fp32, "
                       f"{reps} reps through the reference's own QuantizedLinear.forward on CPU: {kernel}",
                tok_s=1.0 / (dt * MODELS[model]["layers"]))


def cpu_baseline_sample(model, K, nbits, target_seconds):
    """cpu_baseline object: the reference's own CPU code when baseline/_ref is present (kind "reference"), with the
    oracle's C port (all cores) reported beside it; the port alone (kind "port") otherwise."""
    ref = cpu_reference_layer_sample(model, K, nbits, target_seconds)
    port = cpu_layer_sample(model, K, nbits, target_seconds=min(target_seconds, 8.0))
    if ref is None:
        return port
    ref["port"] = {k: port[k] for k in ("value", "unit", "cores", "kind", "sample")}
    return ref


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path -- the UNMODIFIED package in baseline/_ref,
    through its public module API (`aqlm.QuantizedLinear.forward` on CPU tensors) -- on the box's host cores; a bounded
    sample per step = one decoder layer.  Falls back to the oracle port only when baseline/_ref is not installed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    K, nbits = (int(v) for v in args.scheme.split("x"))
    model = args.workload or ("llama3-8b" if args.gpus == 1 else "llama3-70b")
    steps = max(1, args.steps)
    budget = 150.0  # seconds for all steps
    base = cpu_baseline_sample(model, K, nbits, target_seconds=min(20.0, budget / 4))
    per = base["seconds_per_layer"]
    steps_run = max(1, min(steps, int(budget / max(per, 1e-6))))
    cpu = {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if "port" in base:
        cpu["port"] = base["port"]
    line = {
        "impl": "reference", "metric": "aqlm_matvec_code_GBps", "value": base["value"], "unit": "GB/s",
        "n_gpus": args.gpus, "steps": steps_run, "warmup": args.warmup, "ms_per_step": per * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "tok_s_linears_only": base["tok_s"],
        "config": {"workload": f"{model} {K}x{nbits} g8 all-linear matvec sweep, bs=1",
                   "step": "bounded sample: ONE decoder layer (7 linears) per step on host cores"},
        "cpu_baseline": cpu,
        "e2e": {"value": base["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------------------
def build_model(model, K, nbits, n_layers, device, rank, world, peer_comm=None):
    """Random-init modules of the named architecture's linears (no checkpoints offline): per layer a list of
    (module, in_features_local)."""
    import torch

    import aqlm_b200
    from aqlm_b200.sharded import ShardedQuantizedLinear

    gen = torch.Generator(device=device).manual_seed(1234 + rank)
    lo, hi = (-128, 128) if nbits <= 8 else (-(2 ** (nbits - 1)), 2 ** (nbits - 1))
    layers = []
    for _ in range(n_layers):
        mods = []
        for _, fin, fout in layer_linears(model):
            if world == 1:
                m = aqlm_b200.QuantizedLinear(fin, fout, 8, 1, K, nbits, bias=False, device=device, dtype=torch.float16)
                local_groups = fin // 8
            else:
                m = ShardedQuantizedLinear(fin, fout, 8, 1, K, nbits, bias=False, rank=rank, world_size=world,
                                           device=device, dtype=torch.float16, peer_comm=peer_comm)
                local_groups = fin // 8 // world
            m.codes.data = torch.randint(lo, hi, (fout, local_groups, K), dtype=m.codes.dtype, device=device, generator=gen)
            m.codebooks.data = torch.randn((K, 2**nbits, 1, 8), dtype=torch.float16, device=device, generator=gen)
            m.scales.data = (0.75 + 0.5 * torch.rand((fout, 1, 1, 1), device=device, generator=gen)).half()
            mods.append((m, local_groups * 8))
        layers.append(mods)
    return layers


DUMP_LIMIT_BYTES = 64 * 2**20


def dump_outputs(out_dir, model, ys):
    """`--dump-outputs`: what one timed step returned to its caller, so that two builds can be compared output for output.
    `ys` holds every linear's output of the step, layer after layer in layer_linears order; each linear is written as
    `<out_dir>/<name>.npy`, float32 [layers, batch, out_features].  When the whole step exceeds DUMP_LIMIT_BYTES (only with
    a large `--layers`), a fixed, evenly spaced subset of the layers is written instead."""
    import numpy as np

    names = [name for name, _, _ in layer_linears(model)]
    per_layer = [ys[i:i + len(names)] for i in range(0, len(ys), len(names))]
    layer_bytes = 4 * sum(y.numel() for y in per_layer[0])
    keep = max(1, min(len(per_layer), DUMP_LIMIT_BYTES // layer_bytes))
    idx = np.unique(np.linspace(0, len(per_layer) - 1, keep).round().astype(int))
    os.makedirs(out_dir, exist_ok=True)
    for j, name in enumerate(names):
        arr = np.stack([per_layer[i][j].float().cpu().numpy() for i in idx])
        np.save(os.path.join(out_dir, f"{name}.npy"), arr)


def group_layers(layers, K, nbits, world):
    """q/k/v and gate/up read the same activation: run each set as ONE grouped launch (and one exchange when sharded).
    Returns per layer a list of (callable, in_features_local)."""
    from aqlm_b200.grouped import QuantizedLinearGroup, ShardedQuantizedLinearGroup

    out = []
    for mods in layers:
        ms = [m for m, _ in mods]
        n_h, n_i = mods[0][1], mods[6][1]
        if (K, nbits) == (1, 16):
            G = QuantizedLinearGroup if world == 1 else ShardedQuantizedLinearGroup
            out.append([(G(ms[0:3]), n_h), (ms[3], n_h), (G(ms[4:6]), n_h), (ms[6], n_i)])
        else:
            out.append([(m, n) for m, n in mods])
    return out


def sharded_parity(model, K, nbits, device, rank, world, peer_comm):
    """Driver-visible correctness of the multi-GPU data path (run before timing, N > 1): every distinct linear shape of the
    workload goes once through the sharded path -- the fused peer-memory exchange AND the NCCL all-reduce variant, plus the
    grouped q/k/v and gate/up launches the timed step uses -- and is compared with the UNSHARDED single-GPU module on the
    same full tensors (metric of matmul_benchmark.py:108); one shape is also checked against the C oracle (rank 0).
    Every rank builds identical full tensors from a shared seed and keeps its in_features slice."""
    import torch
    import torch.distributed as dist

    import aqlm_b200
    from aqlm_b200.grouped import ShardedQuantizedLinearGroup
    from aqlm_b200.sharded import ShardedQuantizedLinear

    lo, hi = (-128, 128) if nbits <= 8 else (-(2 ** (nbits - 1)), 2 ** (nbits - 1))
    lin = {name: (fin, fout) for name, fin, fout in layer_linears(model)}

    def full(fin, fout, seed):
        g = torch.Generator(device=device).manual_seed(seed)
        return dict(codes=torch.randint(lo, hi, (fout, fin // 8, K), dtype=torch.int8 if nbits <= 8 else torch.int16,
                                        device=device, generator=g),
                    codebooks=torch.randn((K, 2**nbits, 1, 8), dtype=torch.float16, device=device, generator=g),
                    scales=(0.75 + 0.5 * torch.rand((fout, 1, 1, 1), device=device, generator=g)).half(),
                    x=torch.randn((1, fin), dtype=torch.float16, device=device, generator=g))

    def unsharded(t):
        m = aqlm_b200.QuantizedLinear(t["codes"].shape[1] * 8, t["codes"].shape[0], 8, 1, K, nbits, bias=False, device=device,
                                      dtype=torch.float16)
        m.codes.data, m.codebooks.data, m.scales.data = t["codes"], t["codebooks"], t["scales"]
        return m(t["x"]).float()

    def rel(y, ref):
        return float(((y.float() - ref).abs().mean() / ref.abs().mean()).item())

    worst, shapes, oracle_rel = 0.0, [], None
    distinct = sorted({v for v in lin.values()})
    for i, (fin, fout) in enumerate(distinct):
        t = full(fin, fout, 4242 + i)
        ref = unsharded(t)
        for kind, comm in (("peer", peer_comm), ("nccl", None)):
            if kind == "peer" and comm is None:
                continue
            m = ShardedQuantizedLinear.from_full(t["codes"], t["codebooks"], t["scales"], None, rank=rank, world_size=world,
                                                 peer_comm=comm)
            for _ in range(2):  # second call exercises the step counter / buffer-set alternation
                y = m(t["x"])
            e = rel(y, ref)
            worst = max(worst, e)
            shapes.append({"shape": f"{fin}x{fout}", "exchange": kind, "rel": e})
            del m
        if i == 0 and rank == 0:
            try:
                from oracle import c_oracle

                f32 = lambda a: a.float().cpu().numpy()  # noqa: E731
                yo = c_oracle.dequantize_gemm(f32(t["x"]), t["codes"].cpu().numpy(), f32(t["codebooks"]), f32(t["scales"]), None)
                oracle_rel = rel(y, torch.from_numpy(yo).to(device))
                worst = max(worst, oracle_rel)
            except Exception as e:  # the checker must not take the bench down; its absence is reported
                oracle_rel = f"unavailable: {type(e).__name__}: {e}"
        del t, ref
    if (K, nbits) == (1, 16):
        for names in (("q_proj", "k_proj", "v_proj"), ("gate_proj", "up_proj")):
            ts = [full(*lin[n], 5151 + j) for j, n in enumerate(names)]
            for t in ts[1:]:
                t["x"] = ts[0]["x"]
            refs = [unsharded(t) for t in ts]
            ms = [ShardedQuantizedLinear.from_full(t["codes"], t["codebooks"], t["scales"], None, rank=rank, world_size=world,
                                                   peer_comm=peer_comm) for t in ts]
            grp = ShardedQuantizedLinearGroup(ms)
            for _ in range(2):
                ys = grp(ts[0]["x"])
            for n, y, ref in zip(names, ys, refs):
                e = rel(y, ref)
                worst = max(worst, e)
                shapes.append({"shape": f"{lin[n][0]}x{lin[n][1]}", "exchange": "grouped " + ("peer" if peer_comm is not None else "nccl"),
                               "rel": e})
            del ts, refs, ms, grp
    torch.cuda.synchronize()
    w = torch.tensor([worst], device=device)
    dist.all_reduce(w, op=dist.ReduceOp.MAX)  # a rank that saw a wrong result fails everyone
    torch.cuda.empty_cache()
    return {"max_rel": float(w.item()), "tolerance": 1e-3, "vs": "unsharded single-GPU aqlm_b200.QuantizedLinear on the same full tensors",
            "c_oracle_rel_first_shape": oracle_rel, "shapes": shapes}


def _json_lines(text):
    rows = []
    for ln in text.splitlines():
        ln = ln.strip()
        if ln.startswith("{"):
            try:
                rows.append(json.loads(ln))
            except Exception:
                pass
    return rows


def _tool(argv, timeout):
    """Run a tools/ script in its own process (the reference and aqlm_b200 both register `aqlm::` ops) and parse its
    JSON lines; errors are reported, never raised."""
    try:
        r = subprocess.run([sys.executable, *argv], capture_output=True, text=True, timeout=timeout, cwd=REPO)
        rows = _json_lines(r.stdout)
        if r.returncode != 0 and not rows:
            return {"error": f"exit {r.returncode}: {r.stderr[-400:]}"}
        return rows
    except subprocess.TimeoutExpired:
        return {"error": f"timeout after {timeout}s"}
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}


def secondary_metrics(device, peak_hbm, args):
    """Extra measurements reported beside the headline (not part of `value`): the fused dequant + tcgen05 GEMM (BASELINE
    configs[3]), the Kx8 matvec on every Llama-2-7B shape (configs[2]), the other schemes of SURVEY §8 f4 (1x8, 1x16 g=16,
    bf16), the reference's own CUDA kernels and Numba CPU kernel timed in the same job, and HF `generate` tok/s (§8 f1).
    Matvec/GEMM numbers: CUDA-graph replay over rotating weight copies (codes come from HBM), CUDA events."""
    import torch

    from aqlm_b200.inference_kernels import cuda_kernel

    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            tpeak = float(json.load(f)["bf16_tflops"])
    except Exception:
        tpeak = 1590.0

    def timed(fns, iters=10):
        for f in fns:
            f()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for f in fns:
                f()
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            g.replay()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) * 1e3 / iters / len(fns)  # us per call

    def weights(fin, fout, K, nbits, copies, dt, g=8):
        ws = []
        for _ in range(copies):
            lo, hi = (-128, 128) if nbits <= 8 else (-32768, 32768)
            codes = torch.randint(lo, hi, (fout, fin // g, K), dtype=torch.int8 if nbits <= 8 else torch.int16, device=device)
            cb = torch.randn((K, 2**nbits, 1, g), dtype=dt, device=device)
            sc = (0.75 + 0.5 * torch.rand((fout, 1, 1, 1), device=device)).to(dt)
            ws.append((codes, cb, sc))
        return ws

    out = {"gemm": [], "kx8_matvec": [], "other_schemes_matvec": []}
    for fin, fout in ((4096, 14336), (4096, 4096)):
        for dt, name in ((torch.float16, "f16"), (torch.bfloat16, "bf16")):
            if (fin, fout) == (4096, 4096) and name == "f16":
                continue
            ws = weights(fin, fout, 1, 16, 12 if fout > 4096 else 32, dt)
            for bs in ((16, 64, 256) if fout > 4096 else (256,)):
                x = torch.randn((bs, fin), dtype=dt, device=device)
                us = timed([(lambda w=w: cuda_kernel.matmat_dequant(x, w[0], w[1], w[2], None)) for w in ws])
                tf = 2.0 * bs * fin * fout / us / 1e6
                cgb = code_bytes(fin, fout, 1, 16) / us / 1e3  # SURVEY §8d: small batches are gather/HBM-bound -- report both
                out["gemm"].append({"shape": f"{fin}x{fout}", "scheme": "1x16", "batch": bs, "operands": name, "us": round(us, 2),
                                    "tflops": round(tf, 1), "frac_of_measured_bf16_peak": round(tf / tpeak, 4),
                                    "code_GBps": round(cgb, 1), "frac_of_hbm_peak": round(cgb / peak_hbm, 4)})
            del ws
    # backward op (fused dequant-transpose GEMM, SURVEY §8 f3): grad_in[bs, in] = (grad_out * scales) @ W
    try:
        ws = weights(4096, 14336, 1, 16, 12, torch.float16)
        go = torch.randn((256, 14336), dtype=torch.float16, device=device)
        us = timed([(lambda w=w: cuda_kernel.matmat_dequant_transposed(go, w[0], w[1], w[2], None)) for w in ws])
        tf = 2.0 * 256 * 4096 * 14336 / us / 1e6
        out["gemm_transposed"] = [{"shape": "14336->4096 (W 4096x14336)", "scheme": "1x16", "batch": 256, "us": round(us, 2),
                                   "tflops": round(tf, 1), "frac_of_measured_bf16_peak": round(tf / tpeak, 4)}]
        del ws, go
    except Exception as e:
        out["gemm_transposed"] = {"error": f"{type(e).__name__}: {e}"}
    kx8 = [(2, (4096, 11008)), (2, (11008, 4096)), (2, (4096, 4096)), (8, (4096, 11008)), (8, (11008, 4096)), (8, (4096, 4096)),
           (1, (4096, 11008))]
    for K, (fin, fout) in kx8:
        cb = fout * (fin // 8) * K
        ws = weights(fin, fout, K, 8, max(2, min(40, 300 * 2**20 // cb)), torch.float16)
        x = torch.randn((1, fin), dtype=torch.float16, device=device)
        us = timed([(lambda w=w: cuda_kernel.matmat(x, w[0], w[1], w[2], None)) for w in ws])
        out["kx8_matvec"].append({"shape": f"{fin}x{fout}", "scheme": f"{K}x8", "us": round(us, 2),
                                  "code_GBps": round(cb / us / 1e3, 1), "frac_of_hbm_peak": round(cb / us / 1e3 / peak_hbm, 4)})
        del ws
    for label, K, nbits, g, dt, (fin, fout) in (("1x16 g16 f16", 1, 16, 16, torch.float16, (4096, 14336)),
                                                ("1x16 g8 bf16", 1, 16, 8, torch.bfloat16, (4096, 14336)),
                                                ("2x8 g8 bf16", 2, 8, 8, torch.bfloat16, (4096, 11008))):
        cb = fout * (fin // g) * K * (2 if nbits > 8 else 1)
        ws = weights(fin, fout, K, nbits, max(2, min(40, 300 * 2**20 // cb)), dt, g)
        x = torch.randn((1, fin), dtype=dt, device=device)
        us = timed([(lambda w=w: cuda_kernel.matmat(x, w[0], w[1], w[2], None)) for w in ws])
        out["other_schemes_matvec"].append({"case": label, "shape": f"{fin}x{fout}", "us": round(us, 2),
                                            "code_GBps": round(cb / us / 1e3, 1),
                                            "frac_of_hbm_peak": round(cb / us / 1e3 / peak_hbm, 4)})
        del ws
    out["tensor_peak_tflops"] = tpeak
    torch.cuda.empty_cache()
    if not args.skip_reference_gpu and os.path.isdir(os.path.join(REF_DIR, "aqlm")):
        # the reference's stock CUDA kernels (baseline/_ref, JIT-built for sm_100) with the same timing protocol
        out["reference_gpu"] = _tool([os.path.join("tools", "compare_reference_gpu.py"), "--cases", "quick"], timeout=420)
        out["generate"] = {
            "ours_fused": _tool([os.path.join("tools", "generate_benchmark.py"), "--impl", "ours", "--fuse", "--output_length", "64",
                                 "--benchmark_iters", "2"], timeout=300),
            "ours": _tool([os.path.join("tools", "generate_benchmark.py"), "--impl", "ours", "--output_length", "64",
                           "--benchmark_iters", "2"], timeout=300),
            "reference": _tool([os.path.join("tools", "generate_benchmark.py"), "--impl", "reference", "--output_length", "64",
                                "--benchmark_iters", "2"], timeout=420),
        }
    if not args.skip_cpu:
        # the reference's Numba LUT kernel (benchmark/matmul_benchmark_cpu.py times this algorithm) on one Llama-2-7B layer, 2x8
        try:
            ref = cpu_reference_layer_sample("llama2-7b", 2, 8, target_seconds=6.0)
            if ref is not None:
                out["reference_cpu_numba_2x8"] = {k: ref[k] for k in ("value", "unit", "cores", "kind", "sample")}
        except Exception as e:
            out["reference_cpu_numba_2x8"] = {"error": f"{type(e).__name__}: {e}"}
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    from aqlm_b200 import _cabi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    K, nbits = (int(v) for v in args.scheme.split("x"))
    model = args.workload or ("llama3-8b" if world == 1 else "llama3-70b")
    n_layers = args.layers or MODELS[model]["layers"]
    total_bytes = model_code_bytes(model, K, nbits, n_layers)
    peak, peak_src = measured_peaks()

    wd = Watchdog(rank, args.watchdog_seconds, enabled=world > 1)
    wd.phase("communicator setup")
    peer_comm, reduce_kind = None, "none"
    if world > 1:
        reduce_kind = "nccl all-reduce + epilogue kernel"
        if os.environ.get("AQLM_B200_ALLREDUCE", "peer") == "peer":
            try:
                from aqlm_b200.peer import PeerComm

                peer_comm = PeerComm(max_elems=MODELS[model]["inter"] * 4)
                reduce_kind = ("exchange fused INTO the GEMV kernel over NVLink peer memory (tagged 64-bit {fp32, step} words pushed with P2P stores, LL-style: no fence/flag/barrier, csrc/gemv.cuh PEER)"
                               if os.environ.get("AQLM_B200_FUSED_EXCHANGE", "1") != "0" else
                               "partial GEMV + fused peer-memory exchange/epilogue kernel (csrc/peer_allreduce.cuh)")
            except Exception as e:
                print(f"[bench] peer-memory communicator unavailable ({type(e).__name__}: {e}); using NCCL", file=sys.stderr)
                peer_comm = None
    parity = None
    if world > 1 and not args.skip_parity:
        wd.phase("sharded_parity (first use of the exchange at this N)")
        parity = sharded_parity(model, K, nbits, device, rank, world, peer_comm)
        if parity["max_rel"] > parity["tolerance"]:
            if rank == 0:
                print(json.dumps({"error": "sharded_parity failed", "sharded_parity": parity}), flush=True)
            torch.cuda.synchronize()
            dist.barrier()
            os._exit(3)
    wd.phase("model build, first steps, graph capture")
    layers = build_model(model, K, nbits, n_layers, device, rank, world, peer_comm)
    grouped = not args.no_group and (K, nbits) == (1, 16)
    if grouped:
        layers = group_layers(layers, K, nbits, world)
    in_sizes = sorted({n for mods in layers for _, n in mods})
    gen_x = torch.Generator(device=device).manual_seed(99)
    x_dev = {n: torch.randn((1, n), dtype=torch.float16, device=device, generator=gen_x) for n in in_sizes}
    x_host = {n: torch.randn((1, n), dtype=torch.float16).pin_memory() for n in in_sizes}
    outs = {}

    def step():
        ys = []
        for mods in layers:
            for m, n in mods:
                y = m(x_dev[n])
                ys.extend(y if isinstance(y, tuple) else (y,))
        outs["all"] = ys  # every linear's output, in layer_linears order per layer
        outs["y"] = ys[-1]

    # bind kernels / NCCL outside capture, count launches of one step
    step()
    torch.cuda.synchronize()
    c0 = _cabi.launch_count()
    step()
    torch.cuda.synchronize()
    launches_per_step = _cabi.launch_count() - c0

    graph, use_graph = None, not args.no_graph
    if use_graph:
        try:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                step()
        except Exception as e:  # e.g. a collective that cannot be captured on this stack
            print(f"[bench] graph capture failed ({type(e).__name__}: {e}); running eagerly", file=sys.stderr)
            graph, use_graph = None, False
            torch.cuda.synchronize()
    run = graph.replay if use_graph else step

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        barrier()
        ms = a.elapsed_time(b)
        if world > 1:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    wd.phase("warm-up and timed steps")
    for _ in range(max(3, args.warmup)):
        run()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms_total = timed(run, args.steps)
    ms_step = ms_total / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, outs["all"])

    # ---- e2e: pinned-host activations in, last output out, every step ---------------------------------
    y_host = torch.empty_like(outs["y"], device="cpu").pin_memory()
    h2d = sum(x_host[n].numel() * 2 for n in in_sizes)
    d2h = y_host.numel() * 2

    def e2e_step():
        for n in in_sizes:
            x_dev[n].copy_(x_host[n], non_blocking=True)
        run()
        y_host.copy_(outs["y"], non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the caller reads the result

    for _ in range(3):
        e2e_step()
    ms_e2e = timed(e2e_step, args.steps) / args.steps
    clocks = sampler.stop() if sampler else None

    # ---- N > 1, reported beside the headline: the Megatron-style pairing (VERDICT r1 item 6) --------------------------
    # q/k/v and gate/up sharded along OUT_features (each rank owns rows, no exchange: their consumers are sharded the same
    # way), o_proj and down_proj sharded along in_features with ONE exchange each: 2 exchanges per layer instead of 4.
    # ---- N > 1: compute vs exchange split (SURVEY §8e).  The exchange lives inside the GEMV kernel, so the split is measured
    # by difference: the same step with every linear's GEMV writing its UNSCALED fp32 partials and no exchange at all
    # (matmat_partial / the grouped partial launch).  Local to each rank (no collective in this leg: a rank-local failure
    # cannot strand the others); rank 0 reports its own clock.
    compute_only = None
    if world > 1:
        wd.phase("compute-only step (no exchange)")
        try:
            from aqlm_b200.grouped import ShardedQuantizedLinearGroup as _SGroup
            from aqlm_b200.inference_kernels import cuda_kernel as _ck

            def cstep():
                for mods in layers:
                    for m, n in mods:
                        if isinstance(m, _SGroup):
                            _ck.matmat_grouped(x_dev[n], m._fused_codes, m._fused_codebooks, None, None, m.seg_rows, partial=True)
                        else:
                            _ck.matmat_partial(x_dev[n], m.codes, m.codebooks)

            cstep()
            torch.cuda.synchronize()
            gc = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gc):
                cstep()
            for _ in range(3):
                gc.replay()
            torch.cuda.synchronize()
            n_it = max(5, args.steps // 2)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(n_it):
                gc.replay()
            ev1.record()
            torch.cuda.synchronize()
            ms_c = ev0.elapsed_time(ev1) / n_it
            compute_only = {"ms_per_step_compute_only": ms_c, "ms_per_step_with_exchange": ms_step,
                            "exchange_share_of_step": max(0.0, 1.0 - ms_c / ms_step),
                            "compute_only_value": total_bytes / (ms_c * 1e-3) / 1e9, "unit": "GB/s",
                            "note": "same sharded step, every GEMV writing unscaled fp32 partials, no exchange; rank 0's clock"}
            gc.reset()
            del gc
        except Exception as e:
            compute_only = {"error": f"{type(e).__name__}: {e}"}
            try:
                torch.cuda.synchronize()
            except Exception:
                pass

    wd.phase("pairing variant / same-workload single-GPU point")
    pairing = None
    if world > 1 and (K, nbits) == (1, 16) and not args.skip_pairing:
        try:
            import aqlm_b200
            from aqlm_b200.grouped import QuantizedLinearGroup
            from aqlm_b200.sharded import ShardedQuantizedLinear

            gen = torch.Generator(device=device).manual_seed(4321 + rank)
            lin = {name: (fin, fout) for name, fin, fout in layer_linears(model)}

            def rows_shard(name):
                fin, fout = lin[name]
                m = aqlm_b200.QuantizedLinear(fin, fout // world, 8, 1, K, nbits, bias=False, device=device, dtype=torch.float16)
                m.codes.data = torch.randint(-32768, 32768, m.codes.shape, dtype=torch.int16, device=device, generator=gen)
                m.codebooks.data = torch.randn(m.codebooks.shape, dtype=torch.float16, device=device, generator=gen)
                m.scales.data = (0.75 + 0.5 * torch.rand(m.scales.shape, device=device, generator=gen)).half()
                return m

            def cols_shard(name):
                fin, fout = lin[name]
                m = ShardedQuantizedLinear(fin, fout, 8, 1, K, nbits, bias=False, rank=rank, world_size=world, device=device,
                                           dtype=torch.float16, peer_comm=peer_comm)
                m.codes.data = torch.randint(-32768, 32768, m.codes.shape, dtype=torch.int16, device=device, generator=gen)
                m.codebooks.data = torch.randn(m.codebooks.shape, dtype=torch.float16, device=device, generator=gen)
                m.scales.data = (0.75 + 0.5 * torch.rand(m.scales.shape, device=device, generator=gen)).half()
                return m

            h, inter = MODELS[model]["hidden"], MODELS[model]["inter"]
            pl = []
            for _ in range(n_layers):
                pl.append([(QuantizedLinearGroup([rows_shard("q_proj"), rows_shard("k_proj"), rows_shard("v_proj")]), h),
                           (cols_shard("o_proj"), h // world),
                           (QuantizedLinearGroup([rows_shard("gate_proj"), rows_shard("up_proj")]), h),
                           (cols_shard("down_proj"), inter // world)])
            xs = {n: torch.randn((1, n), dtype=torch.float16, device=device) for n in {n for mods in pl for _, n in mods}}

            def pstep():
                for mods in pl:
                    for m, n in mods:
                        m(xs[n])
            pstep()
            torch.cuda.synchronize()
            gp = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gp):
                pstep()
            for _ in range(3):
                gp.replay()
            ms_p = timed(gp.replay, max(5, args.steps // 2)) / max(5, args.steps // 2)
            pairing = {"value": total_bytes / (ms_p * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": ms_p,
                       "layout": "q/k/v and gate/up sharded along out_features (no exchange), o_proj and down_proj along "
                                 "in_features with one fused exchange each: 2 exchanges per layer"}
            gp.reset()
            del pl, gp, xs
            torch.cuda.empty_cache()
        except Exception as e:
            pairing = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.synchronize()

    # single-GPU point of the SAME workload when N > 1: rank 0 alone, unsharded, same grouping, FULL depth (Llama-3-70B
    # 1x16 is 16 GiB of codes: fits beside the shard), so the driver's curve can be read as same-workload strong scaling
    same_n1 = None
    if world > 1 and rank == 0 and not args.skip_n1:
        try:
            l1 = build_model(model, K, nbits, n_layers, device, 0, 1)
            if grouped:
                l1 = group_layers(l1, K, nbits, 1)
            xs = {n: torch.randn((1, n), dtype=torch.float16, device=device) for n in {n for mods in l1 for _, n in mods}}

            def s1():
                for mods in l1:
                    for m, n in mods:
                        m(xs[n])
            s1()
            g1 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g1):
                s1()
            for _ in range(3):
                g1.replay()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(5):
                g1.replay()
            b.record()
            torch.cuda.synchronize()
            v1 = total_bytes / (a.elapsed_time(b) / 5 * 1e-3) / 1e9
            same_n1 = {"value": v1, "unit": "GB/s",
                       "note": f"rank 0 alone, unsharded, {n_layers} layers, {'grouped' if grouped else 'ungrouped'} launches"}
            del l1, g1, xs
            torch.cuda.empty_cache()
        except Exception as e:
            same_n1 = {"error": f"{type(e).__name__}: {e}"}
    if world > 1:
        dist.barrier()
    wd.cancel()

    if rank == 0:
        value = total_bytes / (ms_step * 1e-3) / 1e9
        e2e_value = total_bytes / (ms_e2e * 1e-3) / 1e9
        n_lin = n_layers * (4 if grouped else 7)
        per_gpu_bytes = total_bytes / world
        avg_launch_us = ms_step * 1e3 / n_lin
        achieved = per_gpu_bytes / n_lin / (avg_launch_us * 1e-6) / 1e9
        cpu = None
        if world == 1 and not args.skip_cpu:
            cpu_full = cpu_baseline_sample(model, K, nbits, target_seconds=15.0)
            cpu = {k: cpu_full[k] for k in ("value", "unit", "cores", "kind", "sample")}
            if "port" in cpu_full:
                cpu["port"] = cpu_full["port"]
        traffic = None
        tpath = os.path.join(REPO, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):
            try:
                with open(tpath) as f:
                    key = f"{model}:{K}x{nbits}:bytes_per_launch" if world == 1 else f"{model}:{K}x{nbits}:n{world}:bytes_per_launch"
                    traffic = json.load(f).get(key)
            except Exception:
                traffic = None
        line = {
            "metric": "aqlm_matvec_code_GBps", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "tok_s_linears_only": 1e3 / ms_step,
            "config": {"workload": f"{model} {K}x{nbits} g8 all-linear matvec sweep, bs=1, {n_layers} layers x 7 linears",
                       "parallelism": "single GPU" if world == 1 else f"in_features-sharded x{world}, one exchange per linear: {reduce_kind}",
                       "l2_policy": f"inputs larger than L2: {total_bytes / world / 2**20:.0f} MiB of distinct codes per GPU per step",
                       "cuda_graph": bool(use_graph), "code_bytes_per_step": total_bytes,
                       "grouped_launches": "q/k/v and gate/up each run as ONE grouped launch (QuantizedLinearGroup): 4 launches per layer"
                       if grouped else "one launch per linear (7 per layer)"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src,
                         "kernel": "gemv (fused code-gather + dequant + dot), avg over the step's launches incl. launch gaps",
                         "avg_launch_us": avg_launch_us, "algorithmic_bytes_per_launch": per_gpu_bytes / n_lin},
            "e2e": {"value": e2e_value, "unit": "GB/s", "ms_per_step": ms_e2e, "tok_s_linears_only": 1e3 / ms_e2e,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "aqlm_b200.QuantizedLinear.forward per linear (CUDA-graph replay), pinned host in/out"},
            "gpu_launches": int(launches_per_step * args.steps),
            "clocks": clocks,
        }
        if world == 1 and not args.skip_secondary:
            try:
                del layers, graph
                torch.cuda.empty_cache()
                line["secondary"] = secondary_metrics(device, peak, args)
            except Exception as e:  # never lose the headline line to a secondary measurement
                line["secondary"] = {"error": f"{type(e).__name__}: {e}"}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if same_n1 is not None:
            line["same_workload_single_gpu"] = same_n1
            if "value" in same_n1:
                line["same_workload_scaling_efficiency"] = value / (world * same_n1["value"])
        if parity is not None:
            line["sharded_parity"] = parity
        if pairing is not None:
            line["tp_pairing_variant"] = pairing
        if compute_only is not None:
            line["compute_vs_exchange"] = compute_only
        print(json.dumps(line), flush=True)
    if world > 1:
        # Clean teardown: drop the CUDA graphs (they may hold captured NCCL kernels), sync, then destroy the process group.
        # A watchdog leaves through os._exit if the destroy does not return (seen in round 1 with graphs that captured
        # NCCL all-reduces still alive); everything has been printed and synchronised by then.
        try:
            if graph is not None:
                graph.reset()
        except Exception:
            pass
        graph = None
        layers = None
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()

        def _bail():
            print("[bench] destroy_process_group did not return within 20 s; leaving through os._exit", file=sys.stderr, flush=True)
            os._exit(0)

        teardown_timer = threading.Timer(20.0, _bail)
        teardown_timer.daemon = True
        teardown_timer.start()
        dist.destroy_process_group()
        teardown_timer.cancel()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=[None, *MODELS])
    ap.add_argument("--scheme", default="1x16")
    ap.add_argument("--layers", type=int, default=0, help="override the layer count (debug only; invalidates the number)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-group", action="store_true", help="one launch per linear instead of grouped q/k/v and gate/up")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-n1", action="store_true")
    ap.add_argument("--skip-secondary", action="store_true")
    ap.add_argument("--skip-pairing", action="store_true", help="N>1: skip the out/in-features pairing variant")
    ap.add_argument("--skip-parity", action="store_true", help="N>1: skip the sharded-vs-unsharded correctness pass")
    ap.add_argument("--skip-reference-gpu", action="store_true", help="skip the reference CUDA kernels / generate legs")
    ap.add_argument("--watchdog-seconds", type=float, default=420.0,
                    help="N>1: leave with an error line if one phase (parity, build, timing, ...) takes longer than this (0: off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write every linear's output of the last timed step as DIR/<linear>.npy (float32, seeded inputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
