"""GEMM experiment probe: for each (shape, batch) and each environment setting, check the fused dequant + tcgen05 GEMM
against the C oracle (row sample) and time it (CUDA-graph replay over rotating weight copies, CUDA events).
    python tools/probe_gemm.py [--shapes 4096x14336,4096x4096] [--batches 256] [--settings "A=1,B=2;A=0"] [--scheme 1x16]
                               [--in-group 16]
Each setting is a ';'-separated list of comma-separated ENV=VALUE pairs (AQLM_B200_ prefix added); the settings of one
(shape, batch) run back to back, so e.g. --settings "DISABLE_TCGEN05=1;" alternates the GEMV passes and the tensor-core
path.  The first line records the device (name, power limit, SM clocks) the numbers were taken on."""
import argparse
import json
import os
import subprocess
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))
from aqlm_b200 import _cabi  # noqa: E402
from aqlm_b200.inference_kernels import cuda_kernel  # noqa: E402

KEYS = ["DISABLE_TCGEN05", "PDL", "GEMM_A_STAGES", "GEMM_GROUPS", "GEMM_ATMEM", "GEMM_TILE_M", "GEMM_KSPLIT", "GEMM_STAGES", "GEMM_V2", "GEMM_GATHER_MODE", "GEMM_DEBUG", "GEMM_CLUSTER"]


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
    return a.elapsed_time(b) * 1e3 / iters / len(fns)


def main():
    from helpers import c_oracle_check, gpu_case

    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="4096x14336,4096x4096,14336x4096")
    ap.add_argument("--batches", default="256")
    ap.add_argument("--scheme", default="1x16")
    ap.add_argument("--in-group", type=int, default=8, choices=[8, 16])
    ap.add_argument("--dtype", default="f16")
    ap.add_argument("--op", default="matmat_dequant", choices=["matmat_dequant", "matmat_dequant_transposed"])
    ap.add_argument("--settings", default="")
    ap.add_argument("--no-check", action="store_true")
    args = ap.parse_args()
    K, nbits = (int(v) for v in args.scheme.split("x"))
    dt = torch.float16 if args.dtype == "f16" else torch.bfloat16
    settings = [dict(kv.split("=") for kv in st.split(",") if kv) for st in args.settings.split(";")] if args.settings else [{}]
    op = getattr(cuda_kernel, args.op)
    g = args.in_group
    dev = dict(device=torch.cuda.get_device_name(0))
    try:
        dev["nvidia_smi"] = subprocess.run(
            ["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        dev["nvidia_smi"] = f"unavailable: {e}"
    print(json.dumps(dev), flush=True)
    for shape in args.shapes.split(","):
        fin, fout = (int(v) for v in shape.split("x"))
        for bs in (int(b) for b in args.batches.split(",")):
            t = gpu_case(fin, fout, K, nbits, bs, dtype=dt, seed=fin + fout + bs, g=g)
            cbytes = fout * (fin // g) * K * (2 if nbits > 8 else 1)
            copies = max(2, min(24, 300 * 2**20 // cbytes))
            lo, hi = (-128, 128) if nbits <= 8 else (-32768, 32768)
            ws = [(t["codes"], t["codebooks"], t["scales"])] + [
                (torch.randint(lo, hi, t["codes"].shape, dtype=t["codes"].dtype, device="cuda:0"), t["codebooks"], t["scales"])
                for _ in range(copies - 1)]
            transposed = args.op.endswith("transposed")
            x = torch.randn((bs, fout), dtype=dt, device="cuda:0") if transposed else t["x"]
            for st in settings:
                for k in KEYS:
                    os.environ.pop("AQLM_B200_" + k, None)
                for k, v in st.items():
                    os.environ["AQLM_B200_" + k] = v
                _cabi.reload_tunables()
                row = dict(op=args.op, scheme=args.scheme, in_group=g, dtype=args.dtype, shape=shape, batch=bs, setting=st)
                try:
                    c0 = _cabi.launch_count()
                    y = op(x, t["codes"], t["codebooks"], t["scales"], None)
                    torch.cuda.synchronize()
                    row["launches"] = _cabi.launch_count() - c0
                    if not args.no_check:
                        if transposed:
                            W = cuda_kernel.dequant(t["codes"], t["codebooks"], t["scales"]).float()
                            ref = x.float() @ W
                            row["rel_err"] = float(((y.float() - ref).abs().mean() / ref.abs().mean()).item())
                        else:
                            row["rel_err"] = c_oracle_check(t, y)
                    us = timed([(lambda w=w: op(x, w[0], w[1], w[2], None)) for w in ws])
                    row["us"] = round(us, 2)
                    row["tflops"] = round(2.0 * bs * fin * fout / us / 1e6, 1)
                except Exception as e:
                    row["error"] = f"{type(e).__name__}: {str(e)[:200]}"
                    torch.cuda.synchronize()
                print(json.dumps(row), flush=True)
            del ws, t
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
