"""Cost of the edge-length bases: every radial mode of mt_edge_radial (0 soft-one-hot Bessel, 1 Bessel x polynomial
cutoff, 2 its frequency derivative, 3 gaussian, 4 cosine, 5 smooth_finite, 6 fourier) and of mt_edge_radial_bwd
(all but mode 2), on the edge lengths of synthetic_batch(512) (917 504 edges, the lmax-2 benchmark workload) with
8 basis functions, fp32 and fp64, each timed by CUDA events over repeated calls; and the lmax-2 model (bench.HP) with
the bessel and with the gaussian basis: forward under no_grad, and forward + position / cell backward with frozen
parameters, the two bases alternated.  Prints one JSON line with the GPU's name and power limit read in the same run.

    python tools/radial_basis_bench.py [--out profiles/radial_basis_b200.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from matten_b200 import ops  # noqa: E402
from matten_b200.data.synthetic import synthetic_batch  # noqa: E402
from matten_b200.model_factory import ScalarTensorModel  # noqa: E402

DEV = torch.device("cuda:0")
KEYS = ["pos", "edge_index", "edge_cell_shift", "cell", "batch", "atomic_numbers", "num_neigh"]
MODE_NAMES = {0: "bessel", 1: "bessel_poly_cutoff", 2: "bessel_freq_derivative", 3: "gaussian", 4: "cosine",
              5: "smooth_finite", 6: "fourier"}


def timed(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(reps):
        fn()
    ev1.record()
    torch.cuda.synchronize()
    return round(ev0.elapsed_time(ev1) / reps, 4)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unavailable"


def kernels(ln32, reps):
    res = {}
    for dtype in (torch.float32, torch.float64):
        ln = ln32.to(dtype)
        g = torch.randn(ln.shape[0], 8, device=DEV, dtype=dtype)
        per = {}
        for mode, name in MODE_NAMES.items():
            t = {"fwd_ms": timed(lambda: ops.edge_radial(ln, mode, 8, 0.0, 5.0, True), reps)}
            if mode != 2:
                t["bwd_ms"] = timed(lambda: ops.edge_radial_bwd(ln, g, mode, 8, 0.0, 5.0, True), reps)
            per[f"{mode}_{name}"] = t
        res[str(dtype).replace("torch.", "")] = per
    return res


def models(host, reps, rounds):
    data = {k: host[k].to(DEV) for k in KEYS}
    data["num_graphs"] = host["num_graphs"]
    key = "elastic_tensor_full"
    built = {}
    for basis in ("bessel", "gaussian"):
        torch.manual_seed(0)
        m = ScalarTensorModel(dict(bench.HP, radial_basis_type=basis), {"allowed_species": bench.SPECIES})
        m = m.to(DEV).eval()
        for p in m.parameters():
            p.requires_grad_(False)
        built[basis] = m
    res = {b: {"fwd_ms": [], "fwd_geom_bwd_ms": []} for b in built}
    for _ in range(rounds):
        for basis, model in built.items():
            def fwd():
                with torch.no_grad():
                    model(dict(data), check=False)

            def fwd_geom_bwd():
                pos = data["pos"].clone().requires_grad_(True)
                cell = data["cell"].clone().requires_grad_(True)
                out = model(dict(data, pos=pos, cell=cell), check=False)[key]
                torch.autograd.grad(out.sum(), (pos, cell))

            res[basis]["fwd_ms"].append(timed(fwd, reps))
            res[basis]["fwd_geom_bwd_ms"].append(timed(fwd_geom_bwd, reps))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--crystals", type=int, default=512)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--model-reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    host = synthetic_batch(a.crystals)
    d = {k: host[k].to(DEV) for k in KEYS}
    _, ln = ops.edge_vectors(d["pos"], d["edge_index"], d["edge_cell_shift"], d["cell"], d["batch"])
    line = {"workload": f"synthetic_batch({a.crystals}): {ln.shape[0]} edge lengths x 8 basis functions, "
                        "start 0, end 5, cutoff; lmax-2 model (bench.HP) in fp32, eval mode, random weights",
            "gpu": gpu_info(),
            "kernels_ms": kernels(ln, a.reps),
            "model_lmax2_ms": models(host, a.model_reps, a.rounds)}
    s = json.dumps(line)
    print(s, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "a") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
