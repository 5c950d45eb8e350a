"""Cost of the two neighbour searches of ``ops.neighbor_list``: "pairs" (mt_neighbor_count / _fill, every atom of a
crystal against every atom and image) and "cells" (mt_neighbor_cells_*, cell list), r_cut = 5 A, fp64 positions.

Each case times whole ``ops.neighbor_list`` calls (count, the read of the edge count, fill) with CUDA events and a
synchronize, after two warm-up calls per method, the two methods alternated call by call; the median is reported.
The pair search runs only while its predicted time (last measured time x (atoms ratio)^2) stays under --pair-budget
seconds.  Cases: jittered diamond supercells of 64 to ~10^6 atoms, a sheared triclinic supercell, the same supercells
as batches of 64 crystals (for the crossover), the 100 example crystals and the 512 x 64-atom bench batch.  Then
``predict()`` on one ~10^5-atom crystal (lmax-4 architecture, random weights, fp32) with the share of its neighbour
search, and the largest kernels of the model forward on that crystal from torch.profiler (a separate run).
Writes JSON lines with the GPU's name and power limit read in the same run.

    python tools/neighbor_bench.py [--out profiles/neighbor_list_b200.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from matten_b200 import ops  # noqa: E402
from matten_b200.data.synthetic import diamond_supercell  # noqa: E402

DEV = torch.device("cuda:0")
R_CUT = 5.0
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unavailable"


def to_args(crystals):
    n = [len(p) for p, _ in crystals]
    pos = torch.as_tensor(np.concatenate([np.asarray(p, np.float64) for p, _ in crystals]))
    cell = torch.as_tensor(np.stack([np.asarray(c, np.float64) for _, c in crystals]))
    batch = torch.repeat_interleave(torch.arange(len(crystals)), torch.as_tensor(n))
    ptr = torch.as_tensor(np.concatenate([[0], np.cumsum(n)]), dtype=torch.int64)
    return (pos.to(DEV), cell.to(DEV), batch.to(DEV), ptr.to(DEV)), max(n)


def diamond(rep, seed, shear=False):
    pos, cell = diamond_supercell(rep)
    pos = pos + np.random.default_rng(seed).normal(0.0, 0.05, pos.shape)
    if shear:  # same fractional coordinates in a strongly sheared cell of the same volume
        frac = pos @ np.linalg.inv(cell)
        cell = cell @ np.array([[1.0, 0.0, 0.0], [0.9, 1.0, 0.0], [-0.8, 0.7, 1.0]])
        pos = frac @ cell
    return pos, cell


def time_call(fn):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    fn()
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1)


def measure(args, methods, reps):
    """median ms per call of each method, alternated; edges of the (last) call"""
    out, edges = {m: [] for m in methods}, None
    calls = {m: (lambda m=m: ops.neighbor_list(*args, R_CUT, method=m)) for m in methods}
    for m in methods:
        for _ in range(2):
            edges = int(calls[m]()[0].shape[1])
    for _ in range(reps):
        for m in methods:
            out[m].append(time_call(calls[m]))
    return {m: round(float(np.median(v)), 4) for m, v in out.items()}, edges


class PairBudget:
    def __init__(self, seconds):
        self.seconds, self.last = seconds, None

    def allows(self, atoms):
        if self.last is None:
            return True
        n0, ms = self.last
        return ms * (atoms / n0) ** 2 <= self.seconds * 1e3

    def record(self, atoms, ms):
        self.last = (atoms, ms)


def single_crystals(reps_list, budget, emit, gpu):
    for rep in reps_list:
        atoms = 8 * rep ** 3
        args, _ = to_args([diamond(rep, rep)])
        methods = ["cells"] + (["pairs"] if budget.allows(atoms) else [])
        reps = 10 if atoms <= 50_000 else 5
        ms, edges = measure(args, methods, reps)
        if "pairs" in ms:
            budget.record(atoms, ms["pairs"])
        emit({"case": f"diamond {rep}x{rep}x{rep} supercell, jitter 0.05 A", "crystals": 1, "atoms": atoms,
              "edges": edges, "ms": ms, "pairs_skipped": "pairs" not in ms, "gpu": gpu})
        del args
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "neighbor_list_b200.jsonl"))
    ap.add_argument("--pair-budget", type=float, default=5.0, help="seconds one pair-search call may take")
    ap.add_argument("--max-rep", type=int, default=50, help="largest supercell: 8 rep^3 atoms")
    ap.add_argument("--no-predict", action="store_true")
    a = ap.parse_args()
    gpu = gpu_info()
    lines = []

    def emit(d):
        lines.append(d)
        print(json.dumps(d), flush=True)

    # crossover: small single crystals and batches of 64 crystals of the same size
    cross = []
    for rep in (2, 3, 4, 5, 6, 7, 8):
        atoms = 8 * rep ** 3
        one, _ = to_args([diamond(rep, rep)])
        many, _ = to_args([diamond(rep, 1000 + 64 * rep + k) for k in range(64)])
        m1, e1 = measure(one, ["pairs", "cells"], 20)
        m64, e64 = measure(many, ["pairs", "cells"], 10)
        cross.append((atoms, m1, m64))
        emit({"case": f"crossover: diamond {rep}^3 supercell, one crystal and a batch of 64", "atoms": atoms,
              "edges_one": e1, "ms_one": m1, "edges_64": e64, "ms_64": m64, "gpu": gpu})
    first = next((n for n, m1, m64 in cross if m1["cells"] <= m1["pairs"] and m64["cells"] <= m64["pairs"]), None)
    emit({"case": "crossover", "rule": "smallest crystal size of the sweep above at which the cell search is at least "
          "as fast as the pair search both for one crystal and for a batch of 64", "atoms": first, "gpu": gpu})

    budget = PairBudget(a.pair_budget)
    reps = [r for r in (4, 8, 11, 16, 22, 30, 40, 50) if r <= a.max_rep]
    single_crystals(reps, budget, emit, gpu)

    args, _ = to_args([diamond(16, 7, shear=True)])
    ms, edges = measure(args, ["cells"] + (["pairs"] if budget.allows(8 * 16 ** 3) else []), 5)
    emit({"case": "sheared triclinic diamond 16^3 supercell (cell @ [[1,0,0],[0.9,1,0],[-0.8,0.7,1]])", "crystals": 1,
          "atoms": 8 * 16 ** 3, "edges": edges, "ms": ms, "gpu": gpu})

    structs = json.load(open(os.path.join(ROOT, "tests", "golden", "n100_structures.json")))["structures"]
    args, mx = to_args([(np.array(s["cart_coords"]), np.array(s["lattice"])) for s in structs])
    ms, edges = measure(args, ["pairs", "cells"], 20)
    emit({"case": "the 100 example crystals (predict_config1 batch)", "crystals": 100, "atoms": int(args[0].shape[0]),
          "max_atoms": mx, "edges": edges, "ms": ms, "auto": ops.neighbor_method(args[3], mx), "gpu": gpu})

    b = bench.make_batch(512, 0)
    n = np.bincount(b["batch"].numpy(), minlength=512)
    ptr = torch.as_tensor(np.concatenate([[0], np.cumsum(n)]), dtype=torch.int64)
    args = (b["pos"].double().to(DEV), b["cell"].reshape(-1, 3, 3).double().to(DEV), b["batch"].to(DEV), ptr.to(DEV))
    ms, edges = measure(args, ["pairs", "cells"], 20)
    emit({"case": "the 512 x 64-atom bench batch", "crystals": 512, "atoms": int(args[0].shape[0]), "edges": edges,
          "ms": ms, "auto": ops.neighbor_method(ptr, int(n.max())), "gpu": gpu})

    if not a.no_predict:
        emit(predict_large(gpu))
    with open(a.out, "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")


def predict_large(gpu, rep=24):
    """predict() on one 8 rep^3-atom crystal; its graph building and neighbour search timed on their own; the largest
    kernels of one model forward on that graph from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile

    from matten_b200.data.neighbors import batch_from_structures
    from matten_b200.model_factory import ScalarTensorModel
    from matten_b200.predict import get_pretrained_model, predict, save_pretrained

    pos, cell = diamond(rep, 11)
    z = [6, 14] * (len(pos) // 2)
    structs = [{"lattice": cell.tolist(), "atomic_numbers": z, "cart_coords": pos.tolist()}]
    arrays = [{"cart": pos, "lattice": cell, "Z": z}]
    torch.manual_seed(0)
    model = ScalarTensorModel(bench.HP_LMAX4, {"allowed_species": [6, 14]})
    model.task_name = "elastic_tensor_full"
    res = {"case": f"predict() on one diamond {rep}^3 supercell, lmax-4 architecture, random weights, fp32",
           "atoms": len(pos), "gpu": gpu}
    with tempfile.TemporaryDirectory() as d:
        save_pretrained(model, d, r_cut=R_CUT, tensor_target_name="elastic_tensor_full",
                        tensor_target_formula="ijkl=jikl=klij")
        mdl = get_pretrained_model(d, device=DEV)
        times = []
        for _ in range(4):
            t0 = time.perf_counter()
            predict(structs, model_identifier=d, is_elasticity_tensor=False, device=DEV)
            times.append(time.perf_counter() - t0)
        res["predict_ms"] = round(min(times[1:]) * 1e3, 2)
        args, mx = to_args([(pos, cell)])
        nl, edges = measure(args, ["cells"], 5)
        res["edges"] = edges
        res["neighbor_list_ms"] = nl["cells"]
        bt = []
        for _ in range(4):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            batch = batch_from_structures(arrays, R_CUT, DEV, torch.float32)
            torch.cuda.synchronize()
            bt.append(time.perf_counter() - t0)
        res["batch_from_structures_ms"] = round(min(bt[1:]) * 1e3, 2)
        res["neighbor_list_share_of_predict"] = round(nl["cells"] / res["predict_ms"], 4)
        with torch.no_grad():
            mdl(batch)
            torch.cuda.synchronize()
            fw = []
            for _ in range(3):
                fw.append(time_call(lambda: mdl(batch)))
            res["model_forward_ms"] = round(min(fw), 2)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                mdl(batch)
                torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            per[e.name] = per.get(e.name, 0.0) + e.time_range.elapsed_us() / 1e3
    top = sorted(per.items(), key=lambda kv: -kv[1])[:6]
    res["forward_top_kernels_ms"] = [[k[:120], round(v, 3)] for k, v in top]
    return res


if __name__ == "__main__":
    main()
