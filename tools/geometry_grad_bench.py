"""Cost of the position / cell gradient: the lmax-2 model (bench.HP) and the lmax-4 model (bench.HP_LMAX4) on 512
synthetic crystals (matten_b200.data.synthetic.synthetic_batch(512)), fp32, eval mode, random weights.  Prints one
JSON line with, per model:
  fwd_ms            forward under no_grad
  fwd_param_bwd_ms  forward + backward to every parameter
  fwd_geom_bwd_ms   forward + backward to pos and cell with frozen parameters
  kernels_ms        the new backward kernels alone, by CUDA events over repeated calls on the model's own tensors:
                    conv_bwd_full of every conv layer with and without the edge gradients, edge_sh_bwd,
                    edge_radial_bwd, edge_vectors_bwd
and the GPU's name and power limit, read in the same run.

    python tools/geometry_grad_bench.py [--out profiles/geometry_grad_b200.jsonl]
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
from matten_b200.graph import GraphCache  # noqa: E402
from matten_b200.model_factory import ScalarTensorModel  # noqa: E402

DEV = torch.device("cuda:0")
KEYS = ["pos", "edge_index", "edge_cell_shift", "cell", "batch", "atomic_numbers", "num_neigh"]


def timed(fn, reps):
    for _ in range(2):
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


def run(hp, host, reps):
    torch.manual_seed(0)
    model = ScalarTensorModel(hp, {"allowed_species": bench.SPECIES}).to(DEV).eval()
    data = {k: host[k].to(DEV) for k in KEYS}
    data["num_graphs"] = host["num_graphs"]
    key = "elastic_tensor_full"

    def fwd():
        with torch.no_grad():
            model(dict(data), check=False)

    def fwd_param_bwd():
        model.zero_grad(set_to_none=True)
        model(dict(data), check=False)[key].sum().backward()

    def fwd_geom_bwd():
        pos = data["pos"].clone().requires_grad_(True)
        cell = data["cell"].clone().requires_grad_(True)
        out = model(dict(data, pos=pos, cell=cell), check=False)[key]
        torch.autograd.grad(out.sum(), (pos, cell))

    res = {"fwd_ms": timed(fwd, reps), "fwd_param_bwd_ms": timed(fwd_param_bwd, reps)}
    for p in model.parameters():
        p.requires_grad_(False)
    res["fwd_geom_bwd_ms"] = timed(fwd_geom_bwd, reps)

    # the inputs of every conv layer, recorded from one forward
    calls = []
    real = ops.conv_fwd

    def spy(handle, x, sh, emb, ws, rowptr, perm, src, avg, num_neigh=None, layout=None):
        calls.append((handle, x, sh, emb, ws, avg, num_neigh))
        return real(handle, x, sh, emb, ws, rowptr, perm, src, avg, num_neigh, layout=layout)

    ops.conv_fwd = spy
    try:
        fwd()
    finally:
        ops.conv_fwd = real
    g = GraphCache(data)
    sptr, sperm = g.sender_csr()
    kern = {}
    for i, (h, x, sh, emb, ws, avg, nn_) in enumerate(calls):
        go = torch.randn(x.shape[0], h.plan.out_dim, device=DEV)
        args = (h, x, sh, emb, ws, g.rowptr, g.perm, g.src_sorted, sptr, sperm, avg, nn_, go)
        kern[f"conv{i}_bwd_x_w"] = timed(lambda: ops.conv_bwd_full(*args, True, True), reps)
        kern[f"conv{i}_bwd_x_w_sh_emb"] = timed(lambda: ops.conv_bwd_full(*args, True, True, True, True), reps)
        kern[f"conv{i}_bwd_sh_emb_only"] = timed(lambda: ops.conv_bwd_full(*args, False, False, True, True), reps)
    vec, ln = ops.edge_vectors(data["pos"], data["edge_index"], data["edge_cell_shift"], data["cell"], data["batch"])
    E = vec.shape[0]
    y_dim = calls[0][2].shape[1]
    lmax = int(round(y_dim ** 0.5)) - 1  # edge_sh holds the harmonics 0 .. lmax
    gsh = torch.randn(E, y_dim, device=DEV)
    kern["edge_sh_bwd"] = timed(lambda: ops.edge_sh_bwd(vec, gsh, lmax, True), reps)
    gemb = torch.randn(E, 8, device=DEV)
    kern["edge_radial_bwd_mode0"] = timed(lambda: ops.edge_radial_bwd(ln, gemb, 0, 8, 0.0, 5.0, True), reps)
    gptr = g.graph_ptr(data["batch"], data["num_graphs"])
    gv, gl = torch.randn_like(vec), torch.randn_like(ln)
    kern["edge_vectors_bwd"] = timed(lambda: ops.edge_vectors_bwd(vec, gv, gl, data["edge_cell_shift"], g.rowptr,
                                                                  g.perm, sptr, sperm, gptr, data["pos"].shape[0],
                                                                  data["num_graphs"]), reps)
    res["kernels_ms"] = kern
    res["atoms"], res["edges"] = int(data["pos"].shape[0]), int(E)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--crystals", type=int, default=512)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    host = synthetic_batch(a.crystals)
    line = {"workload": f"synthetic_batch({a.crystals}), fp32, eval mode, random weights", "gpu": gpu_info(),
            "lmax2": run(bench.HP, host, a.reps), "lmax4": run(bench.HP_LMAX4, host, a.reps)}
    s = json.dumps(line)
    print(s, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "a") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
