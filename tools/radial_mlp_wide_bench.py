"""Cost of wide radial MLPs: the lmax-2 model (bench.HP) with invariant_neurons 32 / 64 / 128 on 512 synthetic
crystals (matten_b200.data.synthetic.synthetic_batch(512)), fp32, eval mode, random weights.  Appends one JSON line
with, per width:
  fwd_ms            forward under no_grad
  fwd_param_bwd_ms  forward + backward to every parameter
  fwd_geom_bwd_ms   forward + backward to pos and cell with frozen parameters
and, for every width that takes the per-edge-weight path (last hidden size > 64), per conv layer the kernel times of
radial_mlp_kernel and of the contraction reading w (conv_fwd_kernel<float, 0>) from torch.profiler in a separate run,
the MLP's FLOPs (2 E sum(fan_in fan_out)) and its share of the FP32 FMA peak measured in profiles/r2_microbench.jsonl
(66.8 TFLOP/s).  The GPU's name, power limit and max SM clock are read in the same run.

    python tools/radial_mlp_wide_bench.py [--out profiles/radial_mlp_wide_b200.jsonl]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from matten_b200 import ops  # noqa: E402
from matten_b200.data.synthetic import synthetic_batch  # noqa: E402
from matten_b200.model_factory import ScalarTensorModel  # noqa: E402
from tools.geometry_grad_bench import KEYS, gpu_info, timed  # noqa: E402

DEV = torch.device("cuda:0")
FMA_PEAK_TFLOPS = 66.8  # profiles/r2_microbench.jsonl, FP32 FFMA2 on one B200


def _layer_kernels(model, data):
    """[(mlp_sizes, E, radial_mlp_ms, contraction_ms)] of one forward, by torch.profiler over 5 forwards."""
    from torch.profiler import ProfilerActivity, profile

    calls = []
    real = ops.conv_fwd

    def spy(handle, x, sh, emb, ws, *a, **k):
        calls.append((list(handle.mlp_sizes), int(sh.shape[0])))
        return real(handle, x, sh, emb, ws, *a, **k)

    ops.conv_fwd = spy
    try:
        with torch.no_grad():
            model(dict(data), check=False)
    finally:
        ops.conv_fwd = real
    reps = 5
    with torch.no_grad():
        model(dict(data), check=False)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                model(dict(data), check=False)
            torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    mlp = [e.device_time / 1e3 for e in ev if "radial_mlp_kernel" in e.name]
    con = [e.device_time / 1e3 for e in ev if "conv_fwd_kernel<float, 0>" in e.name]
    n = len(calls)
    out = []
    for i, (sizes, E) in enumerate(calls):
        if len(mlp) != reps * n or len(con) != reps * n:
            break
        t_mlp = sum(mlp[r * n + i] for r in range(reps)) / reps
        t_con = sum(con[r * n + i] for r in range(reps)) / reps
        flops = 2.0 * E * sum(a * b for a, b in zip(sizes, sizes[1:]))
        out.append({"mlp_sizes": sizes, "edges": E, "radial_mlp_ms": round(t_mlp, 4),
                    "contraction_ms": round(t_con, 4), "mlp_gflop": round(flops / 1e9, 2),
                    "mlp_tflops": round(flops / (t_mlp * 1e-3) / 1e12, 2),
                    "mlp_share_of_fma_peak": round(flops / (t_mlp * 1e-3) / 1e12 / FMA_PEAK_TFLOPS, 3)})
    return out


def run(neurons, host, reps):
    torch.manual_seed(0)
    hp = dict(bench.HP, invariant_neurons=neurons)
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
    if neurons > 64:
        res["layers"] = _layer_kernels(model, data)
    res["atoms"], res["edges"] = int(data["pos"].shape[0]), int(data["edge_index"].shape[1])
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--crystals", type=int, default=512)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    host = synthetic_batch(a.crystals)
    line = {"workload": f"synthetic_batch({a.crystals}), lmax 2, fp32, eval mode, random weights", "gpu": gpu_info()}
    for n in (32, 64, 128):
        line[f"neurons{n}"] = run(n, host, a.reps)
    s = json.dumps(line)
    print(s, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "a") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
