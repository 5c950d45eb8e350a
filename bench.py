#!/usr/bin/env python
"""
bench.py -- headline benchmark of the matten_b200 hot path (BASELINE.json metric:
crystals/sec, inference forward, at N B200s, next to the CPU reference path).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1], SURVEY.md section 8d "config 2"): 512 synthetic crystals per
GPU, 64-atom diamond-cubic supercells, r_cut 5 A (N = 32 768 atoms, E = 917 504 edges), lmax-2
backbone of scripts/configs/atomic_tensor.yaml with the pooled rank-2 head; random weights,
fp32.  A "step" is one forward of the whole batch.  Under torchrun (N > 1) every rank runs its own
batch (weak scaling, no data-path collective: crystals are independent graphs).

Prints ONE JSON line (see README / DESIGN.md for the keys).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HP = {
    "species_embedding_dim": 16, "irreps_edge_sh": "0e + 1o + 2e", "num_radial_basis": 8,
    "radial_basis_start": 0.0, "radial_basis_end": 5.0, "radial_basis_type": "bessel", "num_layers": 3,
    "invariant_layers": 2, "invariant_neurons": 32, "average_num_neighbors": 28.0,
    "conv_layer_irreps": "32x0o+32x0e + 16x1o+16x1e + 4x2o+4x2e", "nonlinearity_type": "gate",
    "normalization": "batch", "resnet": True, "conv_to_output_hidden_irreps_out": "16x0e + 2x2e",
    "output_format": "irreps", "output_formula": "ij=ji", "reduce": "mean",
}
# pretrained/20230627/config_final.yaml:24-42 of the reference (BASELINE config 1 and 3)
HP_LMAX4 = dict(HP, irreps_edge_sh="0e + 1o + 2e + 3o + 4e",
                conv_layer_irreps="32x0o+32x0e + 16x1o+16x1e + 4x2o+4x2e + 2x3o+2x3e + 2x4e",
                conv_to_output_hidden_irreps_out="16x0e + 2x2e + 4e", output_formula="ijkl=jikl=klij")
SPECIES = [1, 6, 7, 8, 14, 22, 26, 29]
CRYSTALS_PER_GPU = 512
CPU_SAMPLE = 64  # crystals per CPU step: the unique part of the batch (about 1.5 s per step on 16 cores)
WORKLOAD = "synthetic 512 crystals x 64-atom diamond supercells, r_cut 5 A, lmax=2 inference (fwd)"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def fma_peak():
    """fp32 FMA peak in TFLOP/s measured on this pool's B200 by tools/microbench.cu (FFMA2, all 148 SMs)."""
    p = os.path.join(ROOT, "profiles", "r2_microbench.jsonl")
    best = None
    if os.path.exists(p):
        for line in open(p):
            try:
                d = json.loads(line)
            except ValueError:
                continue
            if d.get("test") == "fma_peak":
                best = max(best or 0.0, float(d["tflops"]))
    if best:
        return best, "measured (profiles/r2_microbench.jsonl, tools/microbench.cu fma_peak)"
    return 2 * 148 * 128 * 1.965e-3, "nominal (148 SMs x 128 lanes x 2 flop x 1.965 GHz)"


def make_batch(num_crystals: int, seed: int):
    """512 crystals: 64 unique jittered crystals from the exact neighbour search, tiled 8x with fresh
    jitter of 0.01 A on the copies (the topology is unchanged: shells at 4.50 / 5.43 A vs r_cut 5)."""
    from matten_b200.data.synthetic import synthetic_batch, tile_batch

    unique = min(64, num_crystals)
    small = synthetic_batch(unique, seed=seed)
    if num_crystals == unique:
        return small
    assert num_crystals % unique == 0
    return tile_batch(small, num_crystals // unique, jitter=0.01, seed=seed + 1)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons, mx = [], set(), None
        try:
            for line in open(self.path):
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 8:
                    continue
                try:
                    sm.append(float(parts[1]))
                    mx = float(parts[2])
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                   parts[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))
        return out


def conv_algorithmic_bytes(key, n_rad: int, mlp_numel: int, s: int = 4) -> int:
    """SURVEY.md section 8(d): bytes = E*(8 + s*(D_sh + D_rad + D_in)) + N*s*D_mid + s*numel(W_mlp)."""
    x_dim, y_dim, out_dim, wn, N, E = key
    return E * (8 + s * (y_dim + n_rad + x_dim)) + N * s * out_dim + s * mlp_numel


def reference_importable():
    """The unmodified reference (baseline/_ref) needs e3nn, torch_scatter, torch_geometric, pymatgen and
    pytorch_lightning, none of which is in this image or its wheelhouse (DESIGN.md section 2)."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(ref):
        return False, "baseline/_ref absent: pip install of /root/reference cannot resolve e3nn / torch_scatter offline"
    sys.path.insert(0, ref)
    try:
        import e3nn  # noqa: F401
        import matten.model_factory.tfn_scalar_tensor  # noqa: F401
        return True, "baseline/_ref"
    except Exception as exc:  # noqa: BLE001
        sys.path.remove(ref)
        return False, f"baseline/_ref present but not importable: {type(exc).__name__}: {exc}"


def cpu_baseline(num_crystals: int, steps: int, warmup: int, seed: int = 0):
    """The reference CPU path on all host cores, on a bounded sample of the same workload: the unmodified reference
    from baseline/_ref when it imports, else the restated oracle (oracle/matten_restated.py: e3nn-style
    materialising einsums + one-hot FCTPs + scatter)."""
    ok, why = reference_importable()
    if ok:
        # the reference's backbone (an nn.Sequential over the graph dict, src/matten/model_factory/
        # tfn_scalar_tensor.py:103-241); untested here: it has never been importable in this image
        from matten.model_factory.tfn_scalar_tensor import create_model as ref_create_model  # type: ignore

        kind = "reference"
        build = lambda: ref_create_model(HP, {"allowed_species": SPECIES})  # noqa: E731
    else:
        from oracle import matten_restated as M

        kind = "port"
        build = lambda: M.ScalarTensorModel(HP, {"allowed_species": SPECIES})  # noqa: E731

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    model = build().eval()
    batch = make_batch(num_crystals, seed)
    b = {k: v for k, v in batch.items() if isinstance(v, torch.Tensor)}
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            out = model(b)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    times.sort()
    med = times[len(times) // 2]
    return {"value": num_crystals / med, "unit": "crystals/s", "cores": cores, "kind": kind,
            "outputs": {"elastic_tensor_full": out},
            "sample": f"{num_crystals} of the 512 crystals per step ({b['edge_index'].shape[1]} edges; the 512 are "
                      f"these 64 unique crystals tiled 8x with fresh jitter), median of {steps} steps after {warmup} "
                      f"warm-up, torch {torch.__version__} CPU fp32, "
                      + ("unmodified reference from baseline/_ref" if ok else f"restated oracle ({why})"),
            "same_config": num_crystals >= 64, "ms_per_step": med * 1e3}


def predict_config1(dev):
    """BASELINE config 1 (CPU-runnable in the reference): ``predict()`` on the 100 example crystals (473 atoms, 14 380
    edges, 73 elements) through the public API: structures on the host -> GPU neighbour search -> lmax-4 forward ->
    Cartesian tensors back on the host.  The pretrained checkpoint is not available offline, so a random-weight model
    of the same architecture is written with save_pretrained() and loaded through the checkpoint loader, as predict()
    does for a named model.  Wall clock (the call includes host work), best of 3 after one warm-up call; the loaded
    model is cached between calls while the checkpoint file is unchanged, its load time is reported separately."""
    import tempfile as _tf

    from matten_b200.model_factory import ScalarTensorModel
    from matten_b200.predict import get_pretrained_model, predict, save_pretrained

    path = os.path.join(ROOT, "tests", "golden", "n100_structures.json")
    if not os.path.exists(path):
        return {"unavailable": "tests/golden/n100_structures.json missing"}
    structs = json.load(open(path))["structures"]
    species = sorted({int(z) for s in structs for z in s["atomic_numbers"]})
    torch.manual_seed(0)
    model = ScalarTensorModel(HP_LMAX4, {"allowed_species": species})
    model.task_name = "elastic_tensor_full"
    with _tf.TemporaryDirectory() as d:
        save_pretrained(model, d, r_cut=5.0, tensor_target_name="elastic_tensor_full",
                        tensor_target_formula="ijkl=jikl=klij")
        t0 = time.perf_counter()
        get_pretrained_model(d, device=dev)
        torch.cuda.synchronize()
        t_load = time.perf_counter() - t0
        times = []
        for _ in range(4):
            t0 = time.perf_counter()
            out = predict(structs, model_identifier=d, is_elasticity_tensor=False, device=dev)
            times.append(time.perf_counter() - t0)
    assert len(out) == 100 and out[0].shape == (3, 3, 3, 3)
    best = min(times[1:])
    return {"workload": "predict() on the 100 example crystals (473 atoms, 14380 edges), lmax-4 architecture, "
                        "random weights, fp32, one batch", "crystals": 100,
            "seconds_per_call": round(best, 4), "first_call_seconds": round(times[0], 4),
            "model_load_seconds_first_use": round(t_load, 4),
            "value": round(100 / best, 1), "unit": "crystals/s",
            "note": "BASELINE.md config 1 (B=100, N=473, E=14380); it publishes no timing for it"}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory: str, outputs) -> None:
    """Writes each prediction of the last timed step as <directory>/<name>.npy: the inputs and weights are seeded, so
    two builds run with the same arguments can be compared output for output."""
    arrays = {name: t.detach().cpu().numpy() for name, t in outputs.items()}
    nbytes = sum(a.nbytes for a in arrays.values())
    if nbytes > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {nbytes} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = CPU_SAMPLE
    res = cpu_baseline(sample, args.steps, args.warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res["outputs"])
    line = {
        "impl": "reference", "metric": "crystals/sec (inference fwd)", "value": res["value"], "unit": "crystals/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample_crystals_per_step": sample},
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample", "same_config")},
        "e2e": {"value": res["value"], "unit": "crystals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch.distributed as dist

    from matten_b200 import ops
    from matten_b200.model_factory import ScalarTensorModel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200: the CUDA path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ.pop("NCCL_DEBUG")  # the version banner goes to stdout; rank 0 must print ONE JSON line
        dist.init_process_group("nccl", device_id=dev)

    per_gpu = CRYSTALS_PER_GPU
    if args.scaling == "strong":
        if CRYSTALS_PER_GPU % world or (CRYSTALS_PER_GPU // world) % 64:
            raise SystemExit("--scaling strong splits the 512 crystals evenly in multiples of 64: use 1, 2, 4 or 8 GPUs")
        per_gpu = CRYSTALS_PER_GPU // world
    torch.manual_seed(0)
    model = ScalarTensorModel(HP, {"allowed_species": SPECIES}).to(dev).eval()
    host = make_batch(per_gpu, seed=rank)
    B = host["num_graphs"]
    N, E = host["pos"].shape[0], host["edge_index"].shape[1]
    keys = ["pos", "edge_index", "edge_cell_shift", "cell", "batch", "atomic_numbers", "num_neigh"]
    pinned = {k: host[k].pin_memory() for k in keys}
    h2d_bytes = sum(v.numel() * v.element_size() for v in pinned.values())
    resident = {k: v.to(dev) for k, v in pinned.items()}
    resident["num_graphs"] = B

    from matten_b200.graphs import CapturedForward

    captured = None if args.no_cuda_graph else CapturedForward(model)

    def step_resident():
        if captured is not None:
            return captured(resident, check=False)
        return model(resident, check=False)

    out_host = torch.empty((B, 6), dtype=torch.float32).pin_memory()
    d2h_bytes = out_host.numel() * out_host.element_size()

    copy_stream = torch.cuda.Stream(device=dev)
    ev_copied = [torch.cuda.Event(), torch.cuda.Event()]
    ev_done = [torch.cuda.Event(), torch.cuda.Event()]
    e2e_state = {"i": 0, "primed": False}

    def _issue_copy(slot):
        """pinned host -> the input buffers of graph `slot`, on the copy stream (overlaps the previous step's kernels)"""
        static = captured.static_inputs(resident, slot)
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_done[slot])  # the step that last used these buffers has finished
            for k, v in pinned.items():
                static[k].copy_(v, non_blocking=True)
            ev_copied[slot].record(copy_stream)
        return static

    def step_e2e():
        """One end-to-end step: H2D of this step's inputs, forward, D2H of the result, device error word checked.
        Steps are double buffered: the H2D of step i+1 is issued before step i's kernels, so it overlaps them; every
        step still pays for its own copy inside the timed region."""
        if captured is not None:
            i = e2e_state["i"]
            slot = i & 1
            if not e2e_state["primed"]:
                _issue_copy(slot)
                e2e_state["primed"] = True
            _issue_copy(slot ^ 1)  # next step's inputs
            static = captured.static_inputs(resident, slot)
            torch.cuda.current_stream(dev).wait_event(ev_copied[slot])
            out = captured(static, check=False, slot=slot)["elastic_tensor_full"]
            out_host.copy_(out, non_blocking=True)
            ev_done[slot].record(torch.cuda.current_stream(dev))
            torch.cuda.current_stream(dev).synchronize()  # the result is on the host: one sync per step
            ops.raise_on_flag(captured.error_flag(resident, slot))
            e2e_state["i"] = i + 1
        else:
            d = {k: v.to(dev, non_blocking=True) for k, v in pinned.items()}
            d["num_graphs"] = B
            out = model(d, check=True)["elastic_tensor_full"]
            out_host.copy_(out, non_blocking=True)
        return out

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    with torch.no_grad():
        # ---------------- resident (inputs already in HBM) ----------------
        for _ in range(args.warmup):
            step_resident()
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(args.steps):
            preds = step_resident()
        ev1.record()
        barrier()
        ms_res = max_over_ranks(ev0.elapsed_time(ev1) / args.steps)
        assert torch.isfinite(preds["elastic_tensor_full"]).all()
        # copied now: the end-to-end steps below replay the same graph into the same output buffers
        last_preds = {k: v.cpu() for k, v in preds.items()} if args.dump_outputs else None
        # per-kernel view of the same step: a CUDA graph replay cannot carry per-kernel events and does not pass
        # through the library's launch counter, so the conv durations (CUDA events around each mt_conv_fwd on the
        # launching stream) and the launch count come from K kernel-by-kernel steps of the identical forward
        ops.CONV_EVENTS = []
        l0 = ops.launch_count()
        ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev2.record()
        for _ in range(args.steps):
            model(resident, check=False)
        ev3.record()
        barrier()
        launches = ops.launch_count() - l0
        ms_eager = max_over_ranks(ev2.elapsed_time(ev3) / args.steps)
        conv_events = ops.CONV_EVENTS
        ops.CONV_EVENTS = None
        # ---------------- end to end (pinned host -> device -> host) ----------------
        for _ in range(min(args.warmup, 3)):
            step_e2e()
        barrier()
        ev0.record()
        for _ in range(args.steps):
            step_e2e()
        ev1.record()
        barrier()
        ms_e2e = max_over_ranks(ev0.elapsed_time(ev1) / args.steps)
        clocks = sampler.stop() if rank == 0 else None

    # ---------------- training step: fwd + bwd + (all-reduce) + Adam ----------------
    # BASELINE config 3: the lmax-4 architecture of the pretrained model, [B, 21] irreps targets, batch 32 (the
    # published batch size) and 512 crystals per GPU; the lmax-2 model of the inference line rides along.
    train = None
    if not args.no_train:
        from matten_b200.train import Trainer

        def train_point(hp, label, ncry, width, state=None):
            tmodel = ScalarTensorModel(hp, {"allowed_species": SPECIES}).to(dev)
            if state is not None:
                tmodel.load_state_dict(state)
            if ncry == B:
                res_t, edges = resident, E
            else:
                hb = make_batch(ncry, seed=100 + rank)
                res_t = {k: hb[k].to(dev) for k in keys}
                res_t["num_graphs"] = hb["num_graphs"]
                edges = hb["edge_index"].shape[1]
            trainer = Trainer(tmodel, lr=0.01, weight_decay=1e-5)
            target = torch.randn(ncry, width, generator=torch.Generator().manual_seed(1 + rank)).to(dev)
            tsteps = max(3, args.steps // 4)
            for _ in range(3):
                trainer.step(dict(res_t), target)
            barrier()
            l0 = ops.launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(tsteps):
                loss = trainer.step(dict(res_t), target)
            e1.record()
            barrier()
            ms = max_over_ranks(e0.elapsed_time(e1) / tsteps)
            assert torch.isfinite(loss).all()
            nconv = hp["num_layers"] + 1
            point = {"model": label, "crystals_per_gpu": ncry, "target": f"[B, {width}] irreps", "steps": tsteps,
                     "ms_per_step": round(ms, 4), "value": round(ncry * world / (ms * 1e-3), 1), "unit": "crystals/s",
                     "conv_edges_per_sec_fwd_bwd": round(nconv * edges * world / (ms * 1e-3), 1),
                     "gpu_launches_per_step": round((ops.launch_count() - l0) / tsteps, 1),
                     "allreduce": (f"NCCL all_reduce of the flat fp32 gradient ({trainer.opt.flat_g.numel()} floats) "
                                   f"over {world} ranks" if world > 1 else "none (1 rank)"),
                     "loss": round(float(loss), 6)}
            del trainer, tmodel
            torch.cuda.empty_cache()
            return point

        pts = [train_point(HP_LMAX4, "lmax-4 (pretrained 20230627 architecture, random weights)", 32, 21),
               train_point(HP_LMAX4, "lmax-4 (pretrained 20230627 architecture, random weights)", B, 21),
               train_point(HP, "lmax-2 (the inference line's model)", B, 6, model.state_dict())]
        train = {"metric": "crystals/sec (training step: fwd + bwd + Adam, fp32; BASELINE config 3 = lmax-4, batch 32)",
                 "value": pts[0]["value"], "unit": "crystals/s", "ms_per_step": pts[0]["ms_per_step"], "points": pts}

    # ---------------- BASELINE config 1: predict() on the 100 example crystals ----------------
    # single-GPU runs only: predict() shards over the ranks of an initialised process group, so calling it on rank 0
    # alone would leave the other ranks out of its collectives
    config1 = None
    if world == 1 and not args.no_predict:
        config1 = predict_config1(dev)

    # ---------------- roofline of the dominant kernel (fused conv) ----------------
    from matten_b200.nn.utils import UVUTensorProduct

    peak, peak_src = peaks()
    fpeak, fpeak_src = fma_peak()
    n_rad = HP["num_radial_basis"]
    macs = {}
    for m in model.modules():
        if isinstance(m, UVUTensorProduct):
            pl = m.plan
            macs[(pl.x_dim, pl.y_dim, pl.out_dim, pl.weight_numel)] = pl.cg_macs_per_edge()
    per_layer = {}
    for key, a, b in conv_events:
        per_layer.setdefault(key, []).append(a.elapsed_time(b))
    conv_ms, conv_bytes, conv_flops, layers = 0.0, 0, 0.0, []
    mlp_hidden = n_rad * 32 + 32 * 32
    for key, ts in per_layer.items():
        ms = sum(ts) / len(ts)
        nbytes = conv_algorithmic_bytes(key, n_rad, mlp_hidden + 32 * key[3])
        # fp32 FMA-pipe work per edge: the CG contraction (plan.cg_macs_per_edge: nnz(CG) + 2 l3 + 1 per channel and
        # path) and the two hidden layers of the radial MLP; the last MLP layer runs on the tensor cores
        flops = 2.0 * key[5] * (macs[key[:4]] + mlp_hidden)
        conv_ms += ms
        conv_bytes += nbytes
        conv_flops += flops
        layers.append({"x_dim": key[0], "out_dim": key[2], "weight_numel": key[3], "ms": round(ms, 4),
                       "algorithmic_MB": round(nbytes / 1e6, 2), "GBps": round(nbytes / ms / 1e6, 1),
                       "fma_TFLOPs": round(flops / ms / 1e9, 2)})
    achieved = conv_bytes / conv_ms / 1e6 if conv_ms > 0 else 0.0
    fma_tf = conv_flops / conv_ms / 1e9 if conv_ms > 0 else 0.0
    roofline = {"bound": "hbm",
                "kernel": "mt_conv_fwd = mt::tc_pad_degree/tc_pad_layout/tc_edge_hidden kernels (padded column layout + "
                          "hidden radial-MLP layers as bf16x3 planes) + mt::conv_fwd_tc_kernel<lmax> (TMA gather4 + "
                          "tcgen05 weights + CG bundles); 4 calls per step, one per PointConv layer; CUDA events "
                          "around each call on the launching stream",
                "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "traffic": None, "peak_source": peak_src,
                "fma_frac": round(fma_tf / fpeak, 4), "fma_achieved_TFLOPs": round(fma_tf, 2),
                "fma_peak_TFLOPs": round(fpeak, 2), "fma_peak_source": fpeak_src,
                "conv_ms_per_step": round(conv_ms, 4),
                "conv_share_of_step": round(conv_ms / ms_res, 3), "layers": layers}
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(prof):
        try:
            roofline["traffic"] = json.load(open(prof)).get("conv_fwd_dram_bytes_per_step")
        except Exception:
            pass

    if rank == 0:
        total_crystals = B * world
        line = {
            "metric": "crystals/sec (inference fwd)", "value": round(total_crystals / (ms_res * 1e-3), 1),
            "unit": "crystals/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_res, 4), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "crystals_per_gpu": B, "atoms_per_gpu": N, "edges_per_gpu": E,
                       "parallelism": f"{world} independent shards, no data-path collective",
                       "l2": "no flush: one step streams > 1 GB (edge arrays 92 MB + four [N, D_mid] "
                             "aggregates 436 MB + gathered rows), far above the 126 MB L2"},
            "conv_edges_per_sec": round(4 * E * world / (conv_ms * 1e-3), 1) if conv_ms > 0 else None,
            "e2e": {"value": round(total_crystals / (ms_e2e * 1e-3), 1), "unit": "crystals/s",
                    "ms_per_step": round(ms_e2e, 4), "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": d2h_bytes},
            "gpu_launches": int(launches), "launches_per_step": round(launches / args.steps, 1),
            "launch_mode": ("kernel by kernel" if captured is None else
                            "CUDA graph replay of the forward (one capture per batch shape); gpu_launches counted on "
                            "the same number of kernel-by-kernel steps"),
            "ms_per_step_kernel_by_kernel": round(ms_eager, 4),
            "roofline": roofline, "clocks": clocks, "train": train, "config1_predict": config1,
        }
        if world == 1 and not args.no_cpu_baseline:
            res = cpu_baseline(CPU_SAMPLE, 5, 2)
            line["cpu_baseline"] = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample", "same_config")}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_preds)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step measurement")
    ap.add_argument("--no-cuda-graph", action="store_true", help="launch the forward kernel by kernel from Python")
    ap.add_argument("--no-predict", action="store_true", help="skip the config-1 predict() measurement")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: 512 crystals per GPU; strong: the 512 crystals split over the GPUs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the predictions of the last one as DIR/<name>.npy "
                         "(under torchrun: rank 0's batch)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
