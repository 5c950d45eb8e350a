"""Radial MLPs wider than 64 (up to 128 input / hidden units): the convolution's per-edge-weight path
(radial_mlp_kernel + the contractions that read w from memory) against the CPU oracle, forward, backward (x, MLP
weights, sh, embedding), determinism, whole models with invariant_neurons 96 / 128, and checks that the shapes of
today's kernels do not touch the new path."""
import numpy as np
import pytest
import torch

from tests.helpers import HP_LMAX2, HP_LMAX4, SPECIES8, build_pair, elem_err, rel_err, to_oracle_batch, tol

pytestmark = pytest.mark.gpu
DTYPES = [torch.float32, torch.float64]
DEV = torch.device("cuda:0")
IR2 = "32x0o+32x0e+16x1o+16x1e+4x2o+4x2e"
IR4 = "32x0o+32x0e+16x1o+16x1e+4x2o+4x2e+2x3o+2x3e+2x4e"
RAGGED = lambda n: [0, 1, 65, 500, 28, 0, 3, 64][n % 8]  # noqa: E731
NEW_KERNELS = ("radial_mlp_kernel", "conv_bwd_wide_kernel", "mlp_bwd_last_wide_kernel", "mlp_bwd_hidden_wide_kernel")


def gtol(dtype):
    return 2e-5 if dtype == torch.float32 else 1e-10


def mtol(dtype):
    return 5e-4 if dtype == torch.float32 else 1e-9


def _dev_batch(batch, dtype):
    return {k: (v.to(DEV).to(dtype) if isinstance(v, torch.Tensor) and v.is_floating_point()
                else (v.to(DEV) if isinstance(v, torch.Tensor) else v)) for k, v in batch.items()}


def _conv_pair(dtype, sizes, x_ir, sh_lmax, N, deg_fn, seed, S=4, avg=28.0):
    """PointConv (product, oracle) whose radial MLP has the layer sizes `sizes` (input ... last hidden)."""
    from matten_b200 import o3
    from matten_b200.nn.conv import PointConv
    from matten_b200.nn.utils import RadialMLP
    from oracle import e3nn_restated as E
    from oracle import matten_restated as M

    torch.manual_seed(seed)
    g = torch.Generator().manual_seed(seed)
    n_rad = sizes[0]
    irreps_in = {"node_features": o3.Irreps(x_ir), "node_attrs": o3.Irreps(f"{S}x0e"),
                 "edge_attrs": o3.Irreps.spherical_harmonics(sh_lmax), "edge_embedding": o3.Irreps(f"{n_rad}x0e")}
    old = torch.get_default_dtype()
    torch.set_default_dtype(dtype)
    try:
        conv = PointConv(irreps_in, x_ir, 1, 8, avg)
        oin = {k: o3.parse_irreps_list(v) for k, v in irreps_in.items()}
        ref = M.PointConv(oin, x_ir, 1, 8, avg)
        hs = list(sizes) + [conv.tp.plan.weight_numel]
        conv.tp.weight_nn = RadialMLP(hs, conv.tp.weight_nn.act_name)
        conv.tp._handles = {}
        ref.tp.weight_nn = E.FullyConnectedNet(hs, act=M.ACTIVATION["e"]["silu"])
    finally:
        torch.set_default_dtype(old)
    _, unexpected = ref.load_state_dict(conv.state_dict(), strict=False)
    assert not unexpected
    dst = torch.cat([torch.full((deg_fn(n),), n, dtype=torch.int64) for n in range(N)])
    E_ = len(dst)
    src = torch.randint(0, N, (E_,), generator=g)
    ei = torch.stack([src, dst])[:, torch.randperm(E_, generator=g)]
    sp = torch.randint(0, S, (N,), generator=g)
    data = {"node_features": torch.randn(N, conv.tp.plan.x_dim, dtype=dtype),
            "node_attrs": torch.nn.functional.one_hot(sp, S).to(dtype),
            "edge_attrs": E.spherical_harmonics(sh_lmax, torch.randn(E_, 3, dtype=dtype), True, "component"),
            "edge_embedding": torch.randn(E_, n_rad, dtype=dtype), "edge_index": ei,
            "num_neigh": torch.bincount(ei[0], minlength=N).to(dtype).clamp(min=1)}
    return conv.to(DEV), ref, data, sp


def _run_dev(conv, data, sp, grads):
    d = {k: v.to(DEV) for k, v in data.items()}
    d["species_index"] = sp.to(DEV)
    d["pos"] = torch.zeros(data["node_features"].shape[0], 3, dtype=data["node_features"].dtype, device=DEV)
    leaves = {}
    if grads:
        for k in ("node_features", "edge_attrs", "edge_embedding"):
            leaves[k] = d[k] = d[k].clone().requires_grad_(True)
    return conv(d)["node_features"], leaves


def _wide_case(dtype, sizes, x_ir=IR2, sh_lmax=2, N=24, deg_fn=RAGGED, seed=0):
    conv, ref, data, sp = _conv_pair(dtype, sizes, x_ir, sh_lmax, N, deg_fn, seed)
    # forward
    with torch.no_grad():
        want = ref(dict(data))["node_features"]
        got, _ = _run_dev(conv, data, sp, False)
        got2, _ = _run_dev(conv, data, sp, False)
    assert rel_err(got, want) < tol(dtype)
    assert elem_err(got, want) < (2e-3 if dtype == torch.float32 else 1e-9)
    assert torch.equal(got, got2), "forward must be bitwise repeatable"
    # backward: x, MLP weights, sh and the embedding, against oracle autograd
    o_leaves = {k: data[k].clone().requires_grad_(True) for k in ("node_features", "edge_attrs", "edge_embedding")}
    out_o = ref(dict(data, **o_leaves))["node_features"]
    R = torch.randn(out_o.shape, dtype=dtype, generator=torch.Generator().manual_seed(99))
    (out_o * R).sum().backward()
    ref_w = {k: p.grad for k, p in ref.tp.weight_nn.named_parameters()}
    runs = []
    for _ in range(2):
        for p in conv.parameters():
            p.grad = None
        out_g, leaves = _run_dev(conv, data, sp, True)
        (out_g * R.to(DEV)).sum().backward()
        runs.append(({k: v.grad.clone() for k, v in leaves.items()},
                     {k: p.grad.clone() for k, p in conv.tp.weight_nn.named_parameters()}))
    (gl, gw), (gl2, gw2) = runs
    for k, v in o_leaves.items():
        assert rel_err(gl[k], v.grad) < gtol(dtype), k
        assert torch.equal(gl[k], gl2[k]), k
    for k, v in ref_w.items():
        assert rel_err(gw[k], v.reshape(gw[k].shape)) < gtol(dtype), k
        assert torch.equal(gw[k], gw2[k]), k
    return conv


MLP_SHAPES = [(8, 128, 128), (8, 96), (10, 65, 128, 128), (100,), (8, 128, 32), (8, 32, 128)]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("sizes", MLP_SHAPES, ids=lambda s: "-".join(map(str, s)))
def test_wide_conv_lmax2(dtype, sizes):
    _wide_case(dtype, sizes, seed=len(sizes))


@pytest.mark.parametrize("dtype", DTYPES)
def test_wide_conv_lmax4(dtype):
    _wide_case(dtype, (8, 128, 128), x_ir=IR4, sh_lmax=4, N=16, seed=7)


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def test_limits_raise_without_launching():
    """A last hidden size of 129 fails the forward, any input / hidden size of 129 the backward, before any launch."""
    from matten_b200 import ops

    for sizes in [(8, 129), (129, 32), (8, 129, 32)]:
        conv, _, data, _ = _conv_pair(torch.float32, sizes, "8x0e+8x1o", 1, 6, lambda n: 3, 0)
        h = conv.tp.handle(DEV)
        src, dst = data["edge_index"]
        perm = torch.argsort(dst, stable=True)
        rowptr = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(torch.bincount(dst, minlength=6), 0)])
        g = [t.to(torch.int32).to(DEV) for t in (rowptr, perm, src[perm])]
        x = torch.randn(6, h.plan.x_dim, device=DEV)
        sh, emb = data["edge_attrs"].float().to(DEV), data["edge_embedding"].float().to(DEV)
        ws = [w.detach() for w in conv.tp.weight_nn.weights()]
        n0 = ops.launch_count()
        if sizes[-1] > 128:
            with pytest.raises(RuntimeError, match="> 128"):
                ops.conv_fwd(h, x, sh, emb, ws, *g, 28.0)
        else:  # inner layers up to 256 still run forward (today's kernels)
            out = ops.conv_fwd(h, x, sh, emb, ws, *g, 28.0)
            n0 = ops.launch_count()
            with pytest.raises(RuntimeError, match="<= 128"):
                ops.conv_bwd_full(h, x, sh, emb, ws, *g, None, None, 28.0, None, torch.ones_like(out), need_x=False)
        torch.cuda.synchronize()
        assert ops.launch_count() == n0, sizes


@pytest.mark.parametrize("neurons", [32, 64])
def test_existing_widths_never_take_the_new_path(neurons):
    from matten_b200.data.synthetic import synthetic_batch

    _, prod = build_pair(dict(HP_LMAX2, invariant_neurons=neurons), SPECIES8, torch.float32, DEV, seed=1)
    db = _dev_batch(synthetic_batch(2), torch.float32)
    names = _kernel_names(lambda: prod(dict(db)))
    pos = db["pos"].clone().requires_grad_(True)
    names += _kernel_names(lambda: prod(dict(db, pos=pos))["elastic_tensor_full"].sum().backward())
    prod.train()
    names += _kernel_names(lambda: prod(dict(db))["elastic_tensor_full"].sum().backward())
    assert names and not [n for n in names if any(k in n for k in NEW_KERNELS)]


def test_wide_model_uses_the_new_path():
    from matten_b200.data.synthetic import synthetic_batch

    _, prod = build_pair(dict(HP_LMAX2, invariant_neurons=128), SPECIES8, torch.float32, DEV, seed=1)
    db = _dev_batch(synthetic_batch(2), torch.float32)
    names = _kernel_names(lambda: prod(dict(db)))
    assert any("radial_mlp_kernel" in n for n in names)
    assert any("conv_fwd_kernel<float, 0>" in n or "conv_fwd_kernelIfLi0E" in n for n in names), set(names)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("neurons", [96, 128])
def test_wide_model_parity_and_gradients(dtype, neurons):
    from matten_b200.data.synthetic import synthetic_batch

    hp = dict(HP_LMAX2, invariant_neurons=neurons)
    orac, prod = build_pair(hp, SPECIES8, dtype, DEV, seed=3)
    batch = synthetic_batch(3, dtype=dtype)
    ob, db = to_oracle_batch(batch, dtype), _dev_batch(batch, dtype)
    key = "elastic_tensor_full"
    with torch.no_grad():
        want = orac(dict(ob))
        got = prod(dict(db))[key]
    assert rel_err(got, want) < tol(dtype)
    R = torch.randn(want.shape, dtype=dtype, generator=torch.Generator().manual_seed(4))
    orac.train()
    prod.train()
    # train-mode forward, parameter gradients
    out_o = orac(dict(ob))
    (out_o * R).sum().backward()
    out_g = prod(dict(db))[key]
    assert rel_err(out_g, out_o) < mtol(dtype)
    (out_g * R.to(DEV)).sum().backward()
    ref_g = {k: p.grad for k, p in orac.named_parameters()}
    for k, p in prod.named_parameters():
        if k in ref_g and ref_g[k] is not None:
            assert rel_err(p.grad, ref_g[k].reshape(p.grad.shape)) < mtol(dtype), k
    # position and cell gradients with frozen parameters
    for p in list(orac.parameters()) + list(prod.parameters()):
        p.requires_grad_(False)
    grads = []
    for m, b in ((orac, ob), (prod, db)):
        pos = b["pos"].clone().requires_grad_(True)
        cell = b["cell"].clone().requires_grad_(True)
        out = m(dict(b, pos=pos, cell=cell))
        out = out[key] if isinstance(out, dict) else out
        grads.append(torch.autograd.grad((out * R.to(out.device)).sum(), (pos, cell)))
    assert rel_err(grads[1][0], grads[0][0]) < mtol(dtype), "pos"
    assert rel_err(grads[1][1], grads[0][1]) < mtol(dtype), "cell"


def test_wide_lmax4_model_forward():
    from matten_b200.data.synthetic import synthetic_batch

    dtype = torch.float32
    orac, prod = build_pair(dict(HP_LMAX4, invariant_neurons=128), SPECIES8, dtype, DEV, seed=2)
    batch = synthetic_batch(2, dtype=dtype)
    with torch.no_grad():
        want = orac(to_oracle_batch(batch, dtype))
        got = prod(_dev_batch(batch, dtype))["elastic_tensor_full"]
    assert rel_err(got, want) < tol(dtype)


def test_wide_trainer_steps_follow_the_oracle():
    """Three Trainer steps of a 128-wide model against the oracle trained with the same loss and Adam settings."""
    from matten_b200.data.synthetic import synthetic_batch
    from matten_b200.train import Trainer

    dtype = torch.float64
    orac, prod = build_pair(dict(HP_LMAX2, invariant_neurons=128), SPECIES8, dtype, DEV, seed=6)
    orac.train()
    prod.train()
    batch = synthetic_batch(3, dtype=dtype)
    ob, db = to_oracle_batch(batch, dtype), _dev_batch(batch, dtype)
    with torch.no_grad():
        shape = orac(dict(ob)).shape
    target = torch.randn(shape, dtype=dtype, generator=torch.Generator().manual_seed(1))
    tr = Trainer(prod, lr=1e-3, weight_decay=0.0)
    opt = torch.optim.Adam([p for p in orac.parameters() if p.requires_grad], lr=1e-3)
    losses = []
    for _ in range(3):
        opt.zero_grad()
        lo = torch.nn.functional.mse_loss(orac(dict(ob)), target)
        lo.backward()
        opt.step()
        lg = float(tr.step(dict(db), target.to(DEV)))
        losses.append(lg)
        assert abs(lg - float(lo)) <= 1e-8 * abs(float(lo)), (lg, float(lo))
    assert losses[-1] < losses[0]


def test_wide_predict_round_trip_and_captured_graph(tmp_path):
    from matten_b200.data.synthetic import synthetic_batch
    from matten_b200.graphs import CapturedForward
    from matten_b200.predict import predict, save_pretrained

    hp = dict(HP_LMAX2, invariant_neurons=128)
    _, prod = build_pair(hp, SPECIES8, torch.float32, DEV, seed=5)
    b1 = _dev_batch(synthetic_batch(4, seed=0), torch.float32)
    with torch.no_grad():
        want = prod(dict(b1))["elastic_tensor_full"].clone()
        got = CapturedForward(prod)(b1)["elastic_tensor_full"].clone()
    assert torch.equal(got, want)
    save_pretrained(prod, tmp_path, 5.0)
    s = {"lattice": (np.eye(3) * 3.6).tolist(), "atomic_numbers": [6, 14], "cart_coords": [[0, 0, 0], [0.9, 0.9, 0.9]]}
    p1 = np.asarray(predict(s, model_identifier=str(tmp_path), device=DEV))
    p2 = np.asarray(predict([s, s], model_identifier=str(tmp_path), batch_size=2, device=DEV))
    assert p1.shape == (3, 3) and np.isfinite(p1).all()
    assert np.array_equal(p2[0], p1) and np.array_equal(p2[1], p1)
