"""First derivatives of model outputs with respect to the geometry on the GPU: the convolution's gradients to its edge
inputs (mt_conv_bwd_full), the backward kernels of the spherical harmonics, the radial bases and the edge vectors, and
whole-model gradients with respect to positions and cells, each against autograd through the CPU oracle.

Tolerances follow tests/test_gpu_backward.py (normwise relative, max|a-b| / max|b|): per op 2e-5 in fp32 and 1e-10 in
fp64, whole model 5e-4 in fp32 and 1e-9 in fp64."""
import pytest
import torch

from tests.helpers import HP_LMAX2, HP_LMAX4, SPECIES8, build_pair, rel_err, to_oracle_batch
from tests.test_gpu_backward import _conv_pair, gtol, mtol

pytestmark = pytest.mark.gpu
DTYPES = [torch.float32, torch.float64]
DEV = torch.device("cuda:0")


def _dev_batch(batch, dtype):
    return {k: (v.to(DEV).to(dtype) if isinstance(v, torch.Tensor) and v.is_floating_point()
                else (v.to(DEV) if isinstance(v, torch.Tensor) else v)) for k, v in batch.items()}


def _out(o, key):
    return o[key] if isinstance(o, dict) else o


# ----------------------------------------------------------------------------------------------- per op: conv
def _conv_edge_grad_case(dtype, *args):
    conv, ref, data, sp = _conv_pair(DEV, dtype, *args)
    N = data["node_features"].shape[0]
    sho = data["edge_attrs"].clone().requires_grad_(True)
    embo = data["edge_embedding"].clone().requires_grad_(True)
    out_o = ref(dict(data, edge_attrs=sho, edge_embedding=embo))["node_features"]
    R = torch.randn(out_o.shape, dtype=dtype, generator=torch.Generator().manual_seed(99))
    (out_o * R).sum().backward()
    # CUDA path with frozen parameters and node features: the conv records for its edge inputs alone
    conv = conv.to(DEV)
    for p in conv.parameters():
        p.requires_grad_(False)
    d = {k: v.to(DEV) for k, v in data.items()}
    d["species_index"] = sp.to(DEV)
    d["pos"] = torch.zeros(N, 3, dtype=dtype, device=DEV)
    shg = d["edge_attrs"].clone().requires_grad_(True)
    embg = d["edge_embedding"].clone().requires_grad_(True)
    out_g = conv(dict(d, edge_attrs=shg, edge_embedding=embg))["node_features"]
    gsh, gemb = torch.autograd.grad((out_g * R.to(DEV)).sum(), (shg, embg))
    assert rel_err(gsh, sho.grad) < gtol(dtype), "grad sh"
    assert rel_err(gemb, embo.grad) < gtol(dtype), "grad emb"
    out2 = conv(dict(d, edge_attrs=shg, edge_embedding=embg))["node_features"]
    gsh2, gemb2 = torch.autograd.grad((out2 * R.to(DEV)).sum(), (shg, embg))
    assert torch.equal(gsh, gsh2) and torch.equal(gemb, gemb2)


@pytest.mark.parametrize("dtype", DTYPES)
def test_conv_edge_gradients_lmax2_and_lmax4(dtype):
    _conv_edge_grad_case(dtype, "32x0e+16x1o+4x2e", 2, "72x0e+16x1o+16x1e+4x2o+4x2e", 8, 8, 32, 2, 28.0, 100,
                         lambda n: 28, 1)
    ir4 = "32x0o+32x0e+16x1o+16x1e+4x2o+4x2e+2x3o+2x3e+2x4e"
    deg = lambda n: [0, 1, 3, 200, 28, 0, 64, 65][n % 8]  # noqa: E731
    _conv_edge_grad_case(dtype, ir4, 4, ir4, 5, 8, 32, 2, 30.4, 32, deg, 3)
    irt = "32x0o+32x0e+16x1o+16x1e+8x2o+8x2e+4x3o+4x3e+4x4o+4x4e"
    _conv_edge_grad_case(dtype, irt, 4, irt, 2, 10, 32, 2, None, 24, lambda n: 5 + (n % 7), 4)


@pytest.mark.parametrize("dtype", DTYPES)
def test_conv_edge_gradients_mlp_variants(dtype):
    ir = "8x0e+8x1o+4x2e"
    _conv_edge_grad_case(dtype, ir, 2, ir, 3, 8, 64, 2, 10.0, 64, lambda n: 12, 6)     # 64 hidden units
    _conv_edge_grad_case(dtype, ir, 2, ir, 1, 10, 8, 0, 10.0, 64, lambda n: 12, 7)     # no hidden layer
    _conv_edge_grad_case(dtype, ir, 1, ir, 3, 8, 16, 3, 10.0, 64, lambda n: 12, 8)     # three hidden layers


# ----------------------------------------------------------------------------------------------- per op: geometry
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("lmax", [2, 4])
def test_edge_sh_backward(dtype, lmax):
    from matten_b200 import functional as F
    from oracle import e3nn_restated as E

    g = torch.Generator().manual_seed(lmax)
    vec = torch.randn(3000, 3, generator=g, dtype=dtype) * 2
    vec[:4] = torch.tensor([[0.0, 1.0, 0.0], [0.0, -2.0, 0.0], [1e-7, 3.0, 0.0], [0.0, 0.0, 1e-3]], dtype=dtype)
    R = torch.randn(3000, (lmax + 1) ** 2, generator=g, dtype=dtype)
    vo = vec.clone().requires_grad_(True)
    (E.spherical_harmonics(lmax, vo, True, "component") * R).sum().backward()
    vg = vec.to(DEV).requires_grad_(True)
    (F.edge_sh(vg, lmax, True) * R.to(DEV)).sum().backward()
    assert rel_err(vg.grad, vo.grad) < gtol(dtype)


@pytest.mark.parametrize("dtype", DTYPES)
def test_edge_radial_backward(dtype):
    from matten_b200 import functional as F
    from oracle import e3nn_restated as E
    from oracle import matten_restated as M

    g = torch.Generator().manual_seed(0)
    r = torch.rand(4000, generator=g, dtype=dtype) * 5.8 + 0.2  # some beyond the 5.0 cutoff
    R = torch.randn(4000, 8, generator=g, dtype=dtype)
    # mode 0: soft_one_hot_linspace(bessel) * sqrt(n)
    ro = r.clone().requires_grad_(True)
    (E.soft_one_hot_linspace_bessel(ro, 0.0, 5.0, 8, True) * 8 ** 0.5 * R).sum().backward()
    rg = r.to(DEV).requires_grad_(True)
    (F.edge_radial(rg, 0, 8, 0.0, 5.0, True) * R.to(DEV)).sum().backward()
    assert rel_err(rg.grad, ro.grad) < gtol(dtype), "mode 0"
    # mode 1 with trainable frequencies: both gradients
    basis, cut = M.BesselBasis(5.0, 8, trainable=True).to(dtype), M.PolynomialCutoff(5.0, 6).to(dtype)
    with torch.no_grad():
        basis.bessel_weights.mul_(1 + 0.1 * torch.rand(8, generator=g, dtype=dtype))
    ro = r.clone().requires_grad_(True)
    (basis(ro) * cut(ro).unsqueeze(-1) * R).sum().backward()
    rg = r.to(DEV).requires_grad_(True)
    wg = basis.bessel_weights.detach().to(DEV).requires_grad_(True)
    (F.edge_radial(rg, 1, 8, 0.0, 5.0, True, 6.0, wg) * R.to(DEV)).sum().backward()
    assert rel_err(rg.grad, ro.grad) < gtol(dtype), "mode 1 length"
    assert rel_err(wg.grad, basis.bessel_weights.grad) < gtol(dtype), "mode 1 frequencies"


def _edge_vectors_case(dtype, B, cell_shape, with_batch=True):
    from matten_b200 import functional as F
    from oracle import matten_restated as M

    g = torch.Generator().manual_seed(B)
    n_per = 7
    N = B * n_per
    pos = torch.randn(N, 3, generator=g, dtype=dtype) * 3
    cell = (torch.eye(3, dtype=dtype) * 4 + torch.randn(B, 3, 3, generator=g, dtype=dtype) * 0.3)
    batch = torch.arange(B).repeat_interleave(n_per)
    E_ = 400
    src = torch.randint(0, N, (E_,), generator=g)
    dst = (src // n_per) * n_per + torch.randint(0, n_per, (E_,), generator=g)  # edges stay inside a crystal
    ei = torch.stack([src, dst])
    shift = torch.randint(-1, 2, (E_, 3), generator=g).to(dtype)
    shift[:5] = 0
    ei[1, :5] = ei[0, :5]  # zero vectors: the length term contributes 0 there, as torch's norm backward
    Rv = torch.randn(E_, 3, generator=g, dtype=dtype)
    Rl = torch.randn(E_, generator=g, dtype=dtype)

    def oracle_grads():
        po = pos.clone().requires_grad_(True)
        co = cell.reshape(cell_shape).clone().requires_grad_(True)
        d = {"pos": po, "edge_index": ei, "cell": co, "edge_cell_shift": shift, "batch": batch}
        d = M.with_edge_vectors(d)
        ((d["edge_vectors"] * Rv).sum() + (d["edge_lengths"] * Rl).sum()).backward()
        return po.grad, co.grad

    gpo, gco = oracle_grads()
    pg = pos.to(DEV).requires_grad_(True)
    cg = cell.reshape(cell_shape).to(DEV).requires_grad_(True)
    vec, ln = F.edge_vectors(pg, ei.to(DEV), shift.to(DEV), cg, batch.to(DEV) if with_batch else None, None)
    ((vec * Rv.to(DEV)).sum() + (ln * Rl.to(DEV)).sum()).backward()
    assert rel_err(pg.grad, gpo) < gtol(dtype), "pos"
    assert cg.grad.shape == cg.shape
    assert rel_err(cg.grad, gco) < gtol(dtype), "cell"


@pytest.mark.parametrize("dtype", DTYPES)
def test_edge_vectors_backward(dtype):
    _edge_vectors_case(dtype, 3, (3, 3, 3))
    _edge_vectors_case(dtype, 3, (9, 3))
    _edge_vectors_case(dtype, 1, (1, 3, 3), with_batch=False)
    _edge_vectors_case(dtype, 1, (3, 3), with_batch=False)


# ----------------------------------------------------------------------------------------------- whole model
def _geometry_grads(model, batch, key, R, create_graph=False):
    pos = batch["pos"].clone().requires_grad_(True)
    cell = batch["cell"].clone().requires_grad_(True)
    out = _out(model(dict(batch, pos=pos, cell=cell)), key)
    gp, gc = torch.autograd.grad((out * R.to(out.device)).sum(), (pos, cell), create_graph=create_graph)
    return gp, gc


def _model_case(hp, dtype, train, seed, ncrystals=3):
    from matten_b200.data.synthetic import synthetic_batch

    orac, prod = build_pair(hp, SPECIES8, dtype, DEV, seed=seed)
    if train:
        orac.train()
        prod.train()
    batch = synthetic_batch(ncrystals, dtype=dtype)
    key = "elastic_tensor_full"
    ob, db = to_oracle_batch(batch, dtype), _dev_batch(batch, dtype)
    with torch.no_grad():
        shape = _out(orac(dict(ob)), key).shape
    R = torch.randn(shape, generator=torch.Generator().manual_seed(seed), dtype=dtype)
    for p in list(orac.parameters()) + list(prod.parameters()):
        p.requires_grad_(False)  # frozen parameters: the position / cell gradient alone
    gpo, gco = _geometry_grads(orac, ob, key, R)
    gpg, gcg = _geometry_grads(prod, db, key, R)
    assert rel_err(gpg, gpo) < mtol(dtype), "pos"
    assert rel_err(gcg, gco) < mtol(dtype), "cell"
    return prod, db, key, R, gpg


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("train", [False, True])
def test_model_position_and_cell_gradients_lmax2(dtype, train):
    _model_case(HP_LMAX2, dtype, train, seed=1)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("train", [False, True])
def test_model_position_and_cell_gradients_lmax4(dtype, train):
    _model_case(HP_LMAX4, dtype, train, seed=2)


def test_atomic_model_jacobian_of_one_atom():
    """Sensitivity of one atom's NMR-type tensor to every position: the Jacobian, one component at a time."""
    from matten_b200.data.synthetic import synthetic_batch

    dtype = torch.float64
    hp = dict(HP_LMAX2, output_format="cartesian")
    orac, prod = build_pair(hp, [8, 14], dtype, DEV, seed=2, atomic=True)
    batch = synthetic_batch(2, species=[8, 14], dtype=dtype)
    ob, db = to_oracle_batch(batch, dtype), _dev_batch(batch, dtype)
    po = ob["pos"].clone().requires_grad_(True)
    pg = db["pos"].clone().requires_grad_(True)
    out_o = _out(orac(dict(ob, pos=po)), "nmr_tensor")
    out_g = _out(prod(dict(db, pos=pg)), "nmr_tensor")
    assert rel_err(out_g, out_o) < 1e-10
    atom = 5
    for i in range(3):
        for j in range(3):
            (jo,) = torch.autograd.grad(out_o[atom, i, j], po, retain_graph=True)
            (jg,) = torch.autograd.grad(out_g[atom, i, j], pg, retain_graph=True)
            assert rel_err(jg, jo) < mtol(dtype), (i, j)


@pytest.mark.parametrize("dtype", DTYPES)
def test_precomputed_edge_vectors_require_grad(dtype):
    from matten_b200.data.synthetic import synthetic_batch
    from oracle import matten_restated as M

    orac, prod = build_pair(HP_LMAX2, SPECIES8, dtype, DEV, seed=4)
    batch = synthetic_batch(2, dtype=dtype)
    ob, db = to_oracle_batch(batch, dtype), _dev_batch(batch, dtype)
    vec = M.with_edge_vectors(dict(ob), with_lengths=False)["edge_vectors"].detach()
    key = "elastic_tensor_full"
    vo = vec.clone().requires_grad_(True)
    vg = vec.to(DEV).requires_grad_(True)
    out_o = _out(orac(dict(ob, edge_vectors=vo)), key)
    out_g = _out(prod(dict(db, edge_vectors=vg)), key)
    R = torch.randn(out_o.shape, generator=torch.Generator().manual_seed(0), dtype=dtype)
    (go,) = torch.autograd.grad((out_o * R).sum(), vo)
    (gg,) = torch.autograd.grad((out_g * R.to(DEV)).sum(), vg)
    assert rel_err(gg, go) < mtol(dtype)


# ----------------------------------------------------------------------------------------------- properties
def test_translation_invariance_and_finite_differences_fp64():
    """Per crystal, sum over its atoms of grad_pos = 0 (to 1e-10 of max|grad_pos|); and central differences
    (h = 1e-5) on the CUDA model itself agree with its gradient to 1e-6 of max|gradient| (the O(h^2) truncation)."""
    dtype = torch.float64
    prod, db, key, R, gp = _model_case(HP_LMAX2, dtype, False, seed=5)
    scale = float(gp.abs().max())
    for b in range(int(db["num_graphs"])):
        s = gp[db["batch"] == b].sum(0)
        assert float(s.abs().max()) <= 1e-10 * scale, (b, s)
    _, gc = _geometry_grads(prod, db, key, R)
    Rd = R.to(DEV)

    def f(pos, cell):
        with torch.no_grad():
            return float((_out(prod(dict(db, pos=pos, cell=cell)), key) * Rd).sum())

    h = 1e-5
    g = torch.Generator().manual_seed(0)
    for idx in torch.randint(0, db["pos"].numel(), (6,), generator=g).tolist():
        pp, pm = db["pos"].clone(), db["pos"].clone()
        pp.view(-1)[idx] += h
        pm.view(-1)[idx] -= h
        fd = (f(pp, db["cell"]) - f(pm, db["cell"])) / (2 * h)
        assert abs(fd - float(gp.view(-1)[idx])) <= 1e-6 * scale, (idx, fd, float(gp.view(-1)[idx]))
    cscale = float(gc.abs().max())
    for idx in (0, 4, 8, 10):
        cp, cm = db["cell"].clone(), db["cell"].clone()
        cp.view(-1)[idx] += h
        cm.view(-1)[idx] -= h
        fd = (f(db["pos"], cp) - f(db["pos"], cm)) / (2 * h)
        assert abs(fd - float(gc.view(-1)[idx])) <= 1e-6 * cscale, (idx, fd, float(gc.view(-1)[idx]))


def test_geometry_gradients_are_deterministic_and_perturb_nothing_else():
    """Two backward passes give bitwise equal position / cell gradients, and the parameter gradients are bitwise the
    same whether or not the positions require grad."""
    from matten_b200.data.synthetic import synthetic_batch

    dtype = torch.float32
    _, prod = build_pair(HP_LMAX2, SPECIES8, dtype, DEV, seed=6)
    db = _dev_batch(synthetic_batch(4, dtype=dtype), dtype)
    key = "elastic_tensor_full"
    R = torch.randn(4, 6, generator=torch.Generator().manual_seed(0), dtype=dtype).to(DEV)

    def run(pos_grad):
        prod.zero_grad(set_to_none=True)
        pos = db["pos"].clone().requires_grad_(pos_grad)
        cell = db["cell"].clone().requires_grad_(pos_grad)
        (_out(prod(dict(db, pos=pos, cell=cell)), key) * R).sum().backward()
        return {k: p.grad.clone() for k, p in prod.named_parameters()}, pos.grad, cell.grad

    w1, p1, c1 = run(True)
    w2, p2, c2 = run(True)
    w0, p0, c0 = run(False)
    assert p0 is None and c0 is None
    assert torch.equal(p1, p2) and torch.equal(c1, c2)
    for k in w1:
        assert torch.equal(w1[k], w2[k]), k
        assert torch.equal(w1[k], w0[k]), k


def test_node_feature_gradients_unchanged_by_edge_gradients():
    """A conv's node-feature and weight gradients are bitwise the same whether or not sh / emb also want one."""
    conv, _, data, sp = _conv_pair(DEV, torch.float32, "32x0e+16x1o+4x2e", 2, "72x0e+16x1o+16x1e+4x2o+4x2e", 8, 8, 32, 2,
                                   28.0, 100, lambda n: 28, 1)
    conv = conv.to(DEV)
    d = {k: v.to(DEV) for k, v in data.items()}
    d["species_index"] = sp.to(DEV)
    d["pos"] = torch.zeros(d["node_features"].shape[0], 3, device=DEV)

    def run(edge):
        conv.zero_grad(set_to_none=True)
        x = d["node_features"].clone().requires_grad_(True)
        sh = d["edge_attrs"].clone().requires_grad_(edge)
        emb = d["edge_embedding"].clone().requires_grad_(edge)
        out = conv(dict(d, node_features=x, edge_attrs=sh, edge_embedding=emb))["node_features"]
        R = torch.randn(out.shape, generator=torch.Generator().manual_seed(0)).to(DEV)
        (out * R).sum().backward()
        return x.grad, {k: p.grad.clone() for k, p in conv.named_parameters()}

    x1, w1 = run(True)
    x0, w0 = run(False)
    assert torch.equal(x1, x0)
    for k in w1:
        assert torch.equal(w1[k], w0[k]), k


def test_second_derivative_through_the_geometry_raises():
    from matten_b200.data.synthetic import synthetic_batch

    dtype = torch.float64
    _, prod = build_pair(HP_LMAX2, SPECIES8, dtype, DEV, seed=7)
    db = _dev_batch(synthetic_batch(2, dtype=dtype), dtype)
    pos = db["pos"].clone().requires_grad_(True)
    out = _out(prod(dict(db, pos=pos)), "elastic_tensor_full")
    with pytest.raises(RuntimeError, match="second derivatives"):
        torch.autograd.grad(out.sum(), pos, create_graph=True)


def test_graph_without_edges_gives_zero_gradients():
    from matten_b200 import functional as F

    pos = torch.randn(5, 3, dtype=torch.float64, device=DEV, requires_grad=True)
    cell = (torch.eye(3, dtype=torch.float64, device=DEV) * 5).requires_grad_(True)
    ei = torch.zeros(2, 0, dtype=torch.int64, device=DEV)
    shift = torch.zeros(0, 3, dtype=torch.float64, device=DEV)
    vec, ln = F.edge_vectors(pos, ei, shift, cell, None, None)
    sh = F.edge_sh(vec, 2, True)
    emb = F.edge_radial(ln, 0, 8, 0.0, 5.0, True)
    gp, gc = torch.autograd.grad(sh.sum() + emb.sum() + vec.sum() + ln.sum() + 0 * pos.sum() + 0 * cell.sum(),
                                 (pos, cell))
    assert torch.equal(gp, torch.zeros_like(gp)) and torch.equal(gc, torch.zeros_like(gc))
    assert gc.shape == cell.shape
