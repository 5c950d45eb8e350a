"""The gaussian, cosine, smooth_finite and fourier edge-length bases on the GPU (radial modes 3-6 of mt_edge_radial /
mt_edge_radial_bwd), op by op and in whole models, against the e3nn reference of tests/test_radial_basis_host.py.

Tolerances (normwise relative, max|a-b| / max|b|, plus the element-wise metric for the forward) are those of the
Bessel basis: forward 1e-5 / 1e-10 (fp32 / fp64) against the fp64 reference on the lengths the kernel saw; length
gradient gtol, whole models mtol of tests/test_gpu_backward.py."""
import itertools
import json
import math
import os

import numpy as np
import pytest
import torch

from tests.helpers import (GOLDEN, HP_LMAX2, HP_LMAX4, SPECIES8, build_pair, elem_err, rel_err, to_oracle_batch,
                           tol)
from tests.test_gpu_backward import gtol, mtol
from tests.test_radial_basis_host import MODES, EdgeLengthEmbedding, lengths, soft_one_hot_linspace

pytestmark = pytest.mark.gpu
DTYPES = [torch.float32, torch.float64]
DEV = torch.device("cuda:0")
CASES = [(0.0, 5.0, 8), (0.5, 4.0, 2), (-1.0, 6.0, 10)]  # (start, end, n): start != 0 and n in {2, 8, 10}
BASIS_CUTOFF = list(itertools.product(list(MODES), [True, False]))


def _ref(r, start, end, n, basis, cutoff):
    return soft_one_hot_linspace(r, start, end, n, basis, cutoff) * math.sqrt(n)


# ----------------------------------------------------------------------------------------------- per op
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("basis,cutoff", BASIS_CUTOFF)
def test_forward_matches_reference(basis, cutoff, dtype):
    """Lengths below `start`, between the centres, beyond `end`, and exactly on the centres and boundaries.
    Element-wise (floor 1e-3 of the largest value): fp32 rounding of the argument (eps * n pi for fourier) is up to
    2e-3 of that floor, as for the Bessel basis in test_gpu_ops.py."""
    from matten_b200 import ops

    for start, end, n in CASES:
        r = lengths(start, end, n, cutoff, dtype).to(DEV)
        got = ops.edge_radial(r, MODES[basis], n, start, end, cutoff)
        want = _ref(r.cpu().double(), start, end, n, basis, cutoff)
        assert got.shape == (r.numel(), n) and got.dtype == dtype
        assert rel_err(got, want) < tol(dtype), (start, end, n, rel_err(got, want))
        assert elem_err(got, want) < (2e-3 if dtype == torch.float32 else 1e-9), (start, end, n, elem_err(got, want))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("basis,cutoff", BASIS_CUTOFF)
def test_length_gradient_matches_reference_autograd(basis, cutoff, dtype):
    """d (R . emb) / d r through F.edge_radial (EdgeRadialFn -> mt_edge_radial_bwd) against autograd through the fp64
    reference at the same lengths (random ones: a mask that switches has no derivative), where that is finite."""
    from matten_b200 import functional as F

    for start, end, n in CASES:
        r = lengths(start, end, n, cutoff, dtype, boundaries=False, count=4000, seed=n)
        R = torch.randn(r.numel(), n, generator=torch.Generator().manual_seed(1), dtype=dtype)
        ro = r.double().requires_grad_(True)
        (want,) = torch.autograd.grad((_ref(ro, start, end, n, basis, cutoff) * R.double()).sum(), ro)
        rg = r.to(DEV).requires_grad_(True)
        (got,) = torch.autograd.grad((F.edge_radial(rg, MODES[basis], n, start, end, cutoff) * R.to(DEV)).sum(), rg)
        ok = torch.isfinite(want)
        assert ok.sum() > 0.99 * ok.numel()
        assert torch.isfinite(got).all()
        assert rel_err(got.cpu()[ok], want[ok]) < gtol(dtype), (start, end, n, rel_err(got.cpu()[ok], want[ok]))


@pytest.mark.parametrize("dtype", DTYPES)
def test_forward_and_backward_are_bitwise_deterministic(dtype):
    from matten_b200 import ops

    r = lengths(-1.0, 6.0, 10, True, dtype, count=100_000).to(DEV)
    g = torch.randn(r.numel(), 10, generator=torch.Generator().manual_seed(0), dtype=dtype).to(DEV)
    for basis, cutoff in BASIS_CUTOFF:
        m = MODES[basis]
        assert torch.equal(ops.edge_radial(r, m, 10, -1.0, 6.0, cutoff), ops.edge_radial(r, m, 10, -1.0, 6.0, cutoff))
        a = ops.edge_radial_bwd(r, g, m, 10, -1.0, 6.0, cutoff)
        assert torch.equal(a, ops.edge_radial_bwd(r, g, m, 10, -1.0, 6.0, cutoff)), basis


def test_invalid_arguments_raise_before_any_launch():
    from matten_b200 import ops
    from matten_b200.nn.embedding import EdgeLengthEmbedding as ProductEmbedding

    r = torch.rand(64, device=DEV) * 5
    g = torch.randn(64, 8, device=DEV)
    before = ops.launch_count()
    for mode in (-1, 7):
        with pytest.raises(RuntimeError, match=f"radial mode {mode}"):
            ops.edge_radial(r, mode, 8, 0.0, 5.0, True)
    for mode in (-1, 2, 7):  # the frequency derivative (mode 2) has no length gradient
        with pytest.raises(RuntimeError, match=f"radial backward mode {mode}"):
            ops.edge_radial_bwd(r, g, mode, 8, 0.0, 5.0, True)
    for mode in (3, 4, 5):
        with pytest.raises(RuntimeError, match="needs num_basis >= 2"):
            ops.edge_radial(r, mode, 1, 0.0, 5.0, False)
        with pytest.raises(RuntimeError, match="needs num_basis >= 2"):
            ops.edge_radial_bwd(r, g[:, :1].contiguous(), mode, 1, 0.0, 5.0, False)
    with pytest.raises(RuntimeError, match="bad radial basis parameters"):
        ops.edge_radial(r, 3, 8, 5.0, 5.0, True)
    with pytest.raises(ValueError, match='basis="hat" is not a valid entry'):
        ProductEmbedding(basis="hat")
    assert ops.launch_count() == before
    # with cutoff a single function is fine (the centres are the inner point of linspace(start, end, 3))
    got = ops.edge_radial(r, 3, 1, 0.0, 5.0, True)
    assert rel_err(got, _ref(r.cpu().double(), 0.0, 5.0, 1, "gaussian", True)) < tol(torch.float32)


def test_custom_op_matches_the_functional_layer():
    from matten_b200 import ops, torch_ops  # noqa: F401  (registers the ops)

    for dtype in DTYPES:
        r = lengths(-1.0, 6.0, 10, True, dtype).to(DEV)
        for basis, cutoff in BASIS_CUTOFF:
            got = torch.ops.matten_b200.edge_radial(r, MODES[basis], 10, -1.0, 6.0, cutoff, 6.0)
            assert torch.equal(got, ops.edge_radial(r, MODES[basis], 10, -1.0, 6.0, cutoff)), (basis, cutoff)


# ----------------------------------------------------------------------------------------------- whole models
def _pair(monkeypatch, hp, basis, dtype, seed, species=SPECIES8):
    """build_pair with `radial_basis_type = basis`: the oracle's radial layer is the reference for every basis."""
    from oracle import matten_restated as M

    monkeypatch.setattr(M, "EdgeLengthEmbedding", EdgeLengthEmbedding)
    orac, prod = build_pair(dict(hp, radial_basis_type=basis), species, dtype, DEV, seed=seed)
    assert orac.backbone.radial_basis.basis == prod.backbone.radial_basis.basis == basis
    return orac, prod


def _dev_batch(batch, dtype):
    return {k: (v.to(DEV).to(dtype) if isinstance(v, torch.Tensor) and v.is_floating_point()
                else (v.to(DEV) if isinstance(v, torch.Tensor) else v)) for k, v in batch.items()}


def _out(o, key="elastic_tensor_full"):
    return o[key] if isinstance(o, dict) else o


def _model_case(monkeypatch, hp, basis, dtype, train, seed):
    """Forward output, every parameter gradient, then the position and cell gradients with frozen parameters."""
    from matten_b200 import autograd as A
    from matten_b200.data.synthetic import synthetic_batch

    orac, prod = _pair(monkeypatch, hp, basis, dtype, seed)
    if train:
        orac.train()
        prod.train()
    batch = synthetic_batch(3, dtype=dtype)
    ob, db = to_oracle_batch(batch, dtype), _dev_batch(batch, dtype)
    out_o = _out(orac(dict(ob)))
    out_g = _out(prod(dict(db)))
    assert rel_err(out_g, out_o) < (1e-5 if dtype == torch.float32 else 1e-10), "forward"
    target = torch.randn(out_o.shape, dtype=dtype, generator=torch.Generator().manual_seed(seed))
    torch.nn.functional.mse_loss(out_o, target).backward()
    A.mse_loss(out_g, target.to(DEV)).backward()
    og = dict(orac.named_parameters())
    n = 0
    for k, p in prod.named_parameters():
        assert p.grad is not None, k
        assert rel_err(p.grad, og[k].grad.reshape(p.grad.shape)) < mtol(dtype), k
        n += 1
    assert n == len(og)

    for p in list(orac.parameters()) + list(prod.parameters()):
        p.requires_grad_(False)
    R = torch.randn(out_o.shape, generator=torch.Generator().manual_seed(seed + 1), dtype=dtype)
    grads = []
    for model, b in ((orac, ob), (prod, db)):
        pos = b["pos"].clone().requires_grad_(True)
        cell = b["cell"].clone().requires_grad_(True)
        out = _out(model(dict(b, pos=pos, cell=cell)))
        grads.append(torch.autograd.grad((out * R.to(out.device)).sum(), (pos, cell)))
    (gpo, gco), (gpg, gcg) = grads
    assert float(gpo.abs().max()) > 0
    assert rel_err(gpg, gpo) < mtol(dtype), "pos"
    assert rel_err(gcg, gco) < mtol(dtype), "cell"


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("basis", list(MODES))
def test_model_lmax2(monkeypatch, basis, train, dtype):
    _model_case(monkeypatch, HP_LMAX2, basis, dtype, train, seed=11)


def test_model_lmax4_gaussian(monkeypatch):
    _model_case(monkeypatch, HP_LMAX4, "gaussian", torch.float32, False, seed=12)


def test_save_pretrained_predict_round_trip_gaussian(tmp_path):
    """A gaussian-basis checkpoint written by save_pretrained and served by predict gives what the model in memory
    computes on the same crystals."""
    from matten_b200.data.neighbors import collate, make_graph
    from matten_b200.model_factory import ScalarTensorModel
    from matten_b200.nn.readout import CartesianTensorWrapper
    from matten_b200.predict import predict, save_pretrained

    with open(os.path.join(GOLDEN, "n100_structures.json")) as f:
        structs = json.load(f)["structures"][:6]
    species = sorted({z for s in structs for z in s["atomic_numbers"]})
    torch.manual_seed(13)
    model = ScalarTensorModel(dict(HP_LMAX4, radial_basis_type="gaussian"), {"allowed_species": species})
    model = model.to(DEV).eval()
    save_pretrained(model, tmp_path / "m", r_cut=5.0, tensor_target_name="elastic_tensor_full")
    inputs = [{"lattice": s["lattice"], "atomic_numbers": s["atomic_numbers"], "cart_coords": s["cart_coords"]}
              for s in structs]
    got = np.stack([np.asarray(p) for p in predict(inputs, model_identifier=str(tmp_path / "m"), batch_size=len(inputs),
                                                   device=DEV)])
    graphs = [make_graph(np.array(s["cart_coords"]), np.array(s["lattice"]), s["atomic_numbers"], 5.0, torch.float32)
              for s in structs]
    with torch.no_grad():
        out = model(_dev_batch(collate(graphs), torch.float32))["elastic_tensor_full"]
        want = CartesianTensorWrapper("ijkl=jikl=klij").to_cartesian(out).cpu().numpy()
    assert got.shape == want.shape == (6, 3, 3, 3, 3)
    assert np.allclose(got, want, rtol=0, atol=1e-6 * float(np.abs(want).max()))
