"""The e3nn edge-length bases beyond Bessel (gaussian, cosine, smooth_finite, fourier) on the CPU.

* ``soft_one_hot_linspace`` below restates e3nn 0.5.1 ``e3nn.math.soft_one_hot_linspace`` (and its ``soft_unit_step``
  with the custom backward) for every basis; ``EdgeLengthEmbedding`` is the oracle's embedding module
  (oracle.matten_restated.EdgeLengthEmbedding, reference src/matten/nn/embedding.py:158-203) built on it.  The GPU
  tests (tests/test_gpu_radial_basis.py) compare the kernels and whole models with these.  They are pinned here by
  identities of each basis, by finite differences of their autograd, and against e3nn itself where it is installed.
* The basis functions of the CUDA kernels (matten_b200/csrc/soft_one_hot.cuh) are compiled for the host with g++ and
  compared with the reference, values and derivatives, in fp64 and fp32.
* The product's ``EdgeLengthEmbedding`` and model factory accept every basis and reject what e3nn rejects.
"""
import itertools
import math
import os
import shutil
import subprocess

import pytest
import torch

from oracle import matten_restated as M

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "matten_b200", "csrc")

BASES = ["gaussian", "cosine", "smooth_finite", "fourier", "bessel"]
MODES = {"gaussian": 3, "cosine": 4, "smooth_finite": 5, "fourier": 6}


# ----------------------------------------------------------------------------------------------------------
# reference: e3nn 0.5.1 soft_one_hot_linspace
# ----------------------------------------------------------------------------------------------------------
class _SoftUnitStep(torch.autograd.Function):
    """e3nn.math.soft_unit_step: exp(-1/x) for x > 0, else 0, with e3nn's own backward."""

    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        y = torch.zeros_like(x)
        m = x > 0.0
        y[m] = (-1 / x[m]).exp()
        return y

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        dx = torch.zeros_like(x)
        m = x > 0.0
        xm = x[m]
        dx[m] = (-1 / xm).exp() / xm.pow(2)
        return dx * dy


def soft_unit_step(x):
    return _SoftUnitStep.apply(x)


def soft_one_hot_linspace(x: torch.Tensor, start: float, end: float, number: int, basis=None, cutoff=None):
    """e3nn.math.soft_one_hot_linspace: x [...] -> [..., number]."""
    if cutoff not in [True, False]:
        raise ValueError("cutoff must be specified")
    if not cutoff:
        values = torch.linspace(start, end, number, dtype=x.dtype, device=x.device)
        step = values[1] - values[0]
    else:
        values = torch.linspace(start, end, number + 2, dtype=x.dtype, device=x.device)
        step = values[1] - values[0]
        values = values[1:-1]
    diff = (x[..., None] - values) / step
    if basis == "gaussian":
        return diff.pow(2).neg().exp().div(1.12)
    if basis == "cosine":
        return torch.cos(math.pi / 2 * diff) * (diff < 1) * (-1 < diff)
    if basis == "smooth_finite":
        return 1.14136 * torch.exp(torch.tensor(2.0)) * soft_unit_step(diff + 1) * soft_unit_step(1 - diff)
    if basis == "fourier":
        x = (x[..., None] - start) / (end - start)
        if not cutoff:
            i = torch.arange(0, number, dtype=x.dtype, device=x.device)
            return torch.cos(math.pi * i * x) / math.sqrt(0.25 + number / 2)
        i = torch.arange(1, number + 1, dtype=x.dtype, device=x.device)
        return torch.sin(math.pi * i * x) / math.sqrt(0.25 + number / 2) * (0 < x) * (x < 1)
    if basis == "bessel":
        x = x[..., None] - start
        c = end - start
        bessel_roots = torch.arange(1, number + 1, dtype=x.dtype, device=x.device) * math.pi
        out = math.sqrt(2 / c) * torch.sin(bessel_roots * x / c) / x
        if not cutoff:
            return out
        return out * ((x / c) < 1) * (0 < x)
    raise ValueError(f'basis="{basis}" is not a valid entry')


class EdgeLengthEmbedding(torch.nn.Module):
    """oracle.matten_restated.EdgeLengthEmbedding for every basis (reference src/matten/nn/embedding.py:158-203)."""

    def __init__(self, irreps_in=None, num_basis=10, start=0.0, end=5.0, basis="bessel", cutoff=True):
        super().__init__()
        self.num_basis, self.start, self.end, self.basis, self.cutoff = num_basis, start, end, basis, cutoff
        self.irreps_out = dict(irreps_in or {})
        self.irreps_out[M.EDGE_EMBEDDING] = [(num_basis, 0, 1)]

    def forward(self, data):
        data = M.with_edge_vectors(data, with_lengths=True)
        emb = soft_one_hot_linspace(data[M.EDGE_LENGTH], self.start, self.end, self.num_basis, self.basis,
                                    self.cutoff)
        data[M.EDGE_EMBEDDING] = emb.mul(self.num_basis**0.5)
        return data


def centres(start, end, n, cutoff, dtype=torch.float64):
    v = torch.linspace(start, end, n + 2 if cutoff else n, dtype=dtype)
    return v[1:-1] if cutoff else v


def lengths(start, end, n, cutoff, dtype=torch.float64, boundaries=True, count=400, seed=0):
    """Random lengths from below `start` to beyond `end` (between the centres), and with `boundaries` the centres,
    `start`, `end` and the half-way points exactly."""
    g = torch.Generator().manual_seed(seed)
    span = end - start
    r = start - 0.2 * span + torch.rand(count, generator=g, dtype=torch.float64) * 1.4 * span
    if boundaries:
        c = centres(start, end, n, cutoff)
        mids = (c[1:] + c[:-1]) / 2 if n > 1 else c
        r = torch.cat([r, c, mids, torch.tensor([start, end], dtype=torch.float64)])
    return r.to(dtype)


CASES = [(0.0, 5.0, 8), (0.5, 4.0, 2), (-1.0, 6.0, 10)]  # (start, end, n)


# ----------------------------------------------------------------------------------------------------------
# identities of the reference
# ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cutoff", [True, False])
def test_gaussian_peaks_at_one_over_1_12_on_each_centre(cutoff):
    for start, end, n in CASES:
        c = centres(start, end, n, cutoff)
        v = soft_one_hot_linspace(c, start, end, n, "gaussian", cutoff)
        assert torch.allclose(torch.diagonal(v), torch.full((n,), 1 / 1.12, dtype=torch.float64), rtol=0, atol=1e-15)
        grid = torch.linspace(start - 1, end + 1, 4001, dtype=torch.float64)
        assert float(soft_one_hot_linspace(grid, start, end, n, "gaussian", cutoff).max()) <= 1 / 1.12


@pytest.mark.parametrize("cutoff", [True, False])
def test_cosine_squares_sum_to_one_between_first_and_last_centre(cutoff):
    for start, end, n in CASES:
        c = centres(start, end, n, cutoff)
        r = torch.linspace(float(c[0]), float(c[-1]), 1001, dtype=torch.float64)
        s = soft_one_hot_linspace(r, start, end, n, "cosine", cutoff).pow(2).sum(-1)
        assert torch.allclose(s, torch.ones_like(s), rtol=0, atol=1e-14)


@pytest.mark.parametrize("cutoff", [True, False])
def test_smooth_finite_is_1_14136_on_a_centre_and_zero_from_one_step_away(cutoff):
    for start, end, n in CASES:
        c = centres(start, end, n, cutoff)
        v = soft_one_hot_linspace(c, start, end, n, "smooth_finite", cutoff)
        # 1.14136 e^2 e^-2, with e^2 rounded to fp32 as e3nn does
        assert torch.allclose(torch.diagonal(v), torch.full((n,), 1.14136, dtype=torch.float64), rtol=1e-6, atol=0)
        step = (end - start) / (n + 1 if cutoff else n - 1)
        r = torch.linspace(start - 2, end + 2, 2001, dtype=torch.float64)
        d = (r[:, None] - c) / step
        v = soft_one_hot_linspace(r, start, end, n, "smooth_finite", cutoff)
        far = d.abs() >= 1 + 1e-12
        assert far.any() and bool((v[far] == 0).all())
        assert bool((v[d.abs() < 0.99] > 0).all())  # closer to the edge exp(-1/t) underflows


@pytest.mark.parametrize("cutoff", [True, False])
def test_fourier_functions_are_orthogonal_on_the_interval(cutoff):
    for start, end, n in CASES:
        r = torch.linspace(start, end, 20001, dtype=torch.float64)
        f = soft_one_hot_linspace(r, start, end, n, "fourier", cutoff)
        w = torch.full((r.numel(),), (end - start) / (r.numel() - 1), dtype=torch.float64)
        w[0] = w[-1] = w[0] / 2  # trapezoid rule: exact to 1e-8 for these trigonometric products
        gram = f.T @ (f * w[:, None])
        diag = torch.diagonal(gram)
        assert float(diag.min()) > 0
        off = gram - torch.diag(diag)
        assert float(off.abs().max()) <= 1e-7 * float(diag.max()), gram


@pytest.mark.parametrize("basis,cutoff", list(itertools.product(BASES, [True, False])))
def test_reference_autograd_matches_central_differences(basis, cutoff):
    """d (R . f(r)) / d r through autograd against central differences (h = 1e-6, fp64), at lengths at least 1e-3
    away from every point where a mask switches; tolerance 1e-7 of max|gradient| (the O(h^2) truncation)."""
    for start, end, n in CASES:
        c = centres(start, end, n, cutoff)
        step = float(c[1] - c[0]) if n > 1 else (end - start) / 2
        r = lengths(start, end, n, cutoff, boundaries=False)
        kinks = torch.cat([c - step, c + step, torch.tensor([start, end], dtype=torch.float64)])
        r = r[(r[:, None] - kinks).abs().min(1).values > 1e-3]
        R = torch.randn(r.numel(), n, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
        rr = r.clone().requires_grad_(True)
        (g,) = torch.autograd.grad((soft_one_hot_linspace(rr, start, end, n, basis, cutoff) * R).sum(), rr)
        h = 1e-6
        fp = (soft_one_hot_linspace(r + h, start, end, n, basis, cutoff) * R).sum(-1)
        fm = (soft_one_hot_linspace(r - h, start, end, n, basis, cutoff) * R).sum(-1)
        fd = (fp - fm) / (2 * h)
        assert torch.isfinite(g).all()
        assert float((fd - g).abs().max()) <= 1e-7 * float(g.abs().max()), (start, end, n)


@pytest.mark.parametrize("basis,cutoff", list(itertools.product(BASES, [True, False])))
def test_reference_matches_e3nn(basis, cutoff):
    pytest.importorskip("e3nn")
    from e3nn.math import soft_one_hot_linspace as e3nn_soft_one_hot_linspace

    for dtype in (torch.float32, torch.float64):
        for start, end, n in CASES:
            r = lengths(start, end, n, cutoff, dtype)
            want = e3nn_soft_one_hot_linspace(r, start, end, n, basis, cutoff)
            assert torch.equal(soft_one_hot_linspace(r, start, end, n, basis, cutoff), want), (dtype, start, end, n)


def test_reference_rejects_an_unknown_basis():
    with pytest.raises(ValueError, match='basis="hat" is not a valid entry'):
        soft_one_hot_linspace(torch.ones(3), 0.0, 5.0, 8, "hat", True)


# ----------------------------------------------------------------------------------------------------------
# the kernels' basis functions, compiled for the host
# ----------------------------------------------------------------------------------------------------------
PRELUDE = r"""
#include <math.h>
#include <cmath>
#include <cstdio>
#define __device__
#define __forceinline__ inline
using std::exp;
using std::sqrt;
inline void sincos(float x, float* s, float* c) { sincosf(x, s, c); }
#include "soft_one_hot.cuh"
"""


def _host_basis(tmp_path, T: str, basis: str, cutoff: bool, start: float, end: float, n: int, r: torch.Tensor):
    """(values [len(r), n], d/dr [len(r), n]) of mt::soft_one_hot<T> for one basis."""
    body = (f"static const double R[{r.numel()}] = {{" + ", ".join(repr(float(x)) for x in r) + "};\n" + f"""
int main() {{
  for (int i = 0; i < {r.numel()}; ++i) {{
    const {T} x = ({T})R[i];
    for (int k = 0; k < {n}; ++k)
      std::printf("%.17g ", (double)mt::soft_one_hot<{T}, false>({MODES[basis]}, k, {n}, x, ({T}){start!r},
                                                                 ({T}){end!r}, {int(cutoff)}));
    for (int k = 0; k < {n}; ++k)
      std::printf("%.17g ", (double)mt::soft_one_hot<{T}, true>({MODES[basis]}, k, {n}, x, ({T}){start!r},
                                                                ({T}){end!r}, {int(cutoff)}));
    std::printf("\\n");
  }}
  return 0;
}}
""")
    src = tmp_path / "basis.cpp"
    src.write_text(PRELUDE + body)
    exe = tmp_path / "basis"
    subprocess.run(["g++", "-O1", "-std=c++17", "-I", CSRC, "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.strip().splitlines()
    rows = torch.tensor([[float(t) for t in line.split()] for line in out], dtype=torch.float64)
    return rows[:, :n], rows[:, n:]


def _normwise(a, b):
    return float((a - b).abs().max()) / max(float(b.abs().max()), 1e-300)


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
@pytest.mark.parametrize("basis,cutoff", list(itertools.product(list(MODES), [True, False])))
def test_kernel_basis_functions_match_the_reference(tmp_path, basis, cutoff):
    """Values (lengths below, between, beyond the centres and exactly on centres and boundaries) and derivatives (at
    the random lengths, where no mask switches) of the kernels' basis functions against the fp64 reference, evaluated
    on the lengths the kernel saw: fp64 within 1e-12 (normwise), fp32 within 1e-5 for the values and 2e-5 for the
    derivatives (eps(fp32) times the argument of exp / cos / sin)."""
    for start, end, n in CASES:
        for T, dtype in (("double", torch.float64), ("float", torch.float32)):
            r = lengths(start, end, n, cutoff, dtype).double()
            v, dv = _host_basis(tmp_path, T, basis, cutoff, start, end, n, r)
            want = soft_one_hot_linspace(r, start, end, n, basis, cutoff) * math.sqrt(n)
            vtol, gtol = (1e-12, 1e-12) if T == "double" else (1e-5, 2e-5)
            assert _normwise(v, want) < vtol, (T, start, end, n, _normwise(v, want))
            smooth = torch.arange(r.numel()) < 400  # the random lengths; a switching mask has no derivative
            rr = r[smooth].clone().requires_grad_(True)
            R = torch.randn(rr.numel(), n, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
            (g,) = torch.autograd.grad((soft_one_hot_linspace(rr, start, end, n, basis, cutoff) * R).sum(), rr)
            got = (dv[smooth] * R).sum(-1) / math.sqrt(n)
            assert _normwise(got, g) < gtol, (T, start, end, n, _normwise(got, g))


# ----------------------------------------------------------------------------------------------------------
# the product's module and factory (construction only: no kernels run)
# ----------------------------------------------------------------------------------------------------------
def test_edge_length_embedding_accepts_every_e3nn_basis_and_rejects_others():
    from matten_b200.nn.embedding import EdgeLengthEmbedding as ProductEmbedding

    for basis in BASES:
        m = ProductEmbedding(num_basis=8, basis=basis)
        assert m.basis == basis and m.state_dict() == {}
    with pytest.raises(ValueError, match='basis="gauss" is not a valid entry'):
        ProductEmbedding(basis="gauss")
    for basis in ("gaussian", "cosine", "smooth_finite"):
        with pytest.raises(ValueError, match="num_basis >= 2"):
            ProductEmbedding(num_basis=1, basis=basis, cutoff=False)
        ProductEmbedding(num_basis=1, basis=basis, cutoff=True)


def test_model_configs_differing_only_in_the_basis_build():
    from matten_b200.model_factory import ScalarTensorModel
    from tests.helpers import HP_LMAX2, SPECIES8

    sd = None
    for basis in BASES:
        torch.manual_seed(0)
        model = ScalarTensorModel(dict(HP_LMAX2, radial_basis_type=basis), {"allowed_species": SPECIES8})
        assert model.backbone.radial_basis.basis == basis
        keys = sorted(model.state_dict())
        assert sd is None or keys == sd  # the basis carries no parameters or buffers
        sd = keys
    # the factory reports which module failed (model_factory/utils.py), with the ValueError as the cause
    with pytest.raises(RuntimeError, match="EdgeLengthEmbedding") as info:
        ScalarTensorModel(dict(HP_LMAX2, radial_basis_type="Gaussian"), {"allowed_species": SPECIES8})
    assert isinstance(info.value.__cause__, ValueError)
    assert str(info.value.__cause__) == 'basis="Gaussian" is not a valid entry'


def test_custom_op_infers_the_shape_of_every_mode_on_meta():
    from matten_b200 import torch_ops  # noqa: F401  (registers the ops)

    for mode in (3, 4, 5, 6):
        out = torch.ops.matten_b200.edge_radial(torch.empty(7, device="meta"), mode, 10, -1.0, 6.0, False, 6.0)
        assert out.shape == (7, 10)
