"""CPU checks of the pieces of the position / cell gradient that do not need a GPU.

* The generated ``CG<l1,l2,l3>::bwd_y`` and ``sh_component_vjp`` (matten_b200/codegen/gen_tables.py) are compiled for
  the host with g++ (the CUDA qualifiers defined away) in double precision and compared with the oracle:
  bwd_y against sqrt(2 l3 + 1) w einsum(w3j, x, g) for all 65 CG types, the SH vector-Jacobian product against
  autograd through ``E.spherical_harmonics`` for l <= 4, at random directions and next to the poles.
* Autograd through the oracle model (the parity target of the CUDA backward) agrees with central finite differences
  for the positions and the cell of a small periodic crystal.
"""
import math
import os
import shutil
import subprocess

import pytest
import torch

from matten_b200.codegen import gen_tables
from oracle import e3nn_restated as E

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER_DIR = os.path.join(ROOT, "matten_b200", "csrc", "generated")

PRELUDE = r"""
#include <cmath>
#include <cstdio>
#define __device__
#define __host__
#define __forceinline__ inline
#define __restrict__
using std::fma;
#include "cg_gen.cuh"
using namespace mt;
"""


def _c_array(name, vals):
    return f"static const double {name}[{len(vals)}] = {{" + ", ".join(repr(float(v)) for v in vals) + "};\n"


def _run(tmp_path, body: str, name: str):
    src = tmp_path / f"{name}.cpp"
    src.write_text(PRELUDE + body)
    exe = tmp_path / name
    subprocess.run(["g++", "-O1", "-std=c++17", "-I", HEADER_DIR, "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.strip().splitlines()
    return [[float(t) for t in line.split()] for line in out]


def test_generated_header_is_current():
    with open(os.path.join(HEADER_DIR, "cg_gen.cuh")) as f:
        assert f.read() == gen_tables.generate(), "run python -m matten_b200.codegen.gen_tables"


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
def test_cg_bwd_y_matches_the_dense_contraction(tmp_path):
    """dy[m2] = w sum_{m1,m3} sqrt(2 l3 + 1) C[m1,m2,m3] x[m1] g[m3]; tolerance 1e-13 absolute on O(1) values
    (a few ulps of fp64 over at most 9 x 9 products)."""
    g = torch.Generator().manual_seed(0)
    x = torch.rand(9, generator=g, dtype=torch.float64) * 2 - 1
    gg = torch.rand(9, generator=g, dtype=torch.float64) * 2 - 1
    w = 0.73
    body = _c_array("X", x.tolist()) + _c_array("G", gg.tolist()) + r"""
template <int A, int B, int C> void run(int id) {
  double dy[2 * B + 1];
  for (int i = 0; i < 2 * B + 1; ++i) dy[i] = 0.125;  // bwd_y accumulates
  CG<A, B, C>::template bwd_y<double>(X, G, 0.73, dy);
  std::printf("%d", id);
  for (int i = 0; i < 2 * B + 1; ++i) std::printf(" %.17g", dy[i] - 0.125);
  std::printf("\n");
}
int main() {
#define X_(ID, A, B, C) run<A, B, C>(ID);
  MT_FOR_EACH_CG_TYPE(X_)
  return 0;
}
"""
    rows = _run(tmp_path, body, "bwd_y")
    types = gen_tables.cg_types()
    assert len(rows) == len(types) == 65
    for row, (l1, l2, l3) in zip(rows, types):
        C = E.wigner_3j(l1, l2, l3).double() * math.sqrt(2 * l3 + 1)
        want = w * torch.einsum("abc,a,c->b", C, x[:2 * l1 + 1], gg[:2 * l3 + 1])
        got = torch.tensor(row[1:], dtype=torch.float64)
        assert int(row[0]) == types.index((l1, l2, l3))
        assert torch.allclose(got, want, rtol=0, atol=1e-13), ((l1, l2, l3), (got - want).abs().max())


def _directions():
    g = torch.Generator().manual_seed(1)
    v = torch.randn(24, 3, generator=g, dtype=torch.float64)
    poles = torch.tensor([[0.0, 1.0, 0.0], [0.0, -1.0, 0.0], [1e-9, 1.0, -2e-9], [0.0, 0.0, 1.0], [1.0, 0.0, 0.0],
                          [-3e-8, -1.0, 1e-8]], dtype=torch.float64)
    v = torch.cat([v, poles])
    return v / v.norm(dim=1, keepdim=True)


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
@pytest.mark.parametrize("lmax", [0, 1, 2, 3, 4])
def test_sh_vjp_matches_oracle_autograd(tmp_path, lmax):
    """sum_k g[k] d Y_k(u) / d u against autograd of E.spherical_harmonics (no normalisation: the polynomials are
    homogeneous, so the recursion and e3nn's explicit forms agree off the sphere too).  Tolerance: 1e-12 of
    max|gradient| per direction in fp64."""
    u = _directions()
    D = (lmax + 1) ** 2
    gsh = torch.rand(u.shape[0], D, generator=torch.Generator().manual_seed(2), dtype=torch.float64) * 2 - 1
    body = (_c_array("U", u.reshape(-1).tolist()) + _c_array("GS", gsh.reshape(-1).tolist()) + f"""
int main() {{
  for (int i = 0; i < {u.shape[0]}; ++i) {{
    double gu[3];
    sh_component_vjp<{lmax}, double>(U[3 * i], U[3 * i + 1], U[3 * i + 2], GS + {D} * i, gu);
    std::printf("%.17g %.17g %.17g\\n", gu[0], gu[1], gu[2]);
  }}
  return 0;
}}
""")
    got = torch.tensor(_run(tmp_path, body, f"shvjp{lmax}"), dtype=torch.float64)
    ur = u.clone().requires_grad_(True)
    sh = E.spherical_harmonics(lmax, ur, False, "component")
    (want,) = torch.autograd.grad((sh * gsh).sum() + 0 * ur.sum(), ur)  # l = 0 alone does not depend on u
    for i in range(u.shape[0]):
        scale = max(float(want[i].abs().max()), 1.0)
        assert float((got[i] - want[i]).abs().max()) <= 1e-12 * scale, (lmax, u[i], got[i], want[i])


def test_oracle_autograd_matches_finite_differences():
    """The parity target itself: d (R . out) / d pos and / d cell of the oracle's lmax-2 model on the 8-atom
    reference crystal against central differences (h = 1e-5, fp64; the neighbour list is held fixed, as in the
    reference).  Tolerance 1e-6 of max|gradient|: the O(h^2) truncation error of the difference quotients."""
    from oracle import matten_restated as M
    from tests.helpers import HP_LMAX2, load_reference_test_crystal, randomize_bn

    dtype = torch.float64
    batch, d = load_reference_test_crystal(dtype)
    species = sorted(set(d["atomic_numbers"]))
    torch.manual_seed(0)
    old = torch.get_default_dtype()
    torch.set_default_dtype(dtype)
    try:
        model = M.ScalarTensorModel(HP_LMAX2, {"allowed_species": species}).eval()
    finally:
        torch.set_default_dtype(old)
    randomize_bn(model, 0)
    base = {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in batch.items() if isinstance(v, torch.Tensor)}
    key = "elastic_tensor_full"
    R = None

    def f(pos, cell):
        nonlocal R
        out = model(dict(base, pos=pos, cell=cell))
        out = out[key] if isinstance(out, dict) else out
        if R is None:
            R = torch.randn(out.shape, generator=torch.Generator().manual_seed(3), dtype=dtype)
        return (out * R).sum()

    pos = base["pos"].clone().requires_grad_(True)
    cell = base["cell"].clone().requires_grad_(True)
    gp, gc = torch.autograd.grad(f(pos, cell), (pos, cell))
    h = 1e-5
    with torch.no_grad():
        for t, grad in ((base["pos"], gp), (base["cell"], gc)):
            fd = torch.zeros_like(t)
            for i in range(t.numel()):
                tp, tm = t.clone(), t.clone()
                tp.view(-1)[i] += h
                tm.view(-1)[i] -= h
                args_p = (tp, base["cell"]) if t is base["pos"] else (base["pos"], tp)
                args_m = (tm, base["cell"]) if t is base["pos"] else (base["pos"], tm)
                fd.view(-1)[i] = (f(*args_p) - f(*args_m)) / (2 * h)
            scale = float(grad.abs().max())
            assert scale > 0
            assert float((fd - grad).abs().max()) <= 1e-6 * scale, (fd, grad)
