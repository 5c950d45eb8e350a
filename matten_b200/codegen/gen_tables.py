"""
Generates ``matten_b200/csrc/generated/cg_gen.cuh``: fully unrolled Clebsch-Gordan
contractions per (l1, l2, l3) with the coefficients as literals, and the real
spherical-harmonic polynomials up to ``LMAX``.

The reference gets the same arithmetic from e3nn's TorchScript codegen (one
einsum per instruction over a dense w3j buffer: reference
src/matten/nn/utils.py:230-237 -> e3nn.o3.TensorProduct); here every non-zero of
the real Wigner-3j tensor becomes one FMA with an immediate operand.

Run:  python -m matten_b200.codegen.gen_tables
"""
from __future__ import annotations

import math
import os

import torch

from .. import o3

LMAX = 4
EPS = 1e-12


def cg_types(lmax: int = LMAX):
    out = []
    for l1 in range(lmax + 1):
        for l2 in range(lmax + 1):
            for l3 in range(abs(l1 - l2), min(lmax, l1 + l2) + 1):
                out.append((l1, l2, l3))
    return out


def _lit(c: float) -> str:
    return f"T({c!r})"


def _emit_cg(l1, l2, l3) -> str:
    C = o3.wigner_3j(l1, l2, l3) * math.sqrt(2 * l3 + 1)  # path normalisation folded in
    d1, d2, d3 = 2 * l1 + 1, 2 * l2 + 1, 2 * l3 + 1
    nz = [(a, b, c, C[a, b, c].item()) for a in range(d1) for b in range(d2) for c in range(d3)
          if abs(C[a, b, c].item()) > EPS]
    L = []
    L.append(f"template <> struct CG<{l1}, {l2}, {l3}> {{")
    L.append(f"  static constexpr int D1 = {d1}, D2 = {d2}, D3 = {d3}, NNZ = {len(nz)};")

    # ---- fwd: acc[c] += w * sum C x[a] y[b]
    L.append("  template <typename T> static __device__ __forceinline__ void fwd(const T* __restrict__ x, const T* __restrict__ y, T w, T* __restrict__ acc) {")
    pairs = {}
    for a, b, c, v in nz:
        pairs.setdefault((a, b), []).append((c, v))
    if d1 <= d3:
        for a in range(d1):
            L.append(f"    const T xw{a} = w * x[{a}];")
        for (a, b), lst in pairs.items():
            if len(lst) == 1:
                c, v = lst[0]
                L.append(f"    acc[{c}] = fma({_lit(v)} * xw{a}, y[{b}], acc[{c}]);")
            else:
                L.append(f"    {{ const T p = xw{a} * y[{b}];")
                for c, v in lst:
                    L.append(f"      acc[{c}] = fma({_lit(v)}, p, acc[{c}]);")
                L.append("    }")
    else:
        for c in range(d3):
            L.append(f"    T t{c} = T(0);")
        for (a, b), lst in pairs.items():
            if len(lst) == 1:
                c, v = lst[0]
                L.append(f"    t{c} = fma({_lit(v)} * x[{a}], y[{b}], t{c});")
            else:
                L.append(f"    {{ const T p = x[{a}] * y[{b}];")
                for c, v in lst:
                    L.append(f"      t{c} = fma({_lit(v)}, p, t{c});")
                L.append("    }")
        for c in range(d3):
            L.append(f"    acc[{c}] = fma(w, t{c}, acc[{c}]);")
    L.append("  }")

    # ---- dot: returns sum C x[a] y[b] g[c]   (d loss / d w)
    L.append("  template <typename T> static __device__ __forceinline__ T dot(const T* __restrict__ x, const T* __restrict__ y, const T* __restrict__ g) {")
    L.append("    T s = T(0);")
    bc = {}
    for a, b, c, v in nz:
        bc.setdefault((b, c), []).append((a, v))
    # s = sum_a x[a] * (sum_{b,c} C y[b] g[c])
    for a in range(d1):
        terms = [(b, c, v) for (a2, b, c, v) in nz if a2 == a]
        if not terms:
            continue
        L.append("    { T q = T(0);")
        for b, c, v in terms:
            L.append(f"      q = fma({_lit(v)} * y[{b}], g[{c}], q);")
        L.append(f"      s = fma(x[{a}], q, s); }}")
    L.append("    return s;")
    L.append("  }")

    # ---- bwd_x: dx[a] += w * sum C y[b] g[c]
    L.append("  template <typename T> static __device__ __forceinline__ void bwd_x(const T* __restrict__ y, const T* __restrict__ g, T w, T* __restrict__ dx) {")
    for a in range(d1):
        terms = [(b, c, v) for (a2, b, c, v) in nz if a2 == a]
        if not terms:
            continue
        L.append("    { T q = T(0);")
        for b, c, v in terms:
            L.append(f"      q = fma({_lit(v)} * y[{b}], g[{c}], q);")
        L.append(f"      dx[{a}] = fma(w, q, dx[{a}]); }}")
    L.append("  }")

    # ---- bwd_y: dy[b] += w * sum C x[a] g[c]
    L.append("  template <typename T> static __device__ __forceinline__ void bwd_y(const T* __restrict__ x, const T* __restrict__ g, T w, T* __restrict__ dy) {")
    for b in range(d2):
        terms = [(a, c, v) for (a, b2, c, v) in nz if b2 == b]
        if not terms:
            continue
        L.append("    { T q = T(0);")
        for a, c, v in terms:
            L.append(f"      q = fma({_lit(v)} * x[{a}], g[{c}], q);")
        L.append(f"      dy[{b}] = fma(w, q, dy[{b}]); }}")
    L.append("  }")
    L.append("};")
    return "\n".join(L)


def _sh_recursion_coeff(l: int) -> torch.Tensor:
    """C[k,i,j] with Y_{l+1}[k] = sum C[k,i,j] Y_1[i] Y_l[j] for unit-norm ('norm')
    harmonics of a unit vector, sign fixed by Y_{l+1}(e_y)[m=0] = +1."""
    C = o3.wigner_3j(l + 1, 1, l)
    y1 = torch.tensor([0.0, 1.0, 0.0], dtype=torch.float64)
    yl = torch.zeros(2 * l + 1, dtype=torch.float64)
    yl[l] = 1.0
    v = torch.einsum("kij,i,j->k", C, y1, yl)
    return C / v[l + 1]


def _emit_sh(lmax: int) -> str:
    L = []
    L.append("// Real spherical harmonics of a UNIT vector (x,y,z), e3nn basis (y polar axis),")
    L.append("// 'component' normalisation (|Y_l|^2 = 2l+1).  out has (lmax+1)^2 entries.")
    L.append("template <int LMAXV, typename T> __device__ __forceinline__ void sh_component(T x, T y, T z, T* __restrict__ out) {")
    L.append("  out[0] = T(1);")
    L.append("  if constexpr (LMAXV >= 1) {")
    L.append("    const T n1[3] = {x, y, z};")
    L.append(f"    out[1] = {_lit(math.sqrt(3.0))} * x; out[2] = {_lit(math.sqrt(3.0))} * y; out[3] = {_lit(math.sqrt(3.0))} * z;")
    prev = "n1"
    for l in range(1, lmax):
        C = _sh_recursion_coeff(l)
        d = 2 * (l + 1) + 1
        L.append(f"    if constexpr (LMAXV >= {l + 1}) {{")
        L.append(f"      T n{l + 1}[{d}];")
        for k in range(d):
            terms = []
            for i in range(3):
                for j in range(2 * l + 1):
                    v = C[k, i, j].item()
                    if abs(v) > EPS:
                        terms.append(f"{_lit(v)} * n1[{i}] * {prev}[{j}]")
            L.append(f"      n{l + 1}[{k}] = " + " + ".join(terms) + ";")
        base = (l + 1) ** 2
        s = math.sqrt(2 * (l + 1) + 1)
        L.append(f"      #pragma unroll\n      for (int k = 0; k < {d}; ++k) out[{base} + k] = {_lit(s)} * n{l + 1}[k];")
        prev = f"n{l + 1}"
    for l in range(1, lmax):
        L.append("    }")
    L.append("  }")
    L.append("}")
    return "\n".join(L)


def _emit_sh_vjp(lmax: int) -> str:
    """Forward-mode tangents through the recursion of ``_emit_sh``, one per input axis d, contracted with the
    output gradient: gu[d] = sum_k g[k] d out[k] / d u_d (u the unit vector; no normalisation)."""
    L = []
    L.append("// gu[d] = sum_k g[k] d sh_component(u)[k] / d u_d for d = 0, 1, 2 (vector-Jacobian product of sh_component).")
    L.append("template <int LMAXV, typename T> __device__ __forceinline__ void sh_component_vjp(T x, T y, T z, const T* __restrict__ g, T* __restrict__ gu) {")
    L.append("  gu[0] = T(0); gu[1] = T(0); gu[2] = T(0);")
    L.append("  if constexpr (LMAXV >= 1) {")
    L.append("    const T n1[3] = {x, y, z};")
    L.append("    #pragma unroll")
    L.append("    for (int d = 0; d < 3; ++d) {")
    L.append("      const T t1[3] = {T(d == 0 ? 1 : 0), T(d == 1 ? 1 : 0), T(d == 2 ? 1 : 0)};")
    L.append(f"      T s = {_lit(math.sqrt(3.0))} * (g[1] * t1[0] + g[2] * t1[1] + g[3] * t1[2]);")
    prev, tprev = "n1", "t1"
    for l in range(1, lmax):
        C = _sh_recursion_coeff(l)
        d = 2 * (l + 1) + 1
        L.append(f"      if constexpr (LMAXV >= {l + 1}) {{")
        L.append(f"        T n{l + 1}[{d}], t{l + 1}[{d}];")
        for k in range(d):
            terms, tterms = [], []
            for i in range(3):
                for j in range(2 * l + 1):
                    v = C[k, i, j].item()
                    if abs(v) > EPS:
                        terms.append(f"{_lit(v)} * n1[{i}] * {prev}[{j}]")
                        tterms.append(f"{_lit(v)} * (t1[{i}] * {prev}[{j}] + n1[{i}] * {tprev}[{j}])")
            L.append(f"        n{l + 1}[{k}] = " + " + ".join(terms) + ";")
            L.append(f"        t{l + 1}[{k}] = " + " + ".join(tterms) + ";")
        base = (l + 1) ** 2
        L.append(f"        T q = T(0);\n        #pragma unroll\n        for (int k = 0; k < {d}; ++k) q = fma(g[{base} + k], t{l + 1}[k], q);")
        L.append(f"        s = fma({_lit(math.sqrt(2 * (l + 1) + 1))}, q, s);")
        prev, tprev = f"n{l + 1}", f"t{l + 1}"
    for l in range(1, lmax):
        L.append("      }")
    L.append("      gu[d] = s;")
    L.append("    }")
    L.append("  }")
    L.append("}")
    return "\n".join(L)


def generate() -> str:
    types = cg_types()
    L = []
    L.append("// AUTO-GENERATED by matten_b200/codegen/gen_tables.py -- do not edit by hand.")
    L.append("// Real Wigner-3j contractions (e3nn 0.5.x conventions) with sqrt(2*l3+1) folded in,")
    L.append("// one specialisation per (l1,l2,l3), every non-zero an FMA with a literal operand.")
    L.append("#pragma once")
    L.append("namespace mt {")
    L.append(f"constexpr int kLmax = {LMAX};")
    L.append(f"constexpr int kNumCgTypes = {len(types)};")
    L.append("template <int L1, int L2, int L3> struct CG;")
    for t in types:
        L.append(_emit_cg(*t))
    L.append("// X(type_id, l1, l2, l3)")
    L.append("#define MT_FOR_EACH_CG_TYPE(X) \\")
    for i, (a, b, c) in enumerate(types):
        L.append(f"  X({i}, {a}, {b}, {c}) \\")
    L.append("")
    L.append("// the same, restricted to l1, l2, l3 <= 2 (the tcgen05 convolution kernel)")
    L.append("#define MT_FOR_EACH_CG_TYPE_L2(X) \\")
    for i, (a, b, c) in enumerate(types):
        if max(a, b, c) <= 2:
            L.append(f"  X({i}, {a}, {b}, {c}) \\")
    L.append("")
    L.append("__host__ __device__ constexpr int cg_type_id(int l1, int l2, int l3) {")
    L.append("  switch (l1 * 100 + l2 * 10 + l3) {")
    for i, (a, b, c) in enumerate(types):
        L.append(f"    case {a * 100 + b * 10 + c}: return {i};")
    L.append("    default: return -1;")
    L.append("  }")
    L.append("}")
    L.append(_emit_sh(LMAX))
    L.append(_emit_sh_vjp(LMAX))
    L.append("}  // namespace mt")
    return "\n".join(L) + "\n"


def cg_type_id(l1: int, l2: int, l3: int) -> int:
    return cg_types().index((l1, l2, l3))


def cg_nnz(l1: int, l2: int, l3: int) -> int:
    return int((o3.wigner_3j(l1, l2, l3).abs() > EPS).sum())


def main():
    here = os.path.dirname(os.path.abspath(__file__))
    out = os.path.join(here, "..", "csrc", "generated", "cg_gen.cuh")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    src = generate()
    with open(out, "w") as f:
        f.write(src)
    print(f"wrote {os.path.normpath(out)}: {len(cg_types())} CG types, {len(src.splitlines())} lines")


if __name__ == "__main__":
    main()
