"""
Differentiable front-end of the CUDA ops (``matten_b200.ops``).

Every function dispatches to a hand-written kernel through the C ABI; when autograd is
recording and an input requires grad, the op is recorded as a ``torch.autograd.Function``
whose backward is again a C-ABI kernel (see ``matten_b200/autograd.py``).
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch

from . import ops


def _needs_grad(*ts) -> bool:
    return torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in ts)


# ---- geometry (first derivatives w.r.t. positions, cell and edge vectors are recorded when requested) ----
def edge_vectors(pos, edge_index, shift, cell, batch, flag, graph=None):
    """(vec, len) of every edge.  ``graph`` (a GraphCache of ``edge_index``) supplies the CSRs of the backward; one
    is built when it is not given and a gradient is recorded."""
    if _needs_grad(pos, cell):
        from . import autograd as A
        from .graph import GraphCache

        if graph is None:
            graph = GraphCache({"edge_index": edge_index, "pos": pos})
        return A.EdgeVectorsFn.apply(pos, cell, graph, shift, batch)
    return ops.edge_vectors(pos.detach(), edge_index, shift, None if cell is None else cell.detach(), batch, flag)


def vector_lengths(vec):
    """|v| for precomputed edge vectors (reference _nequip.py:226-231) through the same kernel:
    pos = 0, shift = v, cell = I."""
    if _needs_grad(vec):
        from . import autograd as A

        return A.VectorLengthsFn.apply(vec)
    E = vec.shape[0]
    z = torch.zeros((1, 3), dtype=vec.dtype, device=vec.device)
    ei = torch.zeros((2, E), dtype=torch.int64, device=vec.device)
    eye = torch.eye(3, dtype=vec.dtype, device=vec.device)
    _, ln = ops.edge_vectors(z, ei, vec.contiguous(), eye, None, None, want_vec=False)
    return ln


def edge_sh(vec, lmax: int, normalize: bool = True):
    if _needs_grad(vec):
        from . import autograd as A

        return A.EdgeShFn.apply(vec, lmax, normalize)
    return ops.edge_sh(vec.detach(), lmax, normalize)


def edge_radial(length, mode, num_basis, start, end, cutoff=True, poly_p=6.0, bessel_w=None):
    if _needs_grad(bessel_w) and mode != 1:
        raise ValueError("trainable frequencies belong to the BesselBasis encoding (mode 1)")
    if _needs_grad(length, bessel_w):
        from . import autograd as A

        return A.EdgeRadialFn.apply(length, bessel_w, mode, num_basis, start, end, cutoff, poly_p)
    bw = bessel_w.detach() if bessel_w is not None else None
    return ops.edge_radial(length.detach(), mode, num_basis, start, end, cutoff, poly_p, bw)


def species_embed(Z, idx, lut, zmin, zmax, S, lin_w, lin_b, flag):
    if _needs_grad(lin_w, lin_b):
        from . import autograd as A

        return A.species_embed(Z, idx, lut, zmin, zmax, S, lin_w, lin_b, flag)
    return ops.species_embed(Z, idx, lut, zmin, zmax, S, lin_w.detach(), lin_b.detach(), flag)


def linear(handle: ops.LinPlanHandle, x, weight, species_perm=None, species_ptr=None, residual=None):
    """``residual + L(x)`` when ``residual`` is given (fused accumulate), else ``L(x)``."""
    if _needs_grad(x, weight, residual):
        from . import autograd as A

        return A.LinearFn.apply(x, weight, residual, handle, species_perm, species_ptr)
    if residual is not None:
        # the caller hands over ownership of `residual` (a fresh temporary): accumulate in place
        return ops.linear_fwd(handle, x.detach(), weight.detach(), species_perm, species_ptr, out=residual,
                              accumulate=True)
    return ops.linear_fwd(handle, x.detach(), weight.detach(), species_perm, species_ptr)


def _layout(graph, sh, handle):
    """The batch's shared tensor-core layout (GraphCache.conv_layout), when the graph object keeps one."""
    f = getattr(graph, "conv_layout", None)
    return f(sh, handle.tc_y_lmax) if f is not None else None


def conv(handle: ops.ConvPlanHandle, x, sh, emb, mlp_weights: Sequence[torch.Tensor], graph,
         avg_num_neighbors: Optional[float], num_neigh=None):
    if _needs_grad(x, sh, emb, *mlp_weights):
        from . import autograd as A

        return A.ConvFn.apply(x, sh, emb, handle, graph, avg_num_neighbors, num_neigh, *mlp_weights)
    return ops.conv_fwd(handle, x.detach(), sh.detach(), emb.detach(), [w.detach() for w in mlp_weights], graph.rowptr,
                        graph.perm, graph.src_sorted, avg_num_neighbors, num_neigh, layout=_layout(graph, sh, handle))


def gate(x, tables, affine_a=None, affine_b=None):
    """tables = (in_dim, out_dim, src_idx, gate_idx, act_id, act_cst)"""
    if _needs_grad(affine_a, affine_b):
        from . import autograd as A

        # trainable affine (BatchNorm parameters in eval mode under autograd): unfused gate, then affine
        return A.AffineFn.apply(A.GateFn.apply(x, None, None, tables), affine_a, affine_b)
    if _needs_grad(x):
        from . import autograd as A

        return A.GateFn.apply(x, affine_a, affine_b, tables)
    in_dim, out_dim, src, gidx, act, cst = tables[:6]
    return ops.gate_fwd(x.detach(), in_dim, out_dim, src, gidx, act, cst,
                        None if affine_a is None else affine_a.detach(),
                        None if affine_b is None else affine_b.detach())


def segment_reduce(x, ptr, reduce: str):
    if _needs_grad(x):
        from . import autograd as A

        return A.SegmentReduceFn.apply(x, ptr, reduce)
    return ops.segment_reduce(x.detach(), ptr, reduce)
