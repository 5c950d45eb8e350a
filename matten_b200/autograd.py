"""
Autograd bindings of the CUDA ops: every ``torch.autograd.Function`` below runs hand-written kernels through the
C ABI in both directions (``ops.*_fwd`` / ``ops.*_bwd``).  torch only records the graph and owns the memory.

Gradients are produced for what the reference trains (model/model.py: every ``nn.Parameter`` of the backbone and
the heads), for node features, and -- first derivatives only -- for the geometry: the convolution passes gradients to
its edge inputs (spherical harmonics, radial embedding), and ``EdgeShFn`` / ``EdgeRadialFn`` / ``EdgeVectorsFn`` carry
them on to edge vectors, positions and the cell.  The geometry functions are ``once_differentiable``: a second
derivative through them (energy / force-style training) raises instead of returning silent zeros.
"""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable

from . import ops


def _first_order(backward):
    """Backward of a geometry function: first derivatives only.  ``create_graph=True`` raises here (``torch`` runs a
    backward with grad mode on exactly then) instead of leaving a gradient that a second backward cannot follow."""

    def wrapper(ctx, *grads):
        if torch.is_grad_enabled():
            raise RuntimeError("matten_b200: second derivatives through the geometry (create_graph=True) are not "
                               "supported")
        return backward(ctx, *grads)

    return wrapper


def _sender_csr(graph, N: int):
    f = getattr(graph, "sender_csr", None)
    if f is not None:
        return f()
    ptr, perm = ops.csr_by_key(graph.src_sorted.to(torch.int64), N, True, None)
    return ptr, perm


class ConvFn(torch.autograd.Function):
    """fused radial MLP -> uvu tensor product -> receiver sum (reference nn/conv.py:111-120, nn/utils.py:255-263)."""

    @staticmethod
    def forward(ctx, x, sh, emb, handle, graph, avg, num_neigh, *mlp_weights):
        ws = [w.detach() for w in mlp_weights]
        from .functional import _layout

        out = ops.conv_fwd(handle, x.detach(), sh.detach(), emb.detach(), ws, graph.rowptr, graph.perm,
                           graph.src_sorted, avg, num_neigh, layout=_layout(graph, sh.detach(), handle))
        ctx.handle, ctx.graph, ctx.avg = handle, graph, avg
        ctx.nw = len(ws)
        ctx.save_for_backward(x, sh, emb, num_neigh if num_neigh is not None else x.new_empty(0), *mlp_weights)
        return out

    @staticmethod
    def backward(ctx, g):
        x, sh, emb, nn_, *ws = ctx.saved_tensors
        num_neigh = nn_ if nn_.numel() else None
        need_x, need_sh, need_emb = ctx.needs_input_grad[:3]
        need_w = any(ctx.needs_input_grad[7:])
        graph = ctx.graph
        sptr, sperm = _sender_csr(graph, x.shape[0]) if need_x else (None, None)
        gx, gws, gsh, gemb = ops.conv_bwd_full(ctx.handle, x.detach(), sh.detach(), emb.detach(),
                                               [w.detach() for w in ws], graph.rowptr, graph.perm, graph.src_sorted,
                                               sptr, sperm, ctx.avg, num_neigh, g.contiguous(), need_x, need_w,
                                               need_sh, need_emb)
        if gws is None:
            gws = [None] * ctx.nw
        return (gx, gsh, gemb, None, None, None, None, *gws)


class LinearFn(torch.autograd.Function):
    """species-indexed irreps linear (+ fused residual add): ``residual + L(x)``."""

    @staticmethod
    def forward(ctx, x, weight, residual, handle, species_perm, species_ptr):
        ctx.handle, ctx.sp = handle, (species_perm, species_ptr)
        ctx.save_for_backward(x, weight)
        if residual is not None:
            out = residual.detach().clone()  # the residual may be needed by nobody, but never write a saved tensor
            ops.linear_fwd(handle, x.detach(), weight.detach(), species_perm, species_ptr, out=out.reshape(-1, handle.out_dim),
                           accumulate=True)
            return out
        return ops.linear_fwd(handle, x.detach(), weight.detach(), species_perm, species_ptr)

    @staticmethod
    def backward(ctx, g):
        x, weight = ctx.saved_tensors
        g = g.contiguous()
        gx, gw = ops.linear_bwd(ctx.handle, x.detach(), weight.detach(), g, ctx.sp[0], ctx.sp[1],
                                need_x=ctx.needs_input_grad[0], need_w=ctx.needs_input_grad[1])
        if gw is not None:
            gw = gw.reshape(weight.shape)
        return gx, gw, (g if ctx.needs_input_grad[2] else None), None, None, None


class GateFn(torch.autograd.Function):
    """e3nn Gate (+ constant per-element affine).  tables = (in_dim, out_dim, src, gate, act, cst, inv_first, inv_count)."""

    @staticmethod
    def forward(ctx, x, affine_a, affine_b, tables):
        in_dim, out_dim, src, gidx, act, cst = tables[:6]
        ctx.tables = tables
        a = None if affine_a is None else affine_a.detach()
        b = None if affine_b is None else affine_b.detach()
        ctx.save_for_backward(x, a if a is not None else x.new_empty(0))
        return ops.gate_fwd(x.detach(), in_dim, out_dim, src, gidx, act, cst, a, b)

    @staticmethod
    def backward(ctx, g):
        x, a = ctx.saved_tensors
        in_dim, out_dim, src, gidx, act, cst, inv_first, inv_count = ctx.tables
        gx = ops.gate_bwd(x.detach(), g.contiguous(), in_dim, out_dim, src, gidx, act, cst, inv_first, inv_count,
                          a if a.numel() else None)
        return gx, None, None, None


class AffineFn(torch.autograd.Function):
    """y[n,j] = a[j] x[n,j] + b[j] with gradients to x, a and b (eval-mode BatchNorm under autograd)."""

    @staticmethod
    def forward(ctx, x, a, b):
        ctx.save_for_backward(x, a)
        return ops.affine2(x.detach(), a.detach().contiguous(), None, None, b.detach().contiguous())

    @staticmethod
    def backward(ctx, g):
        x, a = ctx.saved_tensors
        g = g.contiguous()
        gx = ops.affine2(g, a.detach().contiguous()) if ctx.needs_input_grad[0] else None
        ga = ops.col_reduce(g, None, x.detach(), None) if ctx.needs_input_grad[1] else None
        gb = ops.col_reduce(g) if ctx.needs_input_grad[2] else None
        return gx, ga, gb


class SegmentReduceFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, ptr, reduce):
        ctx.ptr, ctx.reduce, ctx.N = ptr, reduce, x.shape[0]
        if reduce in ("min", "max"):
            ctx.save_for_backward(x)
        return ops.segment_reduce(x.detach(), ptr, reduce)

    @staticmethod
    def backward(ctx, g):
        if ctx.reduce in ("min", "max"):
            (x,) = ctx.saved_tensors
            return ops.segment_extreme_bwd(x.detach(), g.contiguous(), ctx.ptr, ctx.reduce), None, None
        return ops.segment_reduce_bwd(g.contiguous(), ctx.ptr, ctx.N, ctx.reduce), None, None


class EdgeRadialFn(torch.autograd.Function):
    """Radial basis of the edge lengths (ops.edge_radial, modes 0, 1 and 3-6) with gradients to the lengths and, for
    the trainable BesselBasis (reference src/matten/nn/_nequip.py:80-126), to the frequencies:
    d out[e,k] / d w_k = (2 / r_max^2) cos(w_k r / r_max) env(r), summed over edges in fixed order."""

    @staticmethod
    def forward(ctx, length, bessel_w, mode, num_basis, start, end, cutoff, poly_p):
        ctx.args = (mode, num_basis, start, end, cutoff, poly_p)
        bw = None if bessel_w is None else bessel_w.detach()
        ctx.save_for_backward(length, bw)
        return ops.edge_radial(length.detach(), mode, num_basis, start, end, cutoff, poly_p, bw)

    @staticmethod
    @_first_order
    @once_differentiable
    def backward(ctx, g):
        length, w = ctx.saved_tensors
        mode, num_basis, start, end, cutoff, poly_p = ctx.args
        g = g.contiguous()
        glen = gw = None
        if ctx.needs_input_grad[0]:
            glen = ops.edge_radial_bwd(length, g, mode, num_basis, start, end, cutoff, poly_p, w)
        if ctx.needs_input_grad[1]:
            dw = ops.edge_radial(length, 2, num_basis, start, end, cutoff, poly_p, w)
            gw = ops.col_reduce(g, None, dw, None)
        return glen, gw, None, None, None, None, None, None


class EdgeShFn(torch.autograd.Function):
    """Spherical harmonics of the edge vectors (reference src/matten/nn/_nequip.py:167-176)."""

    @staticmethod
    def forward(ctx, vec, lmax, normalize):
        ctx.args = (lmax, normalize)
        ctx.save_for_backward(vec)
        return ops.edge_sh(vec.detach(), lmax, normalize)

    @staticmethod
    @_first_order
    @once_differentiable
    def backward(ctx, g):
        (vec,) = ctx.saved_tensors
        return ops.edge_sh_bwd(vec, g.contiguous(), *ctx.args), None, None


class EdgeVectorsFn(torch.autograd.Function):
    """Edge vectors and lengths from positions and cells (reference src/matten/nn/_nequip.py:214-268).  The position
    gradient is summed over the receiver CSR and the sender CSR of ``graph``, the cell gradient per graph over the
    sender CSR: fixed order, no atomics."""

    @staticmethod
    def forward(ctx, pos, cell, graph, shift, batch):
        vec, ln = ops.edge_vectors(pos.detach(), graph.edge_index, shift, None if cell is None else cell.detach(),
                                   batch, graph.flag)
        ctx.graph, ctx.shift, ctx.batch, ctx.N = graph, shift, batch, pos.shape[0]
        ctx.cell_shape = None if cell is None else cell.shape
        ctx.save_for_backward(vec)
        ctx.set_materialize_grads(False)
        return vec, ln

    @staticmethod
    @_first_order
    @once_differentiable
    def backward(ctx, gvec, glen):
        (vec,) = ctx.saved_tensors
        need_pos, need_cell = ctx.needs_input_grad[:2]
        need_cell = need_cell and ctx.cell_shape is not None
        if not (need_pos or need_cell) or (gvec is None and glen is None):
            return None, None, None, None, None
        graph = ctx.graph
        B = 1 if ctx.cell_shape is None else ctx.cell_shape.numel() // 9
        sptr, sperm = _sender_csr(graph, ctx.N)
        gptr = graph.graph_ptr(ctx.batch, B) if (need_cell and B > 1) else None
        gpos, gcell = ops.edge_vectors_bwd(vec, gvec, glen, ctx.shift, graph.rowptr, graph.perm, sptr, sperm, gptr,
                                           ctx.N, B, need_pos, need_cell)
        return gpos, (gcell.reshape(ctx.cell_shape) if need_cell else None), None, None, None


class VectorLengthsFn(torch.autograd.Function):
    """|v| of precomputed edge vectors; backward d|v|/dv = v / |v| (0 at v = 0, as torch.linalg.norm)."""

    @staticmethod
    def forward(ctx, vec):
        from .functional import vector_lengths

        ctx.save_for_backward(vec)
        return vector_lengths(vec.detach())

    @staticmethod
    @_first_order
    @once_differentiable
    def backward(ctx, g):
        (vec,) = ctx.saved_tensors
        E = vec.shape[0]
        # the edge-vector backward on a graph in which every edge is its own receiver and nothing is sent:
        # grad_pos[e] = dv[e] = g[e] v[e] / |v[e]|
        ar = torch.arange(E + 1, dtype=torch.int32, device=vec.device)
        none_sent = torch.zeros(E + 1, dtype=torch.int32, device=vec.device)
        gv, _ = ops.edge_vectors_bwd(vec, None, g.contiguous(), None, ar, ar[:E], none_sent, ar[:E], None, E, 1,
                                     True, False)
        return gv


class InstanceNormFn(torch.autograd.Function):
    """Graph InstanceNorm (reference src/matten/nn/utils.py:448-588); the per-graph partial parameter gradients
    are summed over graphs by the fixed-order column reduction."""

    @staticmethod
    def forward(ctx, x, weight, bias, graph_ptr, mod):
        w = None if weight is None else weight.detach()
        b = None if bias is None else bias.detach()
        y, saved = ops.instance_norm_fwd(x.detach(), graph_ptr, mod.tables(), w, b, mod.eps, mod.reduce,
                                         mod.normalization)
        ctx.mod, ctx.graph_ptr, ctx.has_w = mod, graph_ptr, w is not None
        ctx.save_for_backward(x, w if w is not None else x.new_empty(0), *saved)
        return y

    @staticmethod
    def backward(ctx, g):
        x, w, mean, rstd, arg = ctx.saved_tensors
        mod = ctx.mod
        need_p = ctx.has_w and (ctx.needs_input_grad[1] or ctx.needs_input_grad[2])
        gx, gwp, gbp = ops.instance_norm_bwd(x.detach(), g.contiguous(), ctx.graph_ptr, mod.tables(),
                                             w if ctx.has_w else None, (mean, rstd, arg), mod.reduce,
                                             mod.normalization, need_p)
        gw = gb = None
        if need_p:
            gw = ops.col_reduce(gwp)
            gb = ops.col_reduce(gbp).index_select(0, mod.scalar_channels)
        return gx, gw, gb, None, None


class NormActFn(torch.autograd.Function):
    """e3nn NormActivation (reference src/matten/nn/utils.py:142-150)."""

    @staticmethod
    def forward(ctx, x, tables, act_id, epsilon):
        ctx.tables, ctx.act_id, ctx.epsilon = tables, act_id, epsilon
        ctx.save_for_backward(x)
        return ops.norm_act(x.detach(), tables, act_id, epsilon)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return ops.norm_act_bwd(x.detach(), g.contiguous(), ctx.tables, ctx.act_id, ctx.epsilon), None, None, None


class _SpeciesEmbedFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, lin_w, lin_b, Z, idx, lut, zmin, zmax, S, flag):
        species_index, attrs, feats = ops.species_embed(Z, idx, lut, zmin, zmax, S, lin_w.detach(), lin_b.detach(), flag)
        ctx.S = S
        ctx.save_for_backward(species_index)
        ctx.mark_non_differentiable(species_index, attrs)
        return species_index, attrs, feats

    @staticmethod
    def backward(ctx, _gi, _ga, g):
        (species_index,) = ctx.saved_tensors
        sptr, sperm = ops.csr_by_key(species_index, ctx.S, True, None)
        # dW[:, s] = sum of the gradient rows of the nodes of species s (fixed order); tiny [S, dim] result
        gws = ops.segment_sum_gather(g.contiguous(), sperm, sptr, species_index.shape[0])
        return gws.t().contiguous(), gws.sum(0), None, None, None, None, None, None, None


def species_embed(Z, idx, lut, zmin, zmax, S, lin_w, lin_b, flag):
    return _SpeciesEmbedFn.apply(lin_w, lin_b, Z, idx, lut, zmin, zmax, S, flag)


class _BatchNormTrainFn(torch.autograd.Function):
    """Training-mode e3nn BatchNorm (reference nn/utils.py:418): batch statistics over all nodes; only 0e channels are
    centred.  Column reductions and the elementwise passes are kernels; the [D]-sized statistics algebra in between
    is parameter-sized plumbing."""

    @staticmethod
    def forward(ctx, x, weight, bias, mod):
        xd = x.detach()
        N, D = xd.shape
        feat, scal_mask, scal_idx = mod.feat_idx, mod.scal_mask, mod.scal_idx
        dt = xd.dtype
        colsum = ops.col_reduce(xd)
        shift = torch.where(scal_mask, colsum / N, torch.zeros_like(colsum)).contiguous()
        ssq = ops.col_reduce(xd, shift, xd, shift)
        chan = mod.channel_matrix(dt)  # [D, num_features] 0/1: column j belongs to channel feat[j]
        cnt = chan.sum(0) * N
        var = (ssq @ chan) / cnt
        rstd = (var + mod.eps).pow(-0.5)
        w = weight.detach().to(dt)
        a_col = (rstd * w)[feat].contiguous()
        if mod.num_scalar > 0:
            b_col = torch.where(scal_mask, bias.detach().to(dt)[scal_idx] - shift * a_col, torch.zeros_like(a_col))
        else:
            b_col = torch.zeros_like(a_col)
        y = ops.affine2(xd, a_col, None, None, b_col.contiguous())
        with torch.no_grad():
            m = mod.momentum
            if mod.num_scalar > 0:
                mean_s = shift.index_select(0, mod.scal_cols)
                mod.running_mean.mul_(1 - m).add_(m * mean_s.to(mod.running_mean.dtype))
            mod.running_var.mul_(1 - m).add_(m * var.to(mod.running_var.dtype))
        ctx.mod = mod
        ctx.save_for_backward(x, shift, rstd, cnt, w)
        return y

    @staticmethod
    def backward(ctx, g):
        x, shift, rstd, cnt, w = ctx.saved_tensors
        mod = ctx.mod
        feat, scal_mask = mod.feat_idx, mod.scal_mask
        xd, g = x.detach(), g.contiguous()
        N = xd.shape[0]
        s1 = ops.col_reduce(g)                       # sum_n g
        s2c = ops.col_reduce(g, None, xd, shift)     # sum_n g (x - shift)
        s2 = s2c @ mod.channel_matrix(s2c.dtype)
        gw = s2 * rstd
        gb = s1.index_select(0, mod.scal_cols) if mod.num_scalar > 0 else None
        a_col = (rstd * w)[feat]
        cb = -(a_col * (rstd * rstd * s2 / cnt)[feat])
        cc = -cb * shift - torch.where(scal_mask, a_col * s1 / N, torch.zeros_like(s1))
        gx = ops.affine2(g, a_col.contiguous(), xd, cb.contiguous(), cc.contiguous())
        return gx, gw, gb, None


def batchnorm_train(mod, x):
    lead = x.shape[:-1]
    y = _BatchNormTrainFn.apply(x.reshape(-1, x.shape[-1]), mod.weight, mod.bias, mod)
    return y.reshape(lead + (x.shape[-1],))


class MSELossFn(torch.autograd.Function):
    """torch.nn.functional.mse_loss(pred, target) (reference model/model.py:234-274, mean reduction)."""

    @staticmethod
    def forward(ctx, pred, target):
        loss, grad = ops.mse_loss(pred.detach().contiguous(), target.detach().contiguous(), 1.0, True)
        ctx.save_for_backward(grad)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        (grad,) = ctx.saved_tensors
        return grad * g, None


def mse_loss(pred, target):
    return MSELossFn.apply(pred, target)
