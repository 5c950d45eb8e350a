"""
Thin functional layer over the C ABI (include/matten_b200.h): torch tensors in, torch
tensors out.  torch is used for device memory and the current CUDA stream only; every
computation below is a hand-written sm_100a kernel in libmatten_b200.so.

No CPU path exists: CPU tensors raise, and on a GPU that is not sm_100 the library
returns MT_EARCH which is raised as RuntimeError.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import ConvPlanStruct, LinBlockStruct, MT_F32, MT_F64, check

def _on_device(fn):
    """Runs an op with the CUDA device of its first tensor argument current: the C ABI launches on the calling
    thread's current device (like every CUDA library), while the tensors and the stream passed down belong to the
    tensors' device -- a model on cuda:1 called while cuda:0 is current must not launch on cuda:0 (ADVICE r1)."""
    import functools

    def first_cuda(objs):
        for o in objs:
            if isinstance(o, torch.Tensor) and o.is_cuda:
                return o.device
            if isinstance(o, (list, tuple)):
                d = first_cuda(o)
                if d is not None:
                    return d
            if isinstance(o, ConvPlanHandle):
                return o.device
        return None

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        dev = first_cuda(args) or first_cuda(kwargs.values())
        if dev is None or dev.index is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)

    return wrapper


def launch_count() -> int:
    """Kernels launched by libmatten_b200.so in this process (exact, counted in the library)."""
    return int(_lib.load().mt_launch_count())


#: optional profiling hook: when set to a list, conv_fwd appends (tag, start_event, end_event)
CONV_EVENTS = None


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return MT_F32
    if t.dtype == torch.float64:
        return MT_F64
    raise TypeError(f"matten_b200 computes in float32 or float64, got {t.dtype}")


def _p(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(t: torch.Tensor):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _req(t: torch.Tensor, name: str, dtype=None):
    if not t.is_cuda:
        raise RuntimeError(f"matten_b200: `{name}` must be a CUDA tensor (there is no CPU fallback)")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"matten_b200: `{name}` must be {dtype}, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


def new_flag(device) -> torch.Tensor:
    return torch.zeros(1, dtype=torch.int32, device=device)


def raise_on_flag(flag: torch.Tensor):
    """Reads the device error word (one synchronising copy per batch)."""
    v = int(flag.item())
    if v == 0:
        return
    msgs = []
    if v & _lib.FLAG_BAD_SPECIES:
        msgs.append("Invalid atomic numbers: a species is not in the model's allowed_species")
    if v & _lib.FLAG_BAD_INDEX:
        msgs.append("index out of range in edge_index / batch")
    if v & _lib.FLAG_UNSORTED:
        msgs.append("`batch` must be sorted (nodes of a graph contiguous)")
    raise RuntimeError("; ".join(msgs))


# ------------------------------------------------------------------ edges --
@_on_device
def edge_vectors(pos, edge_index, edge_cell_shift=None, cell=None, batch=None, flag=None,
                 want_vec=True, want_len=True):
    lib = _lib.load()
    pos = _req(pos, "pos")
    edge_index = _req(edge_index, "edge_index", torch.int64)
    N, E = pos.shape[0], edge_index.shape[1]
    B = 0
    if cell is not None:
        cell = _req(cell, "cell", pos.dtype).view(-1, 3, 3)
        B = cell.shape[0]
        edge_cell_shift = _req(edge_cell_shift, "edge_cell_shift", pos.dtype)
        if B > 1:
            batch = _req(batch, "batch", torch.int64)
    vec = torch.empty((E, 3), dtype=pos.dtype, device=pos.device) if want_vec else None
    ln = torch.empty((E,), dtype=pos.dtype, device=pos.device) if want_len else None
    if E == 0:  # nothing to compute (and an empty shift tensor has no data pointer)
        return vec, ln
    check(lib.mt_edge_vectors(_dt(pos), _p(pos), _p(edge_index), _p(edge_cell_shift), _p(cell),
                              _p(batch) if B > 1 else None, N, E, B, _p(vec), _p(ln), _p(flag), _stream(pos)))
    return vec, ln


@_on_device
def edge_sh(edge_vec, lmax: int, normalize: bool = True):
    lib = _lib.load()
    edge_vec = _req(edge_vec, "edge_vectors")
    E = edge_vec.shape[0]
    out = torch.empty((E, (lmax + 1) ** 2), dtype=edge_vec.dtype, device=edge_vec.device)
    check(lib.mt_edge_sh(_dt(edge_vec), _p(edge_vec), E, lmax, int(normalize), _p(out), _stream(edge_vec)))
    return out


@_on_device
def edge_radial(edge_len, mode: int, num_basis: int, start: float, end: float, cutoff: bool = True,
                poly_p: float = 6.0, bessel_w=None):
    lib = _lib.load()
    edge_len = _req(edge_len, "edge_lengths")
    E = edge_len.shape[0]
    if bessel_w is not None:
        bessel_w = _req(bessel_w, "bessel_weights", edge_len.dtype)
    out = torch.empty((E, num_basis), dtype=edge_len.dtype, device=edge_len.device)
    check(lib.mt_edge_radial(_dt(edge_len), _p(edge_len), E, mode, num_basis, float(start), float(end),
                             int(cutoff), float(poly_p), _p(bessel_w), _p(out), _stream(edge_len)))
    return out


@_on_device
def edge_sh_bwd(edge_vec, grad_sh, lmax: int, normalize: bool = True):
    """grad_vec [E,3] = J_Y(edge_vec)^T grad_sh (backward of edge_sh)."""
    lib = _lib.load()
    edge_vec = _req(edge_vec, "edge_vectors")
    grad_sh = _req(grad_sh, "grad_sh", edge_vec.dtype)
    E = edge_vec.shape[0]
    out = torch.empty((E, 3), dtype=edge_vec.dtype, device=edge_vec.device)
    check(lib.mt_edge_sh_bwd(_dt(edge_vec), _p(edge_vec), _p(grad_sh), E, lmax, int(normalize), _p(out),
                             _stream(edge_vec)))
    return out


@_on_device
def edge_radial_bwd(edge_len, grad_emb, mode: int, num_basis: int, start: float, end: float, cutoff: bool = True,
                    poly_p: float = 6.0, bessel_w=None):
    """grad_len [E] = sum_k grad_emb[:, k] d edge_radial[:, k] / d edge_len (modes 0, 1 and 3-6)."""
    lib = _lib.load()
    edge_len = _req(edge_len, "edge_lengths")
    grad_emb = _req(grad_emb, "grad_emb", edge_len.dtype)
    E = edge_len.shape[0]
    if bessel_w is not None:
        bessel_w = _req(bessel_w, "bessel_weights", edge_len.dtype)
    out = torch.empty((E,), dtype=edge_len.dtype, device=edge_len.device)
    check(lib.mt_edge_radial_bwd(_dt(edge_len), _p(edge_len), _p(grad_emb), E, mode, num_basis, float(start),
                                 float(end), int(cutoff), float(poly_p), _p(bessel_w), _p(out), _stream(edge_len)))
    return out


@_on_device
def edge_vectors_bwd(edge_vec, grad_vec, grad_len, edge_cell_shift, rowptr, perm, sender_ptr, sender_perm,
                     graph_ptr, N: int, B: int, want_pos: bool = True, want_cell: bool = True):
    """(grad_pos [N,3] | None, grad_cell [B,3,3] | None): backward of edge_vectors, summed over the receiver CSR
    (rowptr, perm) and the sender CSR of the receiver-sorted list (sender_ptr, sender_perm); graph_ptr [B+1] int32
    may be None when B == 1."""
    lib = _lib.load()
    edge_vec = _req(edge_vec, "edge_vectors")
    dt = edge_vec.dtype
    E = edge_vec.shape[0]
    grad_vec = None if grad_vec is None else _req(grad_vec, "grad_vec", dt)
    grad_len = None if grad_len is None else _req(grad_len, "grad_len", dt)
    want_cell = want_cell and edge_cell_shift is not None
    if want_cell:
        edge_cell_shift = _req(edge_cell_shift, "edge_cell_shift", dt)
    if E == 0:
        return (edge_vec.new_zeros((N, 3)) if want_pos else None,
                edge_vec.new_zeros((B, 3, 3)) if want_cell else None)
    gpos = torch.empty((N, 3), dtype=dt, device=edge_vec.device) if want_pos else None
    gcell = torch.empty((B, 3, 3), dtype=dt, device=edge_vec.device) if want_cell else None
    nbytes = lib.mt_edge_vectors_bwd_workspace_bytes(_dt(edge_vec), E, B)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=edge_vec.device)
    check(lib.mt_edge_vectors_bwd(_dt(edge_vec), _p(edge_vec), _p(grad_vec), _p(grad_len),
                                  _p(edge_cell_shift) if want_cell else None, _p(rowptr), _p(perm), _p(sender_ptr),
                                  _p(sender_perm), _p(graph_ptr), N, E, B, _p(gpos), _p(gcell), _p(ws), nbytes,
                                  _stream(edge_vec)))
    return gpos, gcell


#: Crystals of at least this many atoms take the cell-list search (mt_neighbor_cells_*) under method="auto", smaller
#: ones the all-pairs search (mt_neighbor_count / mt_neighbor_fill).  profiles/neighbor_list_b200.jsonl, "crossover"
#: line (one NVIDIA B200, 1000 W): 64 atoms, the smallest size swept, where the cell search took 0.22 ms against 0.95
#: for one crystal and 0.28 against 0.97 for 64 of them.  Batches of smaller crystals, such as the 100 example
#: crystals (at most 48 atoms), stay on the pair kernels they used before.
NL_CELLS_MIN_ATOMS = 64


def neighbor_method(ptr, max_atoms: Optional[int] = None, method: str = "auto") -> str:
    """The search ``neighbor_list`` runs on a batch with node offsets ``ptr``: ``method`` unless it is "auto", else
    "cells" when the largest crystal (``max_atoms``, or read from ``ptr`` when not given) has at least
    NL_CELLS_MIN_ATOMS atoms, "pairs" otherwise."""
    if method not in ("auto", "pairs", "cells"):
        raise ValueError(f"neighbour-list method must be 'auto', 'pairs' or 'cells', got {method!r}")
    if method != "auto":
        return method
    if max_atoms is None:
        max_atoms = int((ptr[1:] - ptr[:-1]).max()) if ptr.numel() > 1 else 0
    return "cells" if max_atoms >= NL_CELLS_MIN_ATOMS else "pairs"


@_on_device
def neighbor_list(pos, cell, batch, ptr, r_max: float, max_atoms: Optional[int] = None, method: str = "auto"):
    """Periodic neighbour list of a batch of crystals on the GPU (reference data/data.py:285-413 semantics).
    pos [N,3], cell [B,3,3] (same float dtype), batch [N] int64, ptr [B+1] int64.
    Returns (edge_index [2,E] int64, edge_cell_shift [E,3], num_neigh [N]) in the canonical (i, j, S) order.
    ``method``: "pairs" (all pairs, quadratic per crystal), "cells" (cell list, linear) or "auto" (cells when the
    largest crystal has at least NL_CELLS_MIN_ATOMS atoms); both give the same outputs bit for bit.  ``max_atoms``
    (atoms of the largest crystal) spares "auto" a read of ``ptr`` from the device."""
    lib = _lib.load()
    pos = _req(pos, "pos")
    cell = _req(cell, "cell", pos.dtype).reshape(-1, 3, 3)
    ptr = _req(ptr, "ptr", torch.int64)
    N, B = pos.shape[0], cell.shape[0]
    cells = neighbor_method(ptr, max_atoms, method) == "cells"
    if B > 1:
        batch = _req(batch, "batch", torch.int64)
    workspace_bytes, count, fill = (
        (lib.mt_neighbor_cells_workspace_bytes, lib.mt_neighbor_cells_count, lib.mt_neighbor_cells_fill) if cells else
        (lib.mt_neighbor_workspace_bytes, lib.mt_neighbor_count, lib.mt_neighbor_fill))
    offsets = torch.empty(N + 1, dtype=torch.int32, device=pos.device)
    nbytes = workspace_bytes(N, B)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=pos.device)
    check(count(_dt(pos), _p(pos), _p(cell), _p(batch) if B > 1 else None, _p(ptr), N, B, float(r_max),
                _p(offsets), _p(ws), nbytes, _stream(pos)))
    E = int(offsets[-1].item())  # the one synchronisation of graph building: the edge count sizes the outputs
    ei = torch.empty((2, max(E, 0)), dtype=torch.int64, device=pos.device)
    shifts = torch.empty((max(E, 0), 3), dtype=pos.dtype, device=pos.device)
    num_neigh = torch.empty(N, dtype=pos.dtype, device=pos.device)
    check(fill(_dt(pos), _p(pos), _p(batch) if B > 1 else None, _p(ptr), N, B, float(r_max),
               _p(offsets), _p(ws), _p(ei), _p(shifts), _p(num_neigh), E, _stream(pos)))
    return ei, shifts, num_neigh


# ------------------------------------------------------------ bookkeeping --
@_on_device
def csr_by_key(keys, num_keys: int, want_perm: bool = True, flag=None):
    """Stable sort of int64 keys -> (rowptr int32 [num_keys+1], perm int32 [E] | None)."""
    lib = _lib.load()
    keys = _req(keys, "keys", torch.int64)
    E = keys.shape[0]
    rowptr = torch.empty(num_keys + 1, dtype=torch.int32, device=keys.device)
    perm = torch.empty(E, dtype=torch.int32, device=keys.device) if want_perm else None
    nbytes = lib.mt_csr_workspace_bytes(num_keys, E)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=keys.device)
    check(lib.mt_csr_by_key(_p(keys), E, num_keys, _p(rowptr), _p(perm), _p(ws), nbytes, _p(flag),
                            _stream(keys)))
    return rowptr, perm


@_on_device
def gather_i64_to_i32(src, perm=None):
    lib = _lib.load()
    src = _req(src, "src", torch.int64)
    n = perm.shape[0] if perm is not None else src.shape[0]
    out = torch.empty(n, dtype=torch.int32, device=src.device)
    check(lib.mt_gather_i64_to_i32(_p(src), _p(perm), n, _p(out), _stream(src)))
    return out


@_on_device
def check_sorted(keys, flag):
    lib = _lib.load()
    keys = _req(keys, "keys", torch.int64)
    check(lib.mt_check_sorted(_p(keys), keys.shape[0], _p(flag), _stream(keys)))


@_on_device
def species_embed(atomic_numbers, species_index, lut, min_z: int, max_z: int, num_species: int,
                  lin_w, lin_b, flag=None, want_attrs=True):
    """Returns (species_index int64 [N], node_attrs [N,S] | None, node_feats [N,dim])."""
    lib = _lib.load()
    lin_w = _req(lin_w, "linear.weight")
    lin_b = _req(lin_b, "linear.bias", lin_w.dtype)
    dev = lin_w.device
    z_given = atomic_numbers is not None
    if z_given:
        atomic_numbers = _req(atomic_numbers, "atomic_numbers", torch.int64)
        N = atomic_numbers.shape[0]
        lut = _req(lut, "_Z_to_index", torch.int64)
        species_index = torch.empty(N, dtype=torch.int64, device=dev)
    else:
        species_index = _req(species_index, "species_index", torch.int64)
        N = species_index.shape[0]
    dim = lin_w.shape[0]
    attrs = torch.empty((N, num_species), dtype=lin_w.dtype, device=dev) if want_attrs else None
    feats = torch.empty((N, dim), dtype=lin_w.dtype, device=dev)
    check(lib.mt_species_embed(_dt(lin_w), _p(atomic_numbers), int(z_given), _p(lut), int(min_z), int(max_z),
                               num_species, dim, _p(lin_w), _p(lin_b), N, _p(species_index), _p(attrs),
                               _p(feats), _p(flag), _stream(lin_w)))
    return species_index, attrs, feats


# ------------------------------------------------------------------- conv --
class ConvPlanHandle:
    """Device copy of a :class:`matten_b200.plan.UVUPlan` + the POD struct of the ABI."""

    def __init__(self, uvu_plan, mlp_sizes: Sequence[int], act_id: int, act_cst: float, device):
        self.plan = uvu_plan
        self.item_hdr = uvu_plan.item_hdr.to(device).contiguous()
        self.slot_tab = uvu_plan.slot_tab.to(device).contiguous()
        s = ConvPlanStruct()
        s.x_dim, s.y_dim, s.out_dim = uvu_plan.x_dim, uvu_plan.y_dim, uvu_plan.out_dim
        s.num_items = uvu_plan.num_items
        s.item_hdr = self.item_hdr.data_ptr()
        s.slot_tab = self.slot_tab.data_ptr()
        nl = len(mlp_sizes) - 1
        if not (1 <= nl <= _lib.MT_MAX_MLP_LAYERS):
            raise ValueError(f"radial MLP with {nl} layers is not supported")
        if mlp_sizes[-1] != uvu_plan.weight_numel:
            raise ValueError("last MLP size must equal the tensor product's weight_numel")
        s.mlp_num_layers = nl
        for i, v in enumerate(mlp_sizes):
            s.mlp_sizes[i] = int(v)
        s.mlp_act = int(act_id)
        s.mlp_act_cst = float(act_cst)
        s.tc_num_parts = 0
        tc = getattr(uvu_plan, "tc", None)
        self.tc_tables = []
        self.tc_y_lmax = None  # set when the plan has a tensor-core path (its layout can then be shared by layers)
        if tc is not None and tc.parts:
            s.tc_num_parts = len(tc.parts)
            s.tc_y_lmax = tc.y_lmax
            self.tc_y_lmax = int(tc.y_lmax)
            for i, part in enumerate(tc.parts):
                tabs = [t.to(device).contiguous() for t in (part.row_wcol, part.bi_hdr, part.bi_lane, part.q_list)]
                self.tc_tables.append(tabs)
                ps = s.tc_parts[i]
                ps.num_tiles, ps.a_rows, ps.num_bi = part.num_tiles, part.a_rows, len(part.bis)
                ps.x_lo, ps.x_cols, ps.lmax = part.x_lo, part.x_cols, part.lmax
                ps.cost = max(1, int(round(part.cost)))
                for q in range(4):
                    ps.q_count[q] = part.q_count[q]
                ps.row_wcol, ps.bi_hdr, ps.bi_lane, ps.q_list = [t.data_ptr() for t in tabs]
        self.bw_tables = [t.to(device).contiguous() for t in (uvu_plan.bw_item_hdr, uvu_plan.bw_lane_tab,
                                                               uvu_plan.bw_path_tab)]
        s.bw_num_items, s.bw_num_paths = uvu_plan.bw_num_items, uvu_plan.bw_num_paths
        s.bw_item_hdr, s.bw_lane_tab, s.bw_path_tab = [t.data_ptr() for t in self.bw_tables]
        self.struct = s
        # the tensor-core forward gathers sender rows with TMA: rows must be multiples of 16 bytes.  Layers whose
        # feature row is not (the lmax-4 layers: 214 / 246 floats) run on a zero-padded copy of x with a padded plan.
        self.x_pad = (-uvu_plan.x_dim) % 4 if s.tc_num_parts > 0 else 0
        self.struct_fwd = s
        if self.x_pad:
            s2 = ConvPlanStruct()
            C.memmove(C.byref(s2), C.byref(s), C.sizeof(ConvPlanStruct))
            s2.x_dim = uvu_plan.x_dim + self.x_pad
            self.struct_fwd = s2
        self.mlp_sizes = list(mlp_sizes)
        self.device = torch.device(device)


@_on_device
def conv_layout(sh, y_lmax: int, rowptr, perm, src_sorted, N: int):
    """The layer-invariant inputs of the fp32 tensor-core convolution (padded column order of the receiver-sorted
    edge list + pair-interleaved sh rows), prepared once per batch and passed to every ``conv_fwd`` of that batch."""
    lib = _lib.load()
    sh = _req(sh, "edge_attrs", torch.float32)
    E = sh.shape[0]
    if sh.shape[1] != (y_lmax + 1) ** 2:
        raise ValueError(f"conv_layout: edge_attrs has {sh.shape[1]} columns, expected {(y_lmax + 1) ** 2}")
    nbytes = lib.mt_conv_layout_bytes(int(y_lmax), N, E)
    if nbytes == 0:
        return None
    buf = torch.empty(nbytes, dtype=torch.uint8, device=sh.device)  # the caching allocator aligns to 512 bytes
    check(lib.mt_conv_layout_prepare(int(y_lmax), _p(sh), _p(rowptr), _p(perm), _p(src_sorted), N, E, _p(buf), nbytes,
                                     _stream(sh)))
    return buf


@_on_device
def conv_fwd(handle: ConvPlanHandle, x, sh, emb, mlp_weights: Sequence[torch.Tensor], rowptr, perm,
             src_sorted, avg_num_neighbors: Optional[float], num_neigh=None, layout=None):
    lib = _lib.load()
    x = _req(x, "node_features")
    sh = _req(sh, "edge_attrs", x.dtype)
    emb = _req(emb, "edge_embedding", x.dtype)
    N, E = x.shape[0], sh.shape[0]
    pl = handle.plan
    if x.shape[1] != pl.x_dim or sh.shape[1] != pl.y_dim or emb.shape[1] != handle.mlp_sizes[0]:
        raise ValueError(f"conv_fwd: shapes {tuple(x.shape)}, {tuple(sh.shape)}, {tuple(emb.shape)} do not match "
                         f"the plan ({pl.x_dim}, {pl.y_dim}, {handle.mlp_sizes[0]})")
    ws = [_req(w, f"weight_nn.layer{i}.weight", x.dtype) for i, w in enumerate(mlp_weights)]
    for i, w in enumerate(ws):
        if tuple(w.shape) != (handle.mlp_sizes[i], handle.mlp_sizes[i + 1]):
            raise ValueError(f"radial MLP layer {i} has shape {tuple(w.shape)}")
    wptrs = (C.c_void_p * len(ws))(*[w.data_ptr() for w in ws])
    if num_neigh is not None:
        num_neigh = _req(num_neigh, "num_neigh", x.dtype)
    out = torch.empty((N, pl.out_dim), dtype=x.dtype, device=x.device)
    st = handle.struct
    if handle.x_pad and x.dtype == torch.float32:
        x = torch.nn.functional.pad(x, (0, handle.x_pad))
        st = handle.struct_fwd
    ws_bytes = lib.mt_conv_fwd_workspace_bytes(C.byref(st), _dt(x), N, E)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device) if ws_bytes else None
    if CONV_EVENTS is not None:
        ev0 = torch.cuda.Event(enable_timing=True)
        ev1 = torch.cuda.Event(enable_timing=True)
        ev0.record()
    check(lib.mt_conv_fwd(C.byref(st), _dt(x), _p(x), _p(sh), _p(emb), wptrs, _p(rowptr), _p(perm),
                          _p(src_sorted), float(avg_num_neighbors) if avg_num_neighbors is not None else 0.0,
                          _p(num_neigh), _p(out), _p(ws), ws_bytes,
                          _p(layout) if x.dtype == torch.float32 else None, N, E, _stream(x)))
    if CONV_EVENTS is not None:
        ev1.record()
        CONV_EVENTS.append(((pl.x_dim, pl.y_dim, pl.out_dim, pl.weight_numel, N, E), ev0, ev1))
    return out


_IMPLS = {"auto": 0, "tc": 1, "fma": 2}


def conv_select_impl(name: str) -> str:
    """Selects the fp32 kernel of conv_fwd ('auto' | 'tc' | 'fma'); returns the previous selection."""
    old = _lib.load().mt_conv_select_impl(_IMPLS[name])
    return {v: k for k, v in _IMPLS.items()}[old]


def conv_bwd(handle: ConvPlanHandle, x, sh, emb, mlp_weights: Sequence[torch.Tensor], rowptr, perm, src_sorted,
             sender_ptr, sender_perm, avg_num_neighbors: Optional[float], num_neigh, grad_out,
             need_x: bool = True, need_w: bool = True):
    """Returns (grad_x | None, [grad of every MLP weight] | None)."""
    gx, gws, _, _ = conv_bwd_full(handle, x, sh, emb, mlp_weights, rowptr, perm, src_sorted, sender_ptr, sender_perm,
                                  avg_num_neighbors, num_neigh, grad_out, need_x, need_w)
    return gx, gws


@_on_device
def conv_bwd_full(handle: ConvPlanHandle, x, sh, emb, mlp_weights: Sequence[torch.Tensor], rowptr, perm, src_sorted,
                  sender_ptr, sender_perm, avg_num_neighbors: Optional[float], num_neigh, grad_out,
                  need_x: bool = True, need_w: bool = True, need_sh: bool = False, need_emb: bool = False):
    """Returns (grad_x | None, [grad of every MLP weight] | None, grad_sh | None, grad_emb | None); the edge
    gradients are in the caller's edge order."""
    lib = _lib.load()
    x = _req(x, "node_features")
    sh = _req(sh, "edge_attrs", x.dtype)
    emb = _req(emb, "edge_embedding", x.dtype)
    grad_out = _req(grad_out, "grad_out", x.dtype)
    N, E = x.shape[0], sh.shape[0]
    ws = [_req(w, f"weight_nn.layer{i}.weight", x.dtype) for i, w in enumerate(mlp_weights)]
    wptrs = (C.c_void_p * len(ws))(*[w.data_ptr() for w in ws])
    gx = torch.empty_like(x) if need_x else None
    gws = [torch.empty_like(w) for w in ws] if need_w else None
    gwptrs = (C.c_void_p * len(ws))(*[g.data_ptr() for g in gws]) if need_w else None
    gsh = torch.empty_like(sh) if need_sh else None
    gemb = torch.empty_like(emb) if need_emb else None
    if num_neigh is not None:
        num_neigh = _req(num_neigh, "num_neigh", x.dtype)
    nbytes = lib.mt_conv_bwd_workspace_bytes(C.byref(handle.struct), _dt(x), N, E)
    wsb = torch.empty(nbytes, dtype=torch.uint8, device=x.device) if nbytes else None
    check(lib.mt_conv_bwd_full(C.byref(handle.struct), _dt(x), _p(x), _p(sh), _p(emb), wptrs, _p(rowptr), _p(perm),
                               _p(src_sorted), _p(sender_ptr), _p(sender_perm),
                               float(avg_num_neighbors) if avg_num_neighbors is not None else 0.0, _p(num_neigh),
                               _p(grad_out), _p(gx), gwptrs, _p(gsh), _p(gemb), _p(wsb), nbytes, N, E, _stream(x)))
    return gx, gws, gsh, gemb


# ----------------------------------------------------------------- linear --
class LinPlanHandle:
    def __init__(self, blocks, in_dim: int, out_dim: int, num_species: int, weight_numel: int):
        self.blocks = blocks
        arr = (LinBlockStruct * len(blocks))()
        for i, b in enumerate(blocks):
            arr[i].in_off, arr[i].out_off = b.in_off, b.out_off
            arr[i].mul_in, arr[i].mul_out, arr[i].dim = b.mul_in, b.mul_out, b.dim
            arr[i].w_off, arr[i].scale = b.w_off, b.scale
        self.arr = arr
        self.n = len(blocks)
        self.in_dim, self.out_dim, self.S, self.weight_numel = in_dim, out_dim, num_species, weight_numel


@_on_device
def linear_fwd(h: LinPlanHandle, x, weight, species_perm=None, species_ptr=None, out=None,
               accumulate: bool = False):
    lib = _lib.load()
    x = _req(x, "x")
    lead = x.shape[:-1]
    x2 = x.reshape(-1, x.shape[-1])
    if x2.shape[1] != h.in_dim:
        raise ValueError(f"linear_fwd: input has {x2.shape[1]} features, plan expects {h.in_dim}")
    weight = _req(weight, "weight", x.dtype)
    if weight.numel() != h.weight_numel:
        raise ValueError(f"linear_fwd: weight has {weight.numel()} elements, plan expects {h.weight_numel}")
    N = x2.shape[0]
    if out is None:
        if accumulate:
            raise ValueError("accumulate needs an output tensor")
        out = torch.empty((N, h.out_dim), dtype=x.dtype, device=x.device)
    check(lib.mt_linear_fwd(_dt(x), h.arr, h.n, h.in_dim, h.out_dim, h.S, _p(x2), _p(weight), _p(species_perm),
                            _p(species_ptr), int(accumulate), _p(out), N, _stream(x)))
    return out.reshape(lead + (h.out_dim,))


@_on_device
def linear_bwd(h: LinPlanHandle, x, weight, grad_out, species_perm=None, species_ptr=None, need_x=True,
               need_w=True):
    """Returns (grad_x | None, grad_weight (flat) | None)."""
    lib = _lib.load()
    x = _req(x, "x")
    x2 = x.reshape(-1, x.shape[-1])
    g2 = _req(grad_out, "grad_out", x.dtype).reshape(-1, h.out_dim)
    weight = _req(weight, "weight", x.dtype)
    N = x2.shape[0]
    gx = torch.empty_like(x2) if need_x else None
    gw = torch.empty(h.weight_numel, dtype=x.dtype, device=x.device) if need_w else None
    nbytes = lib.mt_linear_bwd_workspace_bytes(_dt(x), h.weight_numel) if need_w else 0
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device) if nbytes else None
    check(lib.mt_linear_bwd(_dt(x), h.arr, h.n, h.in_dim, h.out_dim, h.S, h.weight_numel, _p(x2), _p(weight), _p(g2),
                            _p(species_perm), _p(species_ptr), _p(gx), 0, _p(gw), 0, _p(ws), nbytes, N, _stream(x)))
    return (gx.reshape(x.shape) if need_x else None), gw


# ------------------------------------------------------------------- gate --
@_on_device
def gate_bwd(x, grad_out, in_dim, out_dim, src_idx, gate_idx, act_id, act_cst, inv_first, inv_count, affine_a=None):
    lib = _lib.load()
    x = _req(x, "x")
    grad_out = _req(grad_out, "grad_out", x.dtype)
    N = x.numel() // in_dim
    gx = torch.empty_like(x)
    check(lib.mt_gate_bwd(_dt(x), _p(x), _p(grad_out), in_dim, out_dim, _p(src_idx), _p(gate_idx), _p(act_id),
                          _p(act_cst), _p(affine_a), _p(inv_first), _p(inv_count), _p(gx), N, _stream(x)))
    return gx


@_on_device
def col_reduce(a, shift_a=None, b=None, shift_b=None):
    """out[j] = sum_n (a[n,j] - shift_a[j]) * (b[n,j] - shift_b[j])  (b None: plain column sum)."""
    lib = _lib.load()
    a = _req(a, "a")
    a2 = a.reshape(-1, a.shape[-1])
    N, dim = a2.shape
    if b is not None:
        b = _req(b, "b", a.dtype).reshape(-1, dim)
    out = torch.empty(dim, dtype=a.dtype, device=a.device)
    nbytes = lib.mt_col_reduce_workspace_bytes(_dt(a), dim)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=a.device)
    check(lib.mt_col_reduce(_dt(a), _p(a2), _p(shift_a), _p(b), _p(shift_b), N, dim, _p(out), _p(ws), nbytes,
                            _stream(a)))
    return out


@_on_device
def affine2(a, ca, b=None, cb=None, cc=None):
    """ca[j]*a[n,j] + cb[j]*b[n,j] + cc[j]"""
    lib = _lib.load()
    a = _req(a, "a")
    dim = a.shape[-1]
    N = a.numel() // dim
    if b is not None:
        b = _req(b, "b", a.dtype)
    out = torch.empty_like(a)
    check(lib.mt_affine2(_dt(a), _p(a), _p(ca), _p(b), _p(cb), _p(cc), _p(out), N, dim, _stream(a)))
    return out


@_on_device
def gate_fwd(x, in_dim: int, out_dim: int, src_idx, gate_idx, act_id, act_cst, affine_a=None, affine_b=None):
    lib = _lib.load()
    x = _req(x, "x")
    if x.shape[-1] != in_dim:
        raise ValueError(f"gate_fwd: input has {x.shape[-1]} features, expected {in_dim}")
    lead = x.shape[:-1]
    N = x.numel() // in_dim
    out = torch.empty(lead + (out_dim,), dtype=x.dtype, device=x.device)
    check(lib.mt_gate_fwd(_dt(x), _p(x), in_dim, out_dim, _p(src_idx), _p(gate_idx), _p(act_id), _p(act_cst),
                          _p(affine_a), _p(affine_b), _p(out), N, _stream(x)))
    return out


# ------------------------------------------------------------------- pool --
_MODES = {"sum": 0, "add": 0, "mean": 1, "min": 2, "max": 3}


@_on_device
def segment_reduce(x, ptr, reduce: str = "sum"):
    lib = _lib.load()
    x = _req(x, "x")
    B = ptr.shape[0] - 1
    dim = x.shape[1]
    out = torch.empty((B, dim), dtype=x.dtype, device=x.device)
    check(lib.mt_segment_reduce(_dt(x), _p(x), _p(ptr), dim, B, _MODES[reduce], _p(out), _stream(x)))
    return out


@_on_device
def segment_reduce_bwd(grad_out, ptr, N: int, reduce: str):
    lib = _lib.load()
    grad_out = _req(grad_out, "grad_out")
    B, dim = grad_out.shape
    if _MODES[reduce] > 1:
        raise ValueError("min/max pooling backward needs the forward input: use segment_extreme_bwd")
    gx = torch.empty((N, dim), dtype=grad_out.dtype, device=grad_out.device)
    check(lib.mt_segment_reduce_bwd(_dt(grad_out), _p(grad_out), _p(ptr), dim, B, N, _MODES[reduce], _p(gx),
                                    _stream(grad_out)))
    return gx


@_on_device
def segment_extreme_bwd(x, grad_out, ptr, reduce: str):
    """Backward of min/max pooling: the gradient goes to the first row holding the extreme value."""
    lib = _lib.load()
    x = _req(x, "x")
    grad_out = _req(grad_out, "grad_out", x.dtype)
    B, dim = grad_out.shape
    if _MODES[reduce] < 2:
        raise ValueError("segment_extreme_bwd handles min and max")
    gx = torch.zeros_like(x)  # rows outside ptr's span (none for a batch vector) keep 0
    check(lib.mt_segment_extreme_bwd(_dt(x), _p(x), _p(grad_out), _p(ptr), dim, B, _MODES[reduce], _p(gx),
                                     _stream(x)))
    return gx


# -------------------------------------------------------- normalisation (f4) --
_IN_REDUCE = {"mean": 0, "max": 1}
_IN_NORMALIZATION = {"component": 0, "norm": 1}


@_on_device
def instance_norm_fwd(x, graph_ptr, tables, weight, bias, eps: float, reduce: str, normalization: str):
    """Graph InstanceNorm forward; ``tables`` = (chan_first, chan_dim, chan_scalar) int32 [num_channels].
    Returns (out, (mean, rstd, arg)) with the saved per-(graph, channel) statistics."""
    lib = _lib.load()
    x = _req(x, "x")
    first, cdim, scal = tables
    N, dim = x.shape
    G, nf = graph_ptr.shape[0] - 1, first.shape[0]
    out = torch.empty_like(x)
    mean = torch.empty((G, nf), dtype=torch.float64, device=x.device)
    rstd = torch.empty_like(mean)
    arg = torch.empty((G, nf), dtype=torch.int32, device=x.device)
    weight = None if weight is None else _req(weight, "weight", x.dtype)
    bias = None if bias is None else _req(bias, "bias", x.dtype)
    check(lib.mt_instance_norm_fwd(_dt(x), _p(x), _p(graph_ptr), G, dim, nf, _p(first), _p(cdim), _p(scal),
                                   _p(weight), _p(bias), float(eps), _IN_REDUCE[reduce],
                                   _IN_NORMALIZATION[normalization], _p(out), _p(mean), _p(rstd), _p(arg),
                                   _stream(x)))
    return out, (mean, rstd, arg)


@_on_device
def instance_norm_bwd(x, grad_out, graph_ptr, tables, weight, saved, reduce: str, normalization: str,
                      need_params: bool = True):
    """Returns (grad_x, grad_weight_part [G,nf] | None, grad_bias_part [G,nf] | None)."""
    lib = _lib.load()
    x = _req(x, "x")
    grad_out = _req(grad_out, "grad_out", x.dtype)
    first, cdim, scal = tables
    mean, rstd, arg = saved
    N, dim = x.shape
    G, nf = graph_ptr.shape[0] - 1, first.shape[0]
    gx = torch.empty_like(x)
    gw = torch.empty((G, nf), dtype=x.dtype, device=x.device) if need_params else None
    gb = torch.empty((G, nf), dtype=x.dtype, device=x.device) if need_params else None
    weight = None if weight is None else _req(weight, "weight", x.dtype)
    check(lib.mt_instance_norm_bwd(_dt(x), _p(x), _p(grad_out), _p(graph_ptr), G, dim, nf, _p(first), _p(cdim),
                                   _p(scal), _p(weight), _IN_REDUCE[reduce], _IN_NORMALIZATION[normalization],
                                   _p(mean), _p(rstd), _p(arg), _p(gx), _p(gw), _p(gb), _stream(x)))
    return gx, gw, gb


@_on_device
def norm_act(x, tables, act_id: int, epsilon: float = 1e-8):
    lib = _lib.load()
    x = _req(x, "x")
    first, cdim = tables
    dim = x.shape[-1]
    N = x.numel() // dim
    out = torch.empty_like(x)
    check(lib.mt_norm_act_fwd(_dt(x), _p(x), dim, first.shape[0], _p(first), _p(cdim), int(act_id), float(epsilon),
                              _p(out), N, _stream(x)))
    return out


@_on_device
def norm_act_bwd(x, grad_out, tables, act_id: int, epsilon: float = 1e-8):
    lib = _lib.load()
    x = _req(x, "x")
    grad_out = _req(grad_out, "grad_out", x.dtype)
    first, cdim = tables
    dim = x.shape[-1]
    N = x.numel() // dim
    gx = torch.empty_like(x)
    check(lib.mt_norm_act_bwd(_dt(x), _p(x), _p(grad_out), dim, first.shape[0], _p(first), _p(cdim), int(act_id),
                              float(epsilon), _p(gx), N, _stream(x)))
    return gx


@_on_device
def normalize(data, mean, norm, scale: float = 1.0, inverse: bool = False):
    """(data - mean) / (norm * scale), or its inverse data * (norm * scale) + mean."""
    lib = _lib.load()
    data = _req(data, "data")
    mean = _req(mean, "mean", data.dtype)
    norm = _req(norm, "norm", data.dtype)
    dim = data.shape[-1]
    if mean.numel() != dim or norm.numel() != dim:
        raise ValueError(f"mean/norm must have {dim} entries, got {mean.numel()} and {norm.numel()}")
    N = data.numel() // dim
    out = torch.empty_like(data)
    check(lib.mt_normalize(_dt(data), _p(data), _p(mean), _p(norm), float(scale), int(bool(inverse)), _p(out), N, dim,
                           _stream(data)))
    return out


@_on_device
def segment_sum_gather(x, perm, ptr, num_rows: Optional[int] = None):
    """out[s] = sum of the rows x[perm[i]] for i in [ptr[s], ptr[s+1]) in that order."""
    lib = _lib.load()
    x = _req(x, "x")
    S = ptr.shape[0] - 1
    dim = x.shape[1]
    if num_rows is None:
        num_rows = perm.shape[0] if perm is not None else x.shape[0]
    out = torch.empty((S, dim), dtype=x.dtype, device=x.device)
    check(lib.mt_segment_sum_gather(_dt(x), _p(x), _p(perm), _p(ptr), dim, S, num_rows, _p(out), _stream(x)))
    return out


# ------------------------------------------------------- loss / optimiser --
@_on_device
def mse_loss(pred, target, grad_scale: float = 1.0, want_grad: bool = True):
    """(loss [1], d loss / d pred * grad_scale | None) -- torch.nn.functional.mse_loss(reduction='mean')."""
    lib = _lib.load()
    pred = _req(pred, "pred")
    target = _req(target, "target", pred.dtype)
    if pred.shape != target.shape:
        raise ValueError(f"mse_loss: shapes {tuple(pred.shape)} and {tuple(target.shape)} differ")
    loss = torch.empty(1, dtype=pred.dtype, device=pred.device)
    grad = torch.empty_like(pred) if want_grad else None
    check(lib.mt_mse_loss(_dt(pred), _p(pred), _p(target), pred.numel(), float(grad_scale), _p(loss), _p(grad),
                          _stream(pred)))
    return loss, grad


@_on_device
def adam_step(p, g, m, v, step: int, lr: float, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0,
              grad_scale: float = 1.0):
    """In-place torch.optim.Adam update of the flat buffers p, m, v from the flat gradient g."""
    lib = _lib.load()
    for name, t in (("p", p), ("g", g), ("m", m), ("v", v)):
        if not t.is_cuda or not t.is_contiguous() or t.dtype != p.dtype or t.numel() != p.numel():
            raise ValueError(f"adam_step: `{name}` must be a contiguous CUDA tensor matching the parameters")
    check(lib.mt_adam_step(_dt(p), _p(p), _p(g), _p(m), _p(v), p.numel(), float(lr), float(beta1), float(beta2),
                           float(eps), float(weight_decay), float(grad_scale), int(step), _stream(p)))
