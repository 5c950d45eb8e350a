"""
Periodic neighbour list + PyG-style collate with numpy only.

Semantics of the reference's ``neighbor_list_and_relative_vec`` (src/matten/data/data.py:285-413,
which wraps ``ase.neighborlist.primitive_neighbor_list("ijS", self_interaction=True)`` and then
drops the true self edges): every ordered pair (i, j, S) with
``|pos[j] - pos[i] + S @ cell| < r_max`` except (i == j, S == 0); ``edge_index[0] = i`` (centre),
``edge_index[1] = j`` (neighbour); ``edge_cell_shift`` stored as float; ``num_neigh =
bincount(i)``.  ASE's order inside one centre is an artefact of its cell binning, so edges are
emitted in the canonical order (i, j, Sx, Sy, Sz); the model output does not depend on it up to
summation order.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence

import numpy as np
import torch


def neighbor_list(pos: np.ndarray, cell: np.ndarray, r_max: float, pbc=(True, True, True)):
    """Returns (edge_index [2,E] int64, shifts [E,3] float64, num_neigh [N] int64)."""
    pos = np.asarray(pos, dtype=np.float64)
    cell = np.asarray(cell, dtype=np.float64).reshape(3, 3)
    n = len(pos)
    pbc = (pbc,) * 3 if isinstance(pbc, bool) else tuple(pbc)
    vol = abs(np.linalg.det(cell))
    reps = []
    for k in range(3):
        if pbc[k] and vol > 0:
            a, b = cell[(k + 1) % 3], cell[(k + 2) % 3]
            height = vol / np.linalg.norm(np.cross(a, b))
            reps.append(int(np.ceil(r_max / height)))
        else:
            reps.append(0)
    # wrap-independent: images are enumerated relative to the given (possibly unwrapped) positions,
    # one extra shell covers atoms lying outside the cell
    frac_span = 0
    if vol > 0:
        frac = pos @ np.linalg.inv(cell)
        frac_span = int(np.ceil(frac.max() - frac.min())) if n else 0
    rng = [np.arange(-(r + (frac_span if pbc[k] else 0)), r + (frac_span if pbc[k] else 0) + 1)
           for k, r in enumerate(reps)]
    S = np.stack(np.meshgrid(*rng, indexing="ij"), -1).reshape(-1, 3)
    off = S @ cell  # [M,3]
    src, dst, shf = [], [], []
    # chunk over images to bound memory: [n, n] distances per image block
    d0 = pos[None, :, :] - pos[:, None, :]  # [i, j, 3] = pos[j] - pos[i]
    for m0 in range(0, len(S), 64):
        o = off[m0:m0 + 64]
        d = d0[None] + o[:, None, None, :]
        dist2 = (d * d).sum(-1)
        mask = dist2 < r_max * r_max
        mm, ii, jj = np.nonzero(mask)
        keep = ~((ii == jj) & np.all(S[m0 + mm] == 0, axis=1))
        src.append(ii[keep])
        dst.append(jj[keep])
        shf.append(S[m0 + mm[keep]])
    src = np.concatenate(src) if src else np.zeros(0, np.int64)
    dst = np.concatenate(dst) if dst else np.zeros(0, np.int64)
    shf = np.concatenate(shf) if shf else np.zeros((0, 3), np.int64)
    order = np.lexsort((shf[:, 2], shf[:, 1], shf[:, 0], dst, src))
    src, dst, shf = src[order], dst[order], shf[order]
    if len(src) == 0:
        raise ValueError("After eliminating self edges, no edges remain in this system.")
    edge_index = np.stack([src, dst]).astype(np.int64)
    num_neigh = np.bincount(src, minlength=n).astype(np.int64)
    return edge_index, shf.astype(np.float64), num_neigh


def make_graph(pos, cell, atomic_numbers, r_cut: float, dtype=torch.float32, extra: Optional[dict] = None):
    """One crystal -> dict of CPU tensors with the reference's dtypes (``Crystal.from_points``,
    src/matten/data/data.py:212-260: float shifts, float num_neigh, int64 indices)."""
    ei, sh, nn = neighbor_list(pos, cell, r_cut)
    g = {
        "pos": torch.as_tensor(np.asarray(pos), dtype=dtype),
        "edge_index": torch.as_tensor(ei, dtype=torch.int64),
        "edge_cell_shift": torch.as_tensor(sh, dtype=dtype),
        "cell": torch.as_tensor(np.asarray(cell), dtype=dtype).reshape(3, 3),
        "num_neigh": torch.as_tensor(nn, dtype=dtype),
        "atomic_numbers": torch.as_tensor(np.asarray(atomic_numbers), dtype=torch.int64),
    }
    if extra:
        g.update(extra)
    return g


def collate(graphs: Sequence[Dict[str, torch.Tensor]]) -> Dict[str, torch.Tensor]:
    """torch_geometric ``Batch.from_data_list`` for the keys the model reads: node tensors are
    concatenated, ``edge_index`` is offset by the node counts, ``cell`` is stacked along dim 0
    ([3B,3], viewed as [B,3,3] by with_edge_vectors), plus ``batch`` / ``ptr`` / ``num_graphs``."""
    out: Dict[str, torch.Tensor] = {}
    n_nodes = [int(g["pos"].shape[0]) for g in graphs]
    offs = np.concatenate([[0], np.cumsum(n_nodes)])
    node_keys = [k for k in graphs[0] if k not in ("edge_index", "edge_cell_shift", "cell")
                 and graphs[0][k].dim() >= 1 and graphs[0][k].shape[0] == n_nodes[0] and k != "y"]
    for k in node_keys:
        out[k] = torch.cat([g[k] for g in graphs], 0)
    out["edge_index"] = torch.cat([g["edge_index"] + int(o) for g, o in zip(graphs, offs[:-1])], 1)
    out["edge_cell_shift"] = torch.cat([g["edge_cell_shift"] for g in graphs], 0)
    out["cell"] = torch.cat([g["cell"].reshape(3, 3) for g in graphs], 0)
    out["batch"] = torch.cat([torch.full((n,), i, dtype=torch.int64) for i, n in enumerate(n_nodes)])
    out["ptr"] = torch.as_tensor(offs, dtype=torch.int64)
    out["num_graphs"] = len(graphs)
    for k in graphs[0]:
        if k not in out and k not in ("edge_index", "edge_cell_shift", "cell"):
            v = graphs[0][k]
            if isinstance(v, torch.Tensor):
                out[k] = torch.stack([g[k] for g in graphs], 0) if v.dim() == 0 or k == "y" else \
                    torch.cat([g[k] for g in graphs], 0)
    return out


def to_device(batch: Dict[str, torch.Tensor], device, non_blocking: bool = True) -> Dict[str, torch.Tensor]:
    return {k: (v.to(device, non_blocking=non_blocking) if isinstance(v, torch.Tensor) else v)
            for k, v in batch.items()}


def batch_from_structures(structs: Sequence[dict], r_cut: float, device, dtype=torch.float32) -> Dict[str, torch.Tensor]:
    """Batched graph dict built ON THE GPU: positions / cells / atomic numbers of all crystals are uploaded once and the
    periodic neighbour list of the whole batch comes from ``ops.neighbor_list`` (one kernel pair instead of one
    host-side numpy search per crystal).  ``structs``: dicts with ``cart`` [n,3], ``lattice`` [3,3], ``Z`` [n]
    (``matten_b200.predict._structure_arrays``).  Same keys, dtypes and edge order as ``collate(make_graph(...))``."""
    from .. import ops

    n_nodes = [len(s["Z"]) for s in structs]
    offs = np.concatenate([[0], np.cumsum(n_nodes)])
    pos = torch.as_tensor(np.concatenate([np.asarray(s["cart"], dtype=np.float64).reshape(-1, 3) for s in structs]))
    cell = torch.as_tensor(np.stack([np.asarray(s["lattice"], dtype=np.float64).reshape(3, 3) for s in structs]))
    out = {
        "pos": pos.to(device=device, dtype=dtype),
        "cell": cell.to(device=device, dtype=dtype).reshape(-1, 3),
        "atomic_numbers": torch.as_tensor(np.concatenate([np.asarray(s["Z"], dtype=np.int64) for s in structs])).to(device),
        "batch": torch.repeat_interleave(torch.arange(len(structs)), torch.as_tensor(n_nodes)).to(device),
        "ptr": torch.as_tensor(offs, dtype=torch.int64).to(device),
        "num_graphs": len(structs),
    }
    # the search itself runs in fp64 from the fp64 inputs (like the reference's numpy/ASE path), whatever `dtype` is
    ei, sh, nn = ops.neighbor_list(pos.to(device), cell.to(device), out["batch"], out["ptr"], r_cut,
                                   max_atoms=max(n_nodes, default=0))
    out["edge_index"] = ei
    out["edge_cell_shift"] = sh.to(dtype)
    out["num_neigh"] = nn.to(dtype)
    return out
