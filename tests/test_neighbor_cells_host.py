"""Host side of the neighbour-search selection: the "auto" rule and the crystal sizes graph building passes down."""
import numpy as np
import pytest
import torch


def test_auto_rule_from_max_atoms_or_ptr():
    from matten_b200 import ops

    n = ops.NL_CELLS_MIN_ATOMS
    ptr = torch.tensor([0, 3, 3, 3 + n - 1])
    assert ops.neighbor_method(ptr) == "pairs"
    assert ops.neighbor_method(torch.tensor([0, 3, 3 + n, 3 + n + 1])) == "cells"
    # a given max_atoms is trusted: ptr is not read
    assert ops.neighbor_method(ptr, max_atoms=n) == "cells"
    assert ops.neighbor_method(ptr, max_atoms=n - 1) == "pairs"
    assert ops.neighbor_method(torch.tensor([0])) == "pairs"  # no crystal
    for m in ("pairs", "cells"):
        assert ops.neighbor_method(ptr, max_atoms=10 ** 6, method=m) == m
        assert ops.neighbor_method(ptr, max_atoms=0, method=m) == m
    with pytest.raises(ValueError, match="method"):
        ops.neighbor_method(ptr, method="ase")


def test_batch_from_structures_passes_the_largest_crystal(monkeypatch):
    from matten_b200 import ops
    from matten_b200.data.neighbors import batch_from_structures

    seen = {}

    def fake(pos, cell, batch, ptr, r_max, max_atoms=None, method="auto"):
        seen.update(max_atoms=max_atoms, method=method, ptr=ptr.tolist())
        n = pos.shape[0]
        return torch.zeros((2, 0), dtype=torch.int64), torch.zeros((0, 3), dtype=pos.dtype), torch.zeros(n, dtype=pos.dtype)

    monkeypatch.setattr(ops, "neighbor_list", fake)
    structs = [{"cart": np.zeros((k, 3)), "lattice": np.eye(3) * 4, "Z": [14] * k} for k in (3, 7, 1)]
    batch_from_structures(structs, 5.0, "cpu", torch.float64)
    assert seen == {"max_atoms": 7, "method": "auto", "ptr": [0, 3, 10, 11]}
