"""Cell-list neighbour search (mt_neighbor_cells_*) against the all-pairs search (mt_neighbor_count / _fill) and the
numpy twin: the same edge_index, edge_cell_shift and num_neigh, bit for bit, in the canonical (i, j, S) order."""
import json
import os

import numpy as np
import pytest
import torch

from tests.helpers import GOLDEN, HP_LMAX2, HP_LMAX4, build_pair

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
R_CUT = 5.0


def _batch(crystals, dtype=torch.float64):
    """[(pos [n,3], cell [3,3]), ...] -> (pos, cell, batch, ptr) on the GPU."""
    n = [len(p) for p, _ in crystals]
    pos = torch.as_tensor(np.concatenate([np.asarray(p, np.float64).reshape(-1, 3) for p, _ in crystals]), dtype=dtype)
    cell = torch.as_tensor(np.stack([np.asarray(c, np.float64).reshape(3, 3) for _, c in crystals]), dtype=dtype)
    batch = torch.repeat_interleave(torch.arange(len(crystals)), torch.as_tensor(n))
    ptr = torch.as_tensor(np.concatenate([[0], np.cumsum(n)]), dtype=torch.int64)
    return pos.to(DEV), cell.to(DEV), batch.to(DEV), ptr.to(DEV)


def _search(crystals, dtype=torch.float64, r=R_CUT):
    """Both searches on one batch; asserts they agree and returns the cell search's (edge_index, shifts, num_neigh)."""
    from matten_b200 import ops

    args = _batch(crystals, dtype)
    want = ops.neighbor_list(*args, r, method="pairs")
    got = ops.neighbor_list(*args, r, method="cells")
    for g, w, name in zip(got, want, ("edge_index", "edge_cell_shift", "num_neigh")):
        assert g.dtype == w.dtype and torch.equal(g, w), name
    return got


def _host(crystals, r=R_CUT):
    """The numpy twin on each crystal, collated."""
    from matten_b200.data.neighbors import neighbor_list

    eis, shs, nns, off = [], [], [], 0
    for p, c in crystals:
        if len(p):
            try:
                ei, sh, nn = neighbor_list(np.asarray(p, np.float64), np.asarray(c, np.float64), r)
            except ValueError:  # no edges at all
                ei, sh, nn = np.zeros((2, 0), np.int64), np.zeros((0, 3)), np.zeros(len(p), np.int64)
            eis.append(ei + off)
            shs.append(sh)
            nns.append(nn)
        off += len(p)
    return np.concatenate(eis, 1), np.concatenate(shs), np.concatenate(nns)


def _assert_host(got, crystals, r=R_CUT):
    ei, sh, nn = _host(crystals, r)
    assert np.array_equal(got[0].cpu().numpy(), ei)
    assert np.array_equal(got[1].double().cpu().numpy(), sh)
    assert np.array_equal(got[2].double().cpu().numpy(), nn.astype(np.float64))


def _diamond(rep, jitter=0.05, seed=0):
    from matten_b200.data.synthetic import diamond_supercell

    pos, cell = diamond_supercell(rep)
    return pos + np.random.default_rng(seed).normal(0.0, jitter, pos.shape), cell


def test_example_crystals_on_the_cell_search():
    """The 100 example crystals (triclinic cells of 1..20 atoms, up to 5 images per axis), forced to the cell search."""
    with open(os.path.join(GOLDEN, "n100_structures.json")) as f:
        structs = json.load(f)["structures"]
    crystals = [(np.array(s["cart_coords"]), np.array(s["lattice"])) for s in structs]
    got = _search(crystals)
    assert got[0].shape[1] == 14380  # BASELINE.md
    _assert_host(got, crystals)


def test_synthetic_batch():
    from matten_b200.data.synthetic import synthetic_batch

    sb = synthetic_batch(3, dtype=torch.float64)
    crystals = [(sb["pos"][sb["batch"] == b].numpy(), sb["cell"].reshape(-1, 3, 3)[b].numpy()) for b in range(3)]
    ei, sh, nn = _search(crystals)
    assert torch.equal(ei.cpu(), sb["edge_index"]) and torch.equal(sh.cpu(), sb["edge_cell_shift"])
    assert torch.equal(nn.cpu(), sb["num_neigh"])


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("rep", [8, 14])
def test_jittered_diamond_supercells(rep, dtype):
    """4 096 and 21 952 atoms."""
    crystals = [_diamond(rep, seed=rep)]
    ei, _, nn = _search(crystals, dtype)
    assert ei.shape[1] == 28 * 8 * rep ** 3 and float(nn.min()) == 28.0 == float(nn.max())


def test_sheared_triclinic_supercell():
    rng = np.random.default_rng(1)
    cell = np.array([[30.0, 0.0, 0.0], [27.0, 9.0, 0.0], [-24.0, 6.5, 8.0]])  # angles far from 90 degrees
    frac = rng.random((3000, 3))
    got = _search([(frac @ cell, cell)])
    assert got[0].shape[1] > 0


def test_unwrapped_positions_and_atoms_on_faces():
    rng = np.random.default_rng(2)
    pos, cell = _diamond(3, seed=2)
    frac = pos @ np.linalg.inv(cell)
    frac[:20] += rng.integers(-3, 4, (20, 3))          # whole lattice vectors
    frac[20:40] += rng.random((20, 3)) * 2.0 - 1.0     # fractional ones: atoms outside the cell
    frac[40:50, 0] = 0.0                               # exactly on faces
    frac[50:60, 1] = 1.0
    frac[60:64] = [[0.0, 0.0, 0.0], [1.0, 1.0, 1.0], [1.0, 0.0, 1.0], [0.0, 1.0, 0.5]]
    tric = np.array([[6.0, 0.0, 0.0], [2.5, 5.5, 0.0], [1.0, -2.0, 7.0]])
    f2 = rng.random((40, 3)) * 4.0 - 1.5               # a small triclinic cell with atoms up to 2.5 cells out
    crystals = [(frac @ cell, cell), (f2 @ tric, tric)]
    _assert_host(_search(crystals), crystals)


def test_thin_cells_beside_a_large_crystal():
    """Cells thinner than r_cut (many images per axis) in the batch of a 4 096-atom crystal."""
    rng = np.random.default_rng(3)
    thin = [
        (np.zeros((1, 3)), np.eye(3) * 2.0),
        (rng.random((2, 3)) @ np.diag([1.5, 3.0, 7.0]), np.diag([1.5, 3.0, 7.0])),
        (np.array([[0.1, 0.2, 0.3], [1.0, 0.4, 0.2]]), np.array([[2.2, 0.0, 0.0], [1.9, 1.2, 0.0], [0.3, 0.4, 0.9]])),
        (rng.random((5, 3)) @ np.diag([0.8, 12.0, 12.0]), np.diag([0.8, 12.0, 12.0])),
    ]
    crystals = thin[:2] + [_diamond(8, seed=3)] + thin[2:]
    _search(crystals)
    _assert_host(_search(thin), thin)


def test_zero_cell_cluster():
    pos, _ = _diamond(7, seed=4)  # 2 744 atoms, no periodic images
    ei, sh, _ = _search([(pos, np.zeros((3, 3)))])
    assert ei.shape[1] > 0 and not bool(sh.any())
    small = [(pos[:150], np.zeros((3, 3)))]
    _assert_host(_search(small), small)


def test_dense_centres_beyond_1024_neighbours():
    rng = np.random.default_rng(5)
    cell = np.eye(3) * 12.0
    ei, _, nn = _search([(rng.random((5000, 3)) @ cell, cell)])
    assert float(nn.min()) > 1024


def test_empty_and_one_atom_crystals_in_a_batch():
    crystals = [_diamond(2, seed=6), (np.zeros((0, 3)), np.eye(3) * 4.0), (np.array([[0.5, 0.5, 0.5]]), np.eye(3) * 3.0),
                (np.array([[0.0, 0.0, 0.0]]), np.eye(3) * 50.0), _diamond(2, seed=7)]
    got = _search(crystals)
    _assert_host(got, crystals)


def test_nan_coordinates():
    pos, cell = _diamond(3, seed=8)
    pos[5, 1] = np.nan
    pos[100] = np.nan
    ei, _, nn = _search([(pos, cell)])
    assert float(nn[5]) == 0.0 == float(nn[100])
    assert not bool(((ei == 5) | (ei == 100)).any())
    ei2, _, _ = _search([(pos, np.zeros((3, 3)))])  # zero cell
    assert not bool(((ei2 == 5) | (ei2 == 100)).any())


def test_deterministic():
    from matten_b200 import ops

    args = _batch([_diamond(14, seed=9)])
    a = ops.neighbor_list(*args, R_CUT, method="cells")
    b = ops.neighbor_list(*args, R_CUT, method="cells")
    assert all(torch.equal(x, y) for x, y in zip(a, b))


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def test_auto_selection_launches():
    """The 100 example crystals stay on the pair kernels; a 21 952-atom crystal takes the nl_cells_* kernels."""
    from matten_b200.data.neighbors import batch_from_structures

    with open(os.path.join(GOLDEN, "n100_structures.json")) as f:
        structs = json.load(f)["structures"]
    arr = [{"cart": np.array(s["cart_coords"]), "lattice": np.array(s["lattice"]), "Z": s["atomic_numbers"]}
           for s in structs]
    batch_from_structures(arr, R_CUT, DEV, torch.float64)  # warm-up
    names = _kernel_names(lambda: batch_from_structures(arr, R_CUT, DEV, torch.float64))
    assert any("nl_pairs_kernel" in n for n in names) and not any("nl_cells_" in n for n in names)
    pos, cell = _diamond(14, seed=10)
    big = [{"cart": pos, "lattice": cell, "Z": [14] * len(pos)}]
    names = _kernel_names(lambda: batch_from_structures(big, R_CUT, DEV, torch.float64))
    for k in ("nl_cells_extent_kernel", "nl_cells_pairs_kernel", "nl_cells_order_kernel"):
        assert any(k in n for n in names), k
    assert not any("nl_pairs_kernel" in n and "nl_cells" not in n for n in names)


def test_predict_supercell_matches_its_cell(tmp_path):
    """predict() on a diamond cell and its 12x12x12 supercell (13 824 atoms, cell-list search) in one call: the same
    elastic tensor with mean pooling (fp64), and per atom the same atomic tensor (fp32) as the atom's image in the small
    cell."""
    from matten_b200.data.neighbors import batch_from_structures
    from matten_b200.data.synthetic import diamond_supercell
    from matten_b200.predict import predict, save_pretrained

    species = [6, 14]
    small, cell1 = diamond_supercell(1)
    big, cell12 = diamond_supercell(12)
    z1 = [species[a % 2] for a in range(8)]
    structs = [{"lattice": cell1.tolist(), "atomic_numbers": z1, "cart_coords": small.tolist()},
               {"lattice": cell12.tolist(), "atomic_numbers": z1 * 12 ** 3, "cart_coords": big.tolist()}]
    # fp64, so that the fp32 round-off of a sequential mean over 13 824 atoms (~1e-4) does not hide the comparison
    _, prod = build_pair(HP_LMAX4, species, torch.float64, DEV, seed=3)
    save_pretrained(prod, tmp_path, R_CUT, "elastic_tensor_full")
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)  # predict() builds the model in the default dtype
    try:
        a, b = predict(structs, model_identifier=str(tmp_path), device=DEV)
    finally:
        torch.set_default_dtype(old)
    a, b = np.asarray(a), np.asarray(b)
    assert np.abs(a - b).max() <= 1e-5 * np.abs(a).max()

    _, atomic = build_pair(dict(HP_LMAX2, output_format="cartesian"), species, torch.float32, DEV, seed=4, atomic=True)
    arr = [{"cart": np.asarray(s["cart_coords"]), "lattice": np.asarray(s["lattice"]), "Z": s["atomic_numbers"]}
           for s in structs]
    with torch.no_grad():
        out = atomic(batch_from_structures(arr, R_CUT, DEV, torch.float32))["nmr_tensor"].cpu()
    cell_out, super_out = out[:8], out[8:].reshape(12 ** 3, 8, 3, 3)
    scale = float(cell_out.abs().max())
    assert float((super_out - cell_out[None]).abs().max()) <= 1e-5 * scale
