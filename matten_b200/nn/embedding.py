"""Species and edge-length embeddings (reference src/matten/nn/embedding.py)."""
from typing import Dict, List, Tuple

import torch

from .. import functional as F
from ..data.irreps import DataKey, ModuleIrreps
from ..graph import get_graph
from ..o3 import Irreps
from ._nequip import with_edge_vectors


class _AtomicNumberToIndex(torch.nn.Module):
    """Atomic number -> consecutive species index through a LUT (reference
    src/matten/nn/embedding.py:206-263).  The lookup itself happens inside the species
    embedding kernel; ``forward`` is kept for API parity (and the reference's KAT,
    tests/nn/test_embedding.py:6-13) and runs wherever its input lives."""

    def __init__(self, allowed_atomic_numbers: List[int]):
        super().__init__()
        allowed = torch.as_tensor(sorted(allowed_atomic_numbers), dtype=torch.long)
        num_species = len(allowed)
        self.register_buffer("_min_Z", allowed.min())
        self.register_buffer("_max_Z", allowed.max())
        self.register_buffer("_num_species", torch.as_tensor(num_species))
        lut = torch.full((1 + int(self._max_Z) - int(self._min_Z),), -1, dtype=torch.long)
        lut[allowed - self._min_Z] = torch.arange(num_species).to(torch.long)
        self.register_buffer("_Z_to_index", lut)
        self._host = (int(allowed.min()), int(allowed.max()), num_species)

    def forward(self, atomic_numbers: torch.Tensor) -> torch.Tensor:
        if atomic_numbers.min() < self._min_Z or atomic_numbers.max() > self._max_Z:
            raise RuntimeError(
                f"Invalid atomic numbers. Expect atomic numbers to be in the range [{self._min_Z}, "
                f"{self._max_Z}], but got min {atomic_numbers.min()} and max {atomic_numbers.max()}")
        index = self._Z_to_index[atomic_numbers - self._min_Z]
        if index.min() < 0:
            bad = atomic_numbers[index < 0][0]
            raise RuntimeError(f"Expect atomic numbers to be in the allowed species, got invalid atomic "
                               f"number `{int(bad)}`.")
        return index

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)
        self._host = (int(self._min_Z), int(self._max_Z), int(self._num_species))

    @property
    def num_species(self):
        return self._host[2]


class SpeciesEmbedding(ModuleIrreps, torch.nn.Module):
    """One-hot species -> Linear(S, embedding_dim) (reference src/matten/nn/embedding.py:12-110).
    The one-hot is only ever a selector, so the kernel gathers a column of the weight."""

    def __init__(self, irreps_in: Dict[str, Irreps] = None, embedding_dim: int = 16, num_species: int = None,
                 allowed_species: List[int] = None,
                 out_fields: Tuple[str] = (DataKey.NODE_ATTRS, DataKey.NODE_FEATURES),
                 use_atom_feats: bool = False, atom_feats_dim: int = None):
        super().__init__()
        self.embedding_dim, self.out_fields, self.use_atom_feats = embedding_dim, out_fields, use_atom_feats
        if allowed_species is not None and num_species is not None:
            raise ValueError("allowed_species and num_species cannot both be provided.")
        if allowed_species is not None:
            self.atomic_number_to_index = _AtomicNumberToIndex(allowed_species)
            self.num_species = self.atomic_number_to_index.num_species
        elif num_species is not None:
            self.atomic_number_to_index = None
            self.num_species = num_species  # the reference forgets this assignment (embedding.py:53-70)
        else:
            raise ValueError("one of allowed_species / num_species is required")
        if use_atom_feats:
            if atom_feats_dim is None:
                raise ValueError("`atom_feats_dim` must be provided if `use_atom_feats` is True.")
            feats_dim = embedding_dim + atom_feats_dim
        else:
            feats_dim = embedding_dim
        self.init_irreps(irreps_in, {DataKey.NODE_ATTRS: Irreps(f"{self.num_species}x0e"),
                                     DataKey.NODE_FEATURES: Irreps(f"{feats_dim}x0e")})
        self.linear = torch.nn.Linear(self.num_species, embedding_dim)

    def forward(self, data: DataKey.Type) -> DataKey.Type:
        g = get_graph(data)
        if DataKey.SPECIES_INDEX in data:
            Z, idx = None, data[DataKey.SPECIES_INDEX]
            lut, zmin, zmax = None, 0, 0
        elif DataKey.ATOMIC_NUMBERS in data:
            if self.atomic_number_to_index is None:
                raise ValueError("atomic_numbers given but the module was built with num_species")
            Z, idx = data[DataKey.ATOMIC_NUMBERS], None
            a = self.atomic_number_to_index
            lut, zmin, zmax = a._Z_to_index, a._host[0], a._host[1]
        else:
            raise ValueError("Nothing in `data` to encode. Need either species_index or atomic_numbers")
        idx, attrs, embed = F.species_embed(Z, idx, lut, zmin, zmax, self.num_species, self.linear.weight,
                                            self.linear.bias, g.flag)
        data[DataKey.SPECIES_INDEX] = idx
        if self.use_atom_feats:
            embed = torch.hstack((embed, data["atom_feats"]))
        data[DataKey.NODE_ATTRS] = attrs
        data[DataKey.NODE_FEATURES] = embed
        return data


# e3nn soft_one_hot_linspace basis -> radial mode of ops.edge_radial (include/matten_b200.h, mt_edge_radial)
_RADIAL_MODE = {"bessel": 0, "gaussian": 3, "cosine": 4, "smooth_finite": 5, "fourier": 6}


class EdgeLengthEmbedding(ModuleIrreps, torch.nn.Module):
    """e3nn ``soft_one_hot_linspace`` of the edge length times sqrt(num_basis) (reference
    src/matten/nn/embedding.py:158-203), for any of e3nn's bases: bessel, gaussian, cosine, smooth_finite and
    fourier."""

    REQUIRED_KEYS_IRREPS_IN = [DataKey.POSITIONS, DataKey.EDGE_INDEX]

    def __init__(self, irreps_in: Dict[str, Irreps] = None, out_field: str = DataKey.EDGE_EMBEDDING,
                 num_basis: int = 10, start: float = 0.0, end: float = 5.0, basis: str = "bessel",
                 cutoff: bool = True):
        super().__init__()
        if basis not in _RADIAL_MODE:
            raise ValueError(f'basis="{basis}" is not a valid entry')
        if basis in ("gaussian", "cosine", "smooth_finite") and not cutoff and num_basis < 2:
            # the centres are linspace(start, end, num_basis), and their spacing is the width of each function
            raise ValueError(f'basis="{basis}" without cutoff needs num_basis >= 2, got {num_basis}')
        self.num_basis, self.start, self.end, self.basis, self.cutoff = num_basis, start, end, basis, cutoff
        self.out_field = out_field
        self.init_irreps(irreps_in, irreps_out={out_field: Irreps(f"{num_basis}x0e")})

    def forward(self, data: DataKey.Type) -> DataKey.Type:
        data = with_edge_vectors(data, with_lengths=True)
        data[self.out_field] = F.edge_radial(data[DataKey.EDGE_LENGTH], _RADIAL_MODE[self.basis], self.num_basis,
                                             self.start, self.end, self.cutoff)
        return data
