"""Edge geometry modules (reference src/matten/nn/_nequip.py): edge vectors, spherical
harmonic edge attributes, Bessel x polynomial-cutoff radial encoding.  All arithmetic runs
in matten_b200/csrc/graph_ops.cu."""
import math
from typing import Union

import torch

from .. import functional as F
from .. import o3
from ..data.irreps import DataKey, ModuleIrreps
from ..graph import get_graph


def with_edge_vectors(data: DataKey.Type, with_lengths: bool = True) -> DataKey.Type:
    """reference src/matten/nn/_nequip.py:214-268"""
    if DataKey.EDGE_VECTORS in data:
        if with_lengths and DataKey.EDGE_LENGTH not in data:
            # |v| of precomputed vectors: zero positions + the vectors as "shift" through an identity cell
            v = data[DataKey.EDGE_VECTORS]
            data[DataKey.EDGE_LENGTH] = F.vector_lengths(v)
        return data
    g = get_graph(data)
    vec, ln = F.edge_vectors(data[DataKey.POSITIONS], g.edge_index, data.get(DataKey.EDGE_CELL_SHIFT),
                             data.get(DataKey.CELL), data.get(DataKey.BATCH), g.flag, g)
    data[DataKey.EDGE_VECTORS] = vec
    data[DataKey.EDGE_LENGTH] = ln  # computed in the same pass; harmless when not requested
    return data


def with_batch(data: DataKey.Type) -> DataKey.Type:
    """reference src/matten/nn/_nequip.py:272-285"""
    if DataKey.BATCH not in data:
        pos = data[DataKey.POSITIONS]
        data[DataKey.BATCH] = torch.zeros(len(pos), dtype=torch.long, device=pos.device)
    return data


class SphericalHarmonicEdgeAttrs(ModuleIrreps, torch.nn.Module):
    """reference src/matten/nn/_nequip.py:130-176"""

    def __init__(self, irreps_edge_sh: Union[int, str, o3.Irreps], edge_sh_normalization: str = "component",
                 edge_sh_normalize: bool = True, irreps_in=None, out_field: str = DataKey.EDGE_ATTRS):
        super().__init__()
        self.out_field = out_field
        if isinstance(irreps_edge_sh, int):
            self.irreps_edge_sh = o3.Irreps.spherical_harmonics(irreps_edge_sh)
        else:
            self.irreps_edge_sh = o3.Irreps(irreps_edge_sh)
        lmax = len(self.irreps_edge_sh) - 1
        if self.irreps_edge_sh != o3.Irreps.spherical_harmonics(lmax):
            raise NotImplementedError("the CUDA kernel evaluates the full set 0e+1o+...+lmax")
        if edge_sh_normalization != "component":
            raise NotImplementedError("only 'component' normalisation is generated")
        self.lmax = lmax
        self.normalize = edge_sh_normalize
        self.init_irreps(irreps_in=irreps_in, irreps_out={out_field: self.irreps_edge_sh})

    def forward(self, data: DataKey.Type) -> DataKey.Type:
        data = with_edge_vectors(data, with_lengths=False)
        data[self.out_field] = F.edge_sh(data[DataKey.EDGE_VECTORS], self.lmax, self.normalize)
        return data


class BesselBasis(torch.nn.Module):
    """reference src/matten/nn/_nequip.py:80-126 (holds the trainable frequencies)."""

    def __init__(self, r_max, num_basis=8, trainable=True):
        super().__init__()
        self.trainable, self.num_basis, self.r_max = trainable, num_basis, float(r_max)
        self.prefactor = 2.0 / self.r_max
        w = torch.linspace(start=1.0, end=num_basis, steps=num_basis) * math.pi
        if trainable:
            self.bessel_weights = torch.nn.Parameter(w)
        else:
            self.register_buffer("bessel_weights", w)


class PolynomialCutoff(torch.nn.Module):
    """reference src/matten/nn/_nequip.py:43-76"""

    def __init__(self, r_max, p=6):
        super().__init__()
        self.register_buffer("p", torch.Tensor([p]))
        self.register_buffer("r_max", torch.Tensor([r_max]))


class RadialBasisEdgeEncoding(ModuleIrreps, torch.nn.Module):
    """reference src/matten/nn/_nequip.py:180-210 (Bessel basis x polynomial cutoff)."""

    def __init__(self, basis=BesselBasis, cutoff=PolynomialCutoff, basis_kwargs={}, cutoff_kwargs={},
                 out_field: str = DataKey.EDGE_EMBEDDING, irreps_in=None):
        super().__init__()
        self.basis = basis(**basis_kwargs)
        self.cutoff = cutoff(**cutoff_kwargs)
        self.out_field = out_field
        self.init_irreps(irreps_in=irreps_in,
                         irreps_out={self.out_field: o3.Irreps([(self.basis.num_basis, (0, 1))])})

    def forward(self, data: DataKey.Type) -> DataKey.Type:
        data = with_edge_vectors(data, with_lengths=True)
        r = data[DataKey.EDGE_LENGTH]
        data[self.out_field] = F.edge_radial(r, 1, self.basis.num_basis, 0.0, self.basis.r_max, True,
                                             float(self.cutoff.p.item()),
                                             self.basis.bessel_weights.to(r.dtype))
        return data
