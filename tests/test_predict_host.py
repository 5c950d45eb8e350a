"""Host logic of predict(): structure parsing, species check, tolerant checkpoint loading (Lightning checkpoints
reference classes of packages that are not installed here)."""
import pickle

import numpy as np
import pytest
import torch

from matten_b200 import predict as P


def test_structure_arrays_from_dict_variants():
    lat = np.array([[3.348898, 0.0, 1.933487], [1.116299, 3.157372, 1.933487], [0.0, 0.0, 3.866975]])
    frac = [[0.25, 0.25, 0.25], [0, 0, 0]]
    a = P._structure_arrays({"lattice": lat, "species": ["Si", "Si"], "coords": frac})
    assert a["Z"] == [14, 14]
    assert np.allclose(a["cart"], np.asarray(frac) @ lat)
    b = P._structure_arrays({"lattice": {"matrix": lat.tolist()}, "atomic_numbers": [14, 14],
                             "cart_coords": (np.asarray(frac) @ lat).tolist()})
    assert np.allclose(a["cart"], b["cart"]) and b["Z"] == [14, 14]
    # pymatgen Structure.as_dict() layout
    c = P._structure_arrays({"lattice": {"matrix": lat.tolist()},
                             "sites": [{"species": [{"element": "Si", "occu": 1}], "xyz": x.tolist()}
                                       for x in np.asarray(frac) @ lat]})
    assert np.allclose(a["cart"], c["cart"]) and c["Z"] == [14, 14]


def test_check_species_message():
    class M:
        hparams = {"dataset_hparams": {"allowed_species": [8, 14]}}

    P.check_species(M(), [{"Z": [14, 8]}])
    with pytest.raises(RuntimeError, match=r"structure 1.*Fe \(26\).*not supported"):
        P.check_species(M(), [{"Z": [14]}, {"Z": [26, 8]}])


class _Gone:  # stands for e.g. a torchmetrics object pickled into a Lightning checkpoint
    def __init__(self):
        self.value = 3


def test_load_checkpoint_with_missing_classes(tmp_path):
    import sys
    import types

    mod = types.ModuleType("not_installed_pkg")
    cls = type("Metric", (), {"__module__": "not_installed_pkg"})
    mod.Metric = cls
    sys.modules["not_installed_pkg"] = mod
    obj = cls()
    obj.value = 3
    ck = {"state_dict": {"backbone.w": torch.arange(4.0)}, "hyper_parameters": {"dataset_hparams": {"allowed_species": [1]}},
          "callbacks": {"m": obj}}
    path = tmp_path / "model_final.ckpt"
    torch.save(ck, path)
    del sys.modules["not_installed_pkg"]  # the package is "not installed" at load time
    out = P.load_checkpoint(path)
    assert torch.equal(out["state_dict"]["backbone.w"], torch.arange(4.0))
    assert out["hyper_parameters"]["dataset_hparams"]["allowed_species"] == [1]
    # a bare state_dict file is wrapped
    torch.save({"w": torch.ones(2)}, tmp_path / "sd.pt")
    assert "state_dict" in P.load_checkpoint(tmp_path / "sd.pt")


def test_predict_requires_cuda_when_absent(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        P.predict({"lattice": np.eye(3) * 4, "species": ["Si"], "coords": [[0, 0, 0]]})


def test_get_pretrained_model_loads_a_state_dict_with_the_e3nn_layout(tmp_path):
    """A real Lightning checkpoint of the reference carries e3nn's EMPTY placeholder tensors (`tp.tp.weight` of the uvu
    product with external weights, `act.activation.mul.weight`, the `bias` of bias-free o3.Linear, ...), constant
    buffers (`_w3j`, `output_mask`) and `metrics.*` entries.  The oracle's modules register the same placeholders:
    its state_dict, wrapped in the Lightning layout, must load (ADVICE r1, high)."""
    from oracle import matten_restated as M
    from tests.helpers import HP_LMAX2, SPECIES8

    torch.manual_seed(0)
    ds = {"allowed_species": SPECIES8}
    orac = M.ScalarTensorModel(HP_LMAX2, ds)
    sd = {k: v.clone() for k, v in orac.state_dict().items()}
    assert any(v.numel() == 0 for v in sd.values()), "the oracle mirrors e3nn's empty placeholder buffers"
    sd["metrics.train.mae.total"] = torch.zeros(())  # torchmetrics state Lightning stores next to the weights
    d = tmp_path / "pretrained_x"
    d.mkdir()
    torch.save({"state_dict": sd, "hyper_parameters": {"backbone_hparams": dict(HP_LMAX2), "dataset_hparams": ds}},
               d / "model_final.ckpt")
    model = P.get_pretrained_model(str(d))
    got = model.state_dict()
    for k, v in got.items():
        assert torch.equal(v, sd[k]), k
    # a tensor with content that the model does not know is still an error
    sd["backbone.layer0_convnet.conv.bogus"] = torch.ones(3)
    torch.save({"state_dict": sd, "hyper_parameters": {"backbone_hparams": dict(HP_LMAX2), "dataset_hparams": ds}},
               d / "model_final.ckpt")
    with pytest.raises(RuntimeError, match="does not match"):
        P.get_pretrained_model(str(d))


def test_save_pretrained_writes_what_predict_reads(tmp_path):
    from matten_b200.model_factory import ScalarTensorModel
    from tests.helpers import HP_LMAX2, SPECIES8

    model = ScalarTensorModel(HP_LMAX2, {"allowed_species": SPECIES8})
    d = P.save_pretrained(model, tmp_path / "m", r_cut=5.0, tensor_target_name="elastic_tensor_full")
    cfg = P.get_pretrained_config(str(d))
    assert cfg["data"] == {"r_cut": 5.0, "tensor_target_name": "elastic_tensor_full", "tensor_target_formula": "ij=ji"}
    again = P.get_pretrained_model(str(d))
    for k, v in model.state_dict().items():
        assert torch.equal(v, again.state_dict()[k])
