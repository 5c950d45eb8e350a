"""Forward time of the lmax-4 model on 512 synthetic crystals."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from matten_b200.model_factory import ScalarTensorModel  # noqa: E402
from tools.lmax4_hp import HP  # noqa: E402

dev = torch.device("cuda:0")
torch.manual_seed(0)
model = ScalarTensorModel(HP, {"allowed_species": bench.SPECIES}).to(dev).eval()
host = bench.make_batch(512, 0)
keys = ["pos", "edge_index", "edge_cell_shift", "cell", "batch", "atomic_numbers", "num_neigh"]
res = {k: host[k].to(dev) for k in keys}
res["num_graphs"] = host["num_graphs"]
with torch.no_grad():
    for _ in range(2):
        model(res, check=False)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(5):
        model(res, check=False)
    ev1.record()
    torch.cuda.synchronize()
print(f"{ev0.elapsed_time(ev1) / 5:.2f} ms")
