"""The per-batch edge layout of the fp32 tcgen05 convolution: ``ops.conv_fwd`` without a layout builds the same layout
in its workspace that ``ops.conv_layout`` builds for a batch, with the same kernels, so the two calls give bitwise the
same output and launch the same kernels."""
import pytest
import torch

pytestmark = pytest.mark.gpu

# the four lmax-2 layers of the bench model (tools/tc_check.py)
BENCH_XINS = ["16x0e", "32x0e+16x1o+4x2e", "32x0e+16x1o+16x1e+4x2o+4x2e", "32x0o+32x0e+16x1o+16x1e+4x2o+4x2e"]
BENCH_TGTS = ["52x0e+16x1o+4x2e", "72x0e+16x1o+16x1e+4x2o+4x2e", "32x0o+72x0e+16x1o+16x1e+4x2o+4x2e",
              "32x0o+32x0e+16x1o+16x1e+4x2o+4x2e"]
IR2 = "32x0o+32x0e+16x1o+16x1e+4x2o+4x2e"
IR4 = "32x0o+32x0e+16x1o+16x1e+4x2o+4x2e+2x3o+2x3e+2x4e"
RAGGED = [0, 1, 3, 65, 28, 0, 64, 65, 63, 2, 130, 0]


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _check(dev, x_ir, sh_lmax, target_ir, hidden, nlayers, act, N, deg_fn, seed, avg=28.0, min_parts=1):
    from matten_b200 import o3, ops
    from matten_b200.graph import GraphCache
    from matten_b200.nn.utils import UVUTensorProduct

    torch.manual_seed(seed)
    g = torch.Generator().manual_seed(seed)
    tp = UVUTensorProduct(o3.Irreps(x_ir), o3.Irreps.spherical_harmonics(sh_lmax), o3.Irreps(target_ir),
                          mlp_input_size=8, mlp_hidden_size=hidden, mlp_num_hidden_layers=nlayers,
                          mlp_activation=act).to(dev)
    assert len(tp.plan.tc.parts) >= min_parts
    handle = tp.handle(dev)
    ws = [w.detach() for w in tp.weight_nn.weights()]
    dst = torch.cat([torch.full((deg_fn(n),), n, dtype=torch.int64) for n in range(N)])
    E = len(dst)
    src = torch.randint(0, N, (E,), generator=g)
    ei = torch.stack([src, dst])[:, torch.randperm(E, generator=g)].to(dev)
    graph = GraphCache({"edge_index": ei, "pos": torch.zeros(N, 3, device=dev)})
    x = torch.randn(N, tp.plan.x_dim, generator=g).to(dev)
    sh = ops.edge_sh(torch.randn(E, 3, generator=g).to(dev), sh_lmax, True)
    emb = torch.randn(E, 8, generator=g).to(dev)
    num_neigh = None if avg is not None else torch.bincount(ei[1], minlength=N).float().clamp(min=1)

    def fwd(layout):
        return ops.conv_fwd(handle, x, sh, emb, ws, graph.rowptr, graph.perm, graph.src_sorted, avg, num_neigh,
                            layout=layout)

    old = ops.conv_select_impl("tc")  # an error, not a silent fallback, if the plan does not take the tcgen05 path
    try:
        n0 = ops.launch_count()
        without = fwd(None)
        n1 = ops.launch_count()
        layout = ops.conv_layout(sh, handle.tc_y_lmax, graph.rowptr, graph.perm, graph.src_sorted, N)
        with_layout = fwd(layout)
        n2 = ops.launch_count()
    finally:
        ops.conv_select_impl(old)
    torch.cuda.synchronize()
    assert torch.isfinite(without).all() and without.abs().max() > 0
    assert torch.equal(without, with_layout)
    assert n1 - n0 == n2 - n1, "a call without a layout prepares it exactly as conv_layout does"


@pytest.mark.parametrize("layer", range(4))
def test_layout_bench_layers(dev, layer):
    _check(dev, BENCH_XINS[layer], 2, BENCH_TGTS[layer], 32, 2, "silu", 2048, lambda n: 28, layer)


def test_layout_lmax4_parts(dev):
    _check(dev, IR4, 4, IR4, 32, 2, "silu", 300, lambda n: 20 + n % 9, 10, avg=30.4, min_parts=2)


@pytest.mark.parametrize("hidden,nlayers,act", [(8, 1, "silu"), (32, 2, "tanh"), (16, 2, "silu")])
def test_layout_generic_hidden_kernel(dev, hidden, nlayers, act):
    _check(dev, IR2, 2, IR2, hidden, nlayers, act, 256, lambda n: 12 + n % 5, 20 + nlayers)


@pytest.mark.parametrize("sh_lmax,nlayers,avg", [(2, 2, 28.0), (2, 1, None), (4, 2, None)])
def test_layout_ragged_degrees(dev, sh_lmax, nlayers, avg):
    ir = IR2 if sh_lmax == 2 else IR4
    _check(dev, ir, sh_lmax, ir, 32 if nlayers == 2 else 8, nlayers, "silu", 96, lambda n: RAGGED[n % len(RAGGED)],
           30 + sh_lmax + nlayers, avg=avg)
