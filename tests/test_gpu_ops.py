"""GPU parity tests, op by op, through the C ABI (matten_b200.ops -> libmatten_b200.so) against
the CPU oracle on the same seeded inputs.  Integer work is bit-exact; floating point within the
tolerance of BASELINE.json (1e-5 relative in fp32, 1e-10 in fp64; metric = max|a-b| / max|b|)."""
import math

import numpy as np
import pytest
import torch

from tests.helpers import elem_err, rel_err, tol

pytestmark = pytest.mark.gpu
DTYPES = [torch.float32, torch.float64]


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


# ------------------------------------------------------------------ bookkeeping
@pytest.mark.parametrize("E,K", [(0, 5), (1, 1), (37, 3), (5000, 17), (100_000, 70_000), (300_000, 9),
                                 (2048 * 3 + 5, 1 << 17)])
def test_csr_by_key_bit_exact(dev, E, K):
    from matten_b200 import ops

    g = torch.Generator().manual_seed(E + K)
    keys = torch.randint(0, K, (E,), generator=g, dtype=torch.int64)
    flag = ops.new_flag(dev)
    rowptr, perm = ops.csr_by_key(keys.to(dev), K, True, flag)
    ref_perm = np.argsort(keys.numpy(), kind="stable").astype(np.int32)
    ref_ptr = np.concatenate([[0], np.cumsum(np.bincount(keys.numpy(), minlength=K))]).astype(np.int32)
    assert np.array_equal(perm.cpu().numpy(), ref_perm)
    assert np.array_equal(rowptr.cpu().numpy(), ref_ptr)
    rowptr2, none = ops.csr_by_key(keys.to(dev), K, False, flag)
    assert none is None and np.array_equal(rowptr2.cpu().numpy(), ref_ptr)
    assert int(flag.item()) == 0
    if E:
        src = torch.randint(0, 1000, (E,), generator=g, dtype=torch.int64)
        got = ops.gather_i64_to_i32(src.to(dev), perm)
        assert np.array_equal(got.cpu().numpy(), src.numpy()[ref_perm].astype(np.int32))


def test_csr_flags_bad_keys_and_unsorted(dev):
    from matten_b200 import _lib, ops

    flag = ops.new_flag(dev)
    ops.csr_by_key(torch.tensor([0, 7, 2], device=dev), 5, True, flag)
    assert int(flag.item()) & _lib.FLAG_BAD_INDEX
    flag = ops.new_flag(dev)
    ops.check_sorted(torch.tensor([0, 0, 1, 3, 2], device=dev), flag)
    assert int(flag.item()) & _lib.FLAG_UNSORTED
    flag = ops.new_flag(dev)
    ops.check_sorted(torch.tensor([0, 0, 1, 3, 3], device=dev), flag)
    assert int(flag.item()) == 0


# ------------------------------------------------------------------ edge geometry
@pytest.mark.parametrize("dtype", DTYPES)
def test_edge_vectors_sh_radial(dev, dtype):
    from matten_b200 import ops
    from matten_b200.data.synthetic import synthetic_batch
    from oracle import e3nn_restated as E
    from oracle import matten_restated as M

    b = synthetic_batch(3, dtype=dtype)
    ob = {k: v for k, v in b.items() if isinstance(v, torch.Tensor)}
    M.with_edge_vectors(ob)
    d = {k: v.to(dev) for k, v in b.items() if isinstance(v, torch.Tensor)}
    flag = ops.new_flag(dev)
    vec, ln = ops.edge_vectors(d["pos"], d["edge_index"], d["edge_cell_shift"], d["cell"], d["batch"], flag)
    assert rel_err(vec, ob["edge_vectors"]) < tol(dtype)
    assert rel_err(ln, ob["edge_lengths"]) < tol(dtype)
    assert int(flag.item()) == 0
    # single cell without batch vector (cell.shape[0] == 1 branch of the reference)
    one = synthetic_batch(1, dtype=dtype)
    o1 = {k: v for k, v in one.items() if isinstance(v, torch.Tensor) and k != "batch"}
    M.with_edge_vectors(o1)
    v1, l1 = ops.edge_vectors(one["pos"].to(dev), one["edge_index"].to(dev), one["edge_cell_shift"].to(dev),
                              one["cell"].to(dev), None, flag)
    assert rel_err(v1, o1["edge_vectors"]) < tol(dtype)
    # no cell at all
    v2, _ = ops.edge_vectors(one["pos"].to(dev), one["edge_index"].to(dev))
    assert rel_err(v2, one["pos"][one["edge_index"][1]] - one["pos"][one["edge_index"][0]]) < tol(dtype)
    for lmax in range(5):
        sh = ops.edge_sh(vec, lmax)
        ref = E.spherical_harmonics(lmax, ob["edge_vectors"], True, "component")
        assert rel_err(sh, ref) < tol(dtype), lmax
    emb = ops.edge_radial(ln, 0, 8, 0.0, 5.0, True)
    # The yardstick is the oracle evaluated in fp64 on the SAME lengths the kernel saw: north-star bound 1e-5 (fp32),
    # normwise and element-wise.  (Round 1 compared with the fp32 CPU evaluation and once saw 1.5e-4; 300 repetitions
    # of this kernel on a B200 are bitwise identical and 1.2e-6 from fp64, initcheck clean -- profiles/
    # r2_bessel_repeat.json -- so the bound is back where the north star puts it; the fp32 CPU evaluation is only
    # required to agree with fp64 to the same 1e-5, which keeps a libm regression on the host visible as such.)
    ref64 = E.soft_one_hot_linspace_bessel(ln.cpu().double(), 0.0, 5.0, 8, True) * math.sqrt(8)
    assert rel_err(emb, ref64) < tol(dtype)
    # element-wise (floor 1e-3 of the largest value): next to the zeros of sin(n pi x / c) the fp32 rounding of the
    # argument itself (eps * 8 pi ~ 1.5e-6 absolute) is 2e-3 of that floor, so that is the fp32 bound; fp64 has no
    # such excuse
    assert elem_err(emb, ref64) < (2e-3 if dtype == torch.float32 else 1e-9)
    ref = E.soft_one_hot_linspace_bessel(ob["edge_lengths"], 0.0, 5.0, 8, True) * math.sqrt(8)
    assert rel_err(emb, ref) < (2 * tol(dtype) if dtype == torch.float32 else 3 * tol(dtype))
    # cut-off edge cases: beyond r_max -> 0
    far = torch.tensor([4.999, 5.0, 5.5, 7.0], dtype=dtype)
    got = ops.edge_radial(far.to(dev), 0, 8, 0.0, 5.0, True).cpu()
    assert torch.all(got[1:] == 0) and got[0].abs().max() > 0
    # Bessel x polynomial cutoff (nequip style, north star names it)
    rb = M.RadialBasisEdgeEncoding({"r_max": 5.0, "num_basis": 8}, {"r_max": 5.0, "p": 6}).to(dtype)
    o2 = dict(ob)
    rb(o2)
    got = ops.edge_radial(ln, 1, 8, 0.0, 5.0, True, 6.0, rb.basis.bessel_weights.detach().to(dev))
    assert rel_err(got, o2["edge_embedding"]) < 10 * tol(dtype)  # 1-u^6.. envelope cancels near r_max


def test_species_embed_and_kat(dev):
    from matten_b200 import _lib, ops
    from matten_b200.nn.embedding import SpeciesEmbedding, _AtomicNumberToIndex

    # the reference's KAT (tests/nn/test_embedding.py:6-13), on the module and through the kernel
    n2i = _AtomicNumberToIndex([6, 1, 8])
    z = torch.tensor([6, 6, 8, 1, 8])
    assert torch.equal(n2i(z), torch.tensor([1, 1, 2, 0, 2]))
    torch.manual_seed(0)
    lin = torch.nn.Linear(3, 16)
    flag = ops.new_flag(dev)
    idx, attrs, feats = ops.species_embed(z.to(dev), None, n2i._Z_to_index.to(dev), 1, 8, 3, lin.weight.to(dev),
                                          lin.bias.to(dev), flag)
    assert idx.dtype == torch.long and torch.equal(idx.cpu(), torch.tensor([1, 1, 2, 0, 2]))
    onehot = torch.nn.functional.one_hot(idx.cpu(), 3).float()
    assert torch.equal(attrs.cpu(), onehot)
    assert rel_err(feats, lin(onehot)) < 1e-6
    assert int(flag.item()) == 0
    ops.species_embed(torch.tensor([6, 7], device=dev), None, n2i._Z_to_index.to(dev), 1, 8, 3,
                      lin.weight.to(dev), lin.bias.to(dev), flag)
    assert int(flag.item()) & _lib.FLAG_BAD_SPECIES
    flag.zero_()
    ops.species_embed(torch.tensor([6, 9], device=dev), None, n2i._Z_to_index.to(dev), 1, 8, 3,
                      lin.weight.to(dev), lin.bias.to(dev), flag)
    assert int(flag.item()) & _lib.FLAG_BAD_SPECIES


# ------------------------------------------------------------------ linears
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("irr_in,irr_out,S", [
    ("16x0e", "56x0e+16x1o+4x2e+2x3o+2x4e", 8),
    ("54x0o+56x0e+100x1o+100x1e+110x2o+112x2e", "32x0o+32x0e+16x1o+16x1e+4x2o+4x2e", 8),
    ("22x0o+56x0e+100x1o+68x1e+78x2o+112x2e+110x3o+78x3e+90x4e",
     "32x0o+78x0e+16x1o+16x1e+4x2o+4x2e+2x3o+2x3e+2x4e", 3),
    ("32x0e+16x1o", "32x0e+16x1o", 1),
    # unaligned everything (odd row length, multiplicities not multiples of 4: the 4-byte staging paths, zero-padded
    # input channels), short rows (CTA-synchronous kernel) and long rows (warp-private kernel)
    ("5x0e+3x1o+1x2e", "7x0e+3x1o+2x2e", 4),
    ("131x0e+77x1o+45x2e+3x3o", "9x0e+5x1o+3x2e+1x3o", 5),
    # in fp64 too large for one launch: the blocks of one round go into two launches (the widest linear of the
    # reference's hyperparameters), or a dense block is cut into rectangles of its weight
    ("64x0o+64x0e+124x1o+124x1e+148x2o+148x2e+148x3o+148x3e+124x4o+124x4e",
     "32x0o+32x0e+16x1o+16x1e+8x2o+8x2e+4x3o+4x3e+4x4o+4x4e", 2),
    ("600x0e+300x1o", "600x0e+300x1o", 3),
    # in fp64 cut along output channels too, the two blocks of one output range at the same channels
    ("8x0e+4x0e", "7000x0e", 2),
])
def test_species_linear_vs_fctp(dev, dtype, irr_in, irr_out, S):
    from matten_b200 import ops
    from matten_b200.nn.utils import SpeciesLinear
    from oracle import e3nn_restated as E

    torch.manual_seed(1)
    N = 777
    lin = SpeciesLinear(irr_in, S, irr_out).to(dtype)
    ref = E.FullyConnectedTensorProduct(irr_in, f"{S}x0e", irr_out).to(dtype)
    assert ref.weight_numel == lin.weight_numel
    ref.weight.data.copy_(lin.weight.data)
    x = torch.randn(N, lin.irreps_in.dim, dtype=dtype)
    sp = torch.randint(0, S, (N,))
    if S > 2:
        sp[sp == 1] = 0  # an empty species group
    with torch.no_grad():
        want = ref(x, torch.nn.functional.one_hot(sp, S).to(dtype))
    lin = lin.to(dev)
    flag = ops.new_flag(dev)
    ptr, perm = ops.csr_by_key(sp.to(dev), S, True, flag)
    with torch.no_grad():
        got = lin(x.to(dev), perm, ptr)
        assert rel_err(got, want) < tol(dtype)
        res = torch.randn(N, lin.irreps_out.dim, dtype=dtype)
        got2 = lin(x.to(dev), perm, ptr, residual=res.to(dev).clone())
        assert rel_err(got2, want + res) < tol(dtype)
        # a handful of nodes (partial tiles, idle warps) and a single node
        for n_small in (5, 1):
            ptr_s, perm_s = ops.csr_by_key(sp[:n_small].to(dev), S, True, flag)
            got3 = lin(x[:n_small].to(dev), perm_s, ptr_s)
            assert rel_err(got3, want[:n_small]) < tol(dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("irr_in,irr_out,S", [
    ("32x0e+16x1o", "32x0e+16x1o", 1),  # grad_out rows of 80 elements: CTA-synchronous kernel
    ("32x0e+16x1o", "128x0e+96x1o+32x2e", 3),  # rows of 576: warp-private kernel
    ("600x0e+300x1o", "600x0e+300x1o", 3),  # cut along the 600 / 300 output channels of the forward
    ("7000x0e", "8x0e", 2),  # in fp64 cut along the 7000 input channels of the forward as well
])
def test_species_linear_grad_x_vs_autograd(dev, dtype, irr_in, irr_out, S):
    """dL/dx of the species linear (its weights applied transposed) against autograd through the oracle."""
    from matten_b200 import ops
    from matten_b200.nn.utils import SpeciesLinear
    from oracle import e3nn_restated as E

    torch.manual_seed(3)
    N = 777
    lin = SpeciesLinear(irr_in, S, irr_out).to(dtype)
    ref = E.FullyConnectedTensorProduct(irr_in, f"{S}x0e", irr_out).to(dtype)
    ref.weight.data.copy_(lin.weight.data)
    x = torch.randn(N, lin.irreps_in.dim, dtype=dtype)
    g = torch.randn(N, lin.irreps_out.dim, dtype=dtype)
    sp = torch.randint(0, S, (N,))
    xr = x.clone().requires_grad_(True)
    ref(xr, torch.nn.functional.one_hot(sp, S).to(dtype)).backward(g)
    lin = lin.to(dev)
    flag = ops.new_flag(dev)
    ptr, perm = ops.csr_by_key(sp.to(dev), S, True, flag)
    xd = x.to(dev).requires_grad_(True)
    lin(xd, perm, ptr).backward(g.to(dev))
    assert rel_err(xd.grad, xr.grad) < tol(dtype)


@pytest.mark.parametrize("dim", [2, 11])
def test_linear_rejects_block_dims_before_any_launch(dev, dim):
    """Block dims other than 2l+1 <= 9 are MT_EINVAL in the forward and the backward, and nothing runs."""
    from types import SimpleNamespace

    from matten_b200 import ops

    block = SimpleNamespace(in_off=0, out_off=0, mul_in=4, mul_out=4, dim=dim, w_off=0, scale=1.0)
    h = ops.LinPlanHandle([block], 4 * dim, 4 * dim, 1, 16)
    x = torch.randn(37, 4 * dim, device=dev)
    w = torch.randn(16, device=dev)
    before = ops.launch_count()
    with pytest.raises(RuntimeError, match=r"failed \(-1\): bad linear block 0"):
        ops.linear_fwd(h, x, w)
    for need_x, need_w in [(True, True), (True, False), (False, True)]:
        with pytest.raises(RuntimeError, match=r"failed \(-1\): bad linear block 0"):
            ops.linear_bwd(h, x, w, torch.randn_like(x), need_x=need_x, need_w=need_w)
    torch.cuda.synchronize(dev)
    assert ops.launch_count() == before


@pytest.mark.parametrize("dtype", DTYPES)
def test_irreps_linear_and_cartesian(dev, dtype):
    from matten_b200.nn.readout import CartesianTensorWrapper
    from matten_b200.nn.utils import IrrepsLinear
    from oracle import e3nn_restated as E

    torch.manual_seed(2)
    for a, b in [("32x0o+32x0e+16x1o+16x1e+4x2o+4x2e+2x3o+2x3e+2x4e", "16x0e+2x2e+4e"),
                 ("16x0e+2x2e+4e", "2x0e+2x2e+4e"), ("4x0e+6x0e+3x1o", "3x0e+2x1e"),
                 ("8x0e+4x0e", "7000x0e")]:  # cut (in fp64 along output channels too) with a shared output range
        lin = IrrepsLinear(a, b).to(dtype)
        ref = E.Linear(a, b).to(dtype)
        ref.weight.data.copy_(lin.weight.data)
        x = torch.randn(301, lin.irreps_in.dim, dtype=dtype)
        with torch.no_grad():
            assert rel_err(lin.to(dev)(x.to(dev)), ref(x)) < tol(dtype)
    for formula in ["ijkl=jikl=klij", "ij=ji"]:
        ct = CartesianTensorWrapper(formula)
        ref = E.CartesianTensor(formula)
        v = torch.randn(97, ct.dim, dtype=dtype)
        cart = ct.to_cartesian(v.to(dev))
        assert rel_err(cart, ref.to_cartesian(v)) < tol(dtype)
        assert rel_err(ct.from_cartesian(cart), v) < tol(dtype)


# ------------------------------------------------------------------ gate (+ BatchNorm eval)
@pytest.mark.parametrize("dtype", DTYPES)
def test_gate_and_batchnorm_eval(dev, dtype):
    from matten_b200.nn.utils import ActivationLayer, NormalizationLayer
    from oracle import matten_restated as M
    from tests.helpers import HP_LMAX4, randomize_bn

    torch.manual_seed(3)
    sh = "0e+1o+2e+3o+4e"
    for x_ir in ["16x0e", "32x0e+16x1o+4x2e+2x3o+2x4e", "32x0o+32x0e+16x1o+16x1e+4x2o+4x2e+2x3o+2x3e+2x4e"]:
        kw = dict(activation_type="gate", activation_scalars={"e": "silu", "o": "tanh"},
                  activation_gates={"e": "sigmoid", "o": "tanh"})
        act = ActivationLayer(x_ir, sh, HP_LMAX4["conv_layer_irreps"], **kw)
        ref = M.ActivationLayer(x_ir, sh, HP_LMAX4["conv_layer_irreps"], **kw)
        assert act.irreps_in.dim == sum(m * (2 * l + 1) for m, l, _ in ref.irreps_in)
        norm = NormalizationLayer(act.irreps_out, "batch").to(dtype)
        rnorm = M.NormalizationLayer(ref.irreps_out, "batch").to(dtype)
        randomize_bn(torch.nn.ModuleDict({"norm": norm}), 3)
        norm.n.weight.data.uniform_(0.5, 1.5)
        norm.n.bias.data.normal_()
        norm.n.running_mean.normal_()
        norm.n.running_var.uniform_(0.5, 2.0)
        rnorm.load_state_dict(norm.state_dict())
        norm.eval(), rnorm.eval()
        x = torch.randn(513, act.irreps_in.dim, dtype=dtype) * 1.5
        with torch.no_grad():
            want = ref(x)
            got = act.to(dev)(x.to(dev))
            assert rel_err(got, want) < tol(dtype)
            want2 = rnorm(want, None)
            norm = norm.to(dev)
            assert rel_err(norm(got), want2) < tol(dtype)
            a, b = norm.n.eval_affine(dtype)
            assert rel_err(act(x.to(dev), a, b), want2) < tol(dtype)  # fused gate + BN affine
    # default activations of the reference (ssp / abs) and odd gates
    act = ActivationLayer("8x0o+8x1o", "0e+1o", "8x0o+8x0e+8x1o+8x1e")
    ref = M.ActivationLayer("8x0o+8x1o", "0e+1o", "8x0o+8x0e+8x1o+8x1e")
    x = torch.randn(64, act.irreps_in.dim, dtype=dtype)
    with torch.no_grad():
        assert rel_err(act.to(dev)(x.to(dev)), ref(x)) < tol(dtype)


# ------------------------------------------------------------------ pooling
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("mode", ["sum", "mean", "min", "max"])
def test_segment_reduce(dev, dtype, mode):
    from matten_b200 import ops
    from oracle import e3nn_restated as E

    torch.manual_seed(4)
    counts = [3, 1, 0, 64, 7, 0]
    batch = torch.cat([torch.full((c,), i, dtype=torch.int64) for i, c in enumerate(counts)])
    x = torch.randn(len(batch), 35, dtype=dtype)
    flag = ops.new_flag(dev)
    ptr, _ = ops.csr_by_key(batch.to(dev), len(counts), False, flag)
    got = ops.segment_reduce(x.to(dev), ptr, mode)
    want = E.scatter(x, batch, dim_size=len(counts), reduce=mode)
    assert rel_err(got, want) < tol(dtype)


# ------------------------------------------------------------------ fused convolution
def _conv_case(dev, dtype, x_ir, sh_lmax, target_ir, S, n_rad, hidden, nlayers, avg, N, deg_fn, seed):
    from matten_b200 import o3, ops
    from matten_b200.graph import GraphCache
    from matten_b200.nn.conv import PointConv
    from oracle import e3nn_restated as E
    from oracle import matten_restated as M

    torch.manual_seed(seed)
    g = torch.Generator().manual_seed(seed)
    sh_ir = o3.Irreps.spherical_harmonics(sh_lmax)
    irreps_in = {"node_features": o3.Irreps(x_ir), "node_attrs": o3.Irreps(f"{S}x0e"), "edge_attrs": sh_ir,
                 "edge_embedding": o3.Irreps(f"{n_rad}x0e")}
    old = torch.get_default_dtype()
    torch.set_default_dtype(dtype)
    try:
        conv = PointConv(irreps_in, target_ir, nlayers, hidden, avg)
        oin = {k: o3.parse_irreps_list(v) for k, v in irreps_in.items()}
        ref = M.PointConv(oin, target_ir, nlayers, hidden, avg)
    finally:
        torch.set_default_dtype(old)
    missing, unexpected = ref.load_state_dict(conv.state_dict(), strict=False)
    assert not unexpected
    # random graph: receiver n gets deg_fn(n) incoming edges from random senders
    dst = torch.cat([torch.full((deg_fn(n),), n, dtype=torch.int64) for n in range(N)])
    E_ = len(dst)
    src = torch.randint(0, N, (E_,), generator=g)
    shuffle = torch.randperm(E_, generator=g)
    ei = torch.stack([src, dst])[:, shuffle]
    x = torch.randn(N, conv.tp.plan.x_dim, dtype=dtype)
    vec = torch.randn(E_, 3, dtype=dtype)
    sh = E.spherical_harmonics(sh_lmax, vec, True, "component")
    emb = torch.randn(E_, n_rad, dtype=dtype)
    sp = torch.randint(0, S, (N,), generator=g)
    num_neigh = torch.bincount(ei[0], minlength=N).to(dtype).clamp(min=1)
    data = {"node_features": x, "node_attrs": torch.nn.functional.one_hot(sp, S).to(dtype), "edge_attrs": sh,
            "edge_embedding": emb, "edge_index": ei, "num_neigh": num_neigh}
    with torch.no_grad():
        want = ref(dict(data))["node_features"]
        # the un-fused pieces too: aggregated messages
        msg = ref.tp(ref.lin1(x, data["node_attrs"])[ei[0]], sh, emb)
    conv = conv.to(dev)
    d = {k: v.to(dev) for k, v in data.items()}
    d["species_index"] = sp.to(dev)
    d["pos"] = torch.zeros(N, 3, dtype=dtype, device=dev)
    with torch.no_grad():
        got = conv(d)["node_features"]
        graph = d["_mt_graph"]
        graph.raise_if_invalid()
        # per-edge contract of UVUTensorProduct.forward (reference nn/utils.py:255-265)
        sperm, sptr = graph.species_groups(d["species_index"], S)
        h = conv.lin1(d["node_features"] if False else x.to(dev), sperm, sptr)
        got_msg = conv.tp(h[ei[0].to(dev)], sh.to(dev), emb.to(dev))
        got2 = conv(dict(d, node_features=x.to(dev)))["node_features"]
    assert rel_err(got_msg, msg) < tol(dtype)
    assert rel_err(got, want) < tol(dtype)
    assert torch.equal(got, got2), "segmented reduction must be bit-deterministic"
    return conv, ref


@pytest.mark.parametrize("dtype", DTYPES)
def test_conv_lmax2_layers(dev, dtype):
    ir = "32x0o+32x0e+16x1o+16x1e+4x2o+4x2e"
    _conv_case(dev, dtype, "16x0e", 2, "52x0e+16x1o+4x2e", 8, 8, 32, 2, 28.0, 300, lambda n: 28, 0)
    _conv_case(dev, dtype, "32x0e+16x1o+4x2e", 2, "72x0e+16x1o+16x1e+4x2o+4x2e", 8, 8, 32, 2, 28.0, 200,
               lambda n: 28, 1)
    _conv_case(dev, dtype, ir, 2, ir, 8, 8, 32, 2, 28.0, 150, lambda n: 28, 2)


@pytest.mark.parametrize("dtype", DTYPES)
def test_conv_lmax4_and_ragged(dev, dtype):
    ir4 = "32x0o+32x0e+16x1o+16x1e+4x2o+4x2e+2x3o+2x3e+2x4e"
    # ragged: nodes without in-edges, nodes with more edges than one shared-memory chunk
    deg = lambda n: [0, 1, 3, 500, 28, 0, 64, 65][n % 8]  # noqa: E731
    _conv_case(dev, dtype, ir4, 4, ir4, 5, 8, 32, 2, 30.4, 48, deg, 3)
    # per-node sqrt(num_neigh) normalisation (average_num_neighbors = None), test-config irreps
    irt = "32x0o+32x0e+16x1o+16x1e+8x2o+8x2e+4x3o+4x3e+4x4o+4x4e"
    _conv_case(dev, dtype, irt, 4, irt, 2, 10, 32, 2, None, 40, lambda n: 5 + (n % 7), 4)


@pytest.mark.parametrize("dtype", DTYPES)
def test_conv_mlp_variants(dev, dtype):
    ir = "8x0e+8x1o+4x2e"
    # default fc sizes of the reference (1 hidden layer of 8), 64 hidden units, and no hidden layer
    _conv_case(dev, dtype, ir, 2, ir, 3, 8, 8, 1, 10.0, 64, lambda n: 12, 5)
    _conv_case(dev, dtype, ir, 2, ir, 3, 8, 64, 2, 10.0, 64, lambda n: 12, 6)
    _conv_case(dev, dtype, ir, 2, ir, 1, 10, 8, 0, 10.0, 64, lambda n: 12, 7)
    _conv_case(dev, dtype, ir, 1, ir, 3, 8, 16, 3, 10.0, 64, lambda n: 12, 8)


# ------------------------------------------------------------------ tcgen05 path of the convolution
def _with_impl(impl, fn):
    from matten_b200 import ops

    old = ops.conv_select_impl(impl)
    try:
        return fn()
    finally:
        ops.conv_select_impl(old)


@pytest.mark.parametrize("impl", ["tc", "fma"])
def test_conv_tensor_core_and_fma_paths(dev, impl):
    """Both fp32 implementations of mt_conv_fwd (tcgen05 radial MLP + TMEM weights, and the FMA-pipe
    kernel) against the oracle: the bench layers, packed small types, ragged degrees (empty nodes,
    exactly 64 / 65 / 500 edges: chunk boundaries and split nodes), per-node normalisation."""
    ir = "32x0o+32x0e+16x1o+16x1e+4x2o+4x2e"
    f32 = torch.float32
    deg = lambda n: [0, 1, 3, 500, 28, 0, 64, 65, 63, 2, 130, 0][n % 12]  # noqa: E731

    def run():
        _conv_case(dev, f32, "16x0e", 2, "52x0e+16x1o+4x2e", 8, 8, 32, 2, 28.0, 300, lambda n: 28, 10)
        _conv_case(dev, f32, "32x0e+16x1o+4x2e", 2, "72x0e+16x1o+16x1e+4x2o+4x2e", 8, 8, 32, 2, 28.0, 300,
                   lambda n: 27 + (n % 3), 11)
        _conv_case(dev, f32, ir, 2, ir, 8, 8, 32, 2, 28.0, 333, lambda n: 28, 12)
        _conv_case(dev, f32, ir, 2, ir, 4, 8, 32, 2, 30.4, 60, deg, 13)
        _conv_case(dev, f32, ir, 2, ir, 4, 8, 32, 2, None, 60, deg, 14)
        _conv_case(dev, f32, "8x0e+8x1o+4x2e", 2, "8x0e+8x1o+4x2e", 3, 8, 8, 1, 10.0, 64, lambda n: 12, 15)
        _conv_case(dev, f32, "8x0e+8x1o+4x2e", 2, "8x0e+8x1o+4x2e", 1, 10, 8, 0, 10.0, 64, lambda n: 12, 16)
        _conv_case(dev, f32, "20x0e+12x1o+4x2e+4x1e", 2, "20x0e+12x1o+4x2e+4x1e", 2, 8, 16, 2, 9.0, 100,
                   lambda n: n % 40, 17)

    _with_impl(impl, run)
    # row length not a multiple of 4 floats (TMA rows are multiples of 16 bytes): automatic fallback to the FMA kernel
    _with_impl("auto", lambda: _conv_case(dev, f32, "20x0e+12x1o+5x2e+3x1e", 2, "20x0e+12x1o+5x2e+3x1e", 2, 8, 16, 2,
                                          9.0, 60, lambda n: n % 30, 20))
    # three hidden layers: the tensor-core path keeps at most two in registers -> automatic fallback
    _with_impl("auto", lambda: _conv_case(dev, f32, "20x0e+12x1o+5x2e", 2, "20x0e+12x1o+5x2e", 2, 8, 16, 3, 9.0,
                                          50, lambda n: n % 20, 19))


def test_conv_tc_matches_fma_bitwise_determinism(dev):
    """the tensor-core path is deterministic run to run as well"""
    ir = "32x0o+32x0e+16x1o+16x1e+4x2o+4x2e"
    _with_impl("tc", lambda: _conv_case(dev, torch.float32, ir, 2, ir, 8, 8, 32, 2, 28.0, 500,
                                        lambda n: 20 + (n % 17), 18))


# ------------------------------------------------------------------ periodic neighbour list on the GPU
def test_neighbor_list_bit_exact_against_host_search(dev):
    """mt_neighbor_count / mt_neighbor_fill against the numpy search (same semantics as the reference's ASE call):
    identical edge lists (index bookkeeping is bit exact), shifts and neighbour counts -- the 100 example crystals
    (triclinic cells, 1..20 atoms, up to 5 images per axis) and jittered 64-atom supercells."""
    import json
    import os

    import numpy as np

    from matten_b200.data.neighbors import batch_from_structures, collate, make_graph
    from matten_b200.data.synthetic import synthetic_batch
    from tests.helpers import GOLDEN

    with open(os.path.join(GOLDEN, "n100_structures.json")) as f:
        structs = json.load(f)["structures"]
    arr = [{"cart": np.array(s["cart_coords"]), "lattice": np.array(s["lattice"]), "Z": s["atomic_numbers"]}
           for s in structs]
    want = collate([make_graph(a["cart"], a["lattice"], a["Z"], 5.0, torch.float64) for a in arr])
    got = batch_from_structures(arr, 5.0, dev, torch.float64)
    assert got["edge_index"].shape[1] == 14380  # BASELINE.md
    for k in ("edge_index", "edge_cell_shift", "num_neigh", "batch", "atomic_numbers"):
        assert torch.equal(got[k].cpu(), want[k]), k
    assert torch.equal(got["pos"].cpu(), want["pos"]) and torch.equal(got["cell"].cpu(), want["cell"])
    # synthetic supercells (every atom has exactly 28 neighbours)
    sb = synthetic_batch(3, dtype=torch.float64)
    B = sb["num_graphs"]
    ptr = torch.as_tensor(np.concatenate([[0], np.cumsum(np.bincount(sb["batch"].numpy(), minlength=B))]))
    ei, sh, nn = ops_neighbor(dev, sb, ptr)
    assert torch.equal(ei.cpu(), sb["edge_index"]) and torch.equal(sh.cpu(), sb["edge_cell_shift"])
    assert torch.equal(nn.cpu(), sb["num_neigh"]) and float(nn.min()) == 28.0 == float(nn.max())


def ops_neighbor(dev, sb, ptr):
    from matten_b200 import ops

    return ops.neighbor_list(sb["pos"].to(dev), sb["cell"].reshape(-1, 3, 3).to(dev), sb["batch"].to(dev), ptr.to(dev), 5.0)


def test_ops_follow_the_tensor_device_not_the_current_one():
    """A model / tensor on cuda:1 while cuda:0 is the current device: the C ABI launches on the current device, so the
    op layer must switch to the tensors' device around every call (ADVICE r1, medium).  Needs two GPUs."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    from matten_b200 import ops

    torch.cuda.set_device(0)
    d1 = torch.device("cuda:1")
    vec = torch.randn(1000, 3, device=d1)
    got = ops.edge_sh(vec, 2)
    with torch.cuda.device(d1):
        want = ops.edge_sh(vec, 2)
    assert got.device == d1 and torch.equal(got, want)
    assert torch.cuda.current_device() == 0
