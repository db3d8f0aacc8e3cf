"""GPU parity: every layer of the product ``sparseconvnet`` (hand-written sm_100a kernels behind the
C ABI) against the CPU oracle (oracle/scn_oracle.py through oracle/sparseconvnet_oracle) on the same
seeded inputs.

Bars (written here, per BASELINE.json north_star):
  * rulebooks / row numbering / coordinates: bit-exact, order-normalised per kernel offset
  * "fp32" mode (exact FMA path): relative max-norm error <= 1e-4
  * "mixed" / "bf16" modes (bf16 tensor-core operands, fp32 accumulate): relative L2 error <= 2e-3
    against the oracle evaluated under the SAME stated precision (oracle float64 arithmetic on the
    bf16-rounded operands / bf16-stored features the kernels see: oscn.set_numerics)
"""
import numpy as np
import pytest
import torch

from helpers import blob_sites, random_sites, rel_err, rel_l2
from oracle import scn_oracle as O
from oracle import sparseconvnet_oracle as oscn

pytestmark = pytest.mark.gpu

TOL_FP32 = 1e-4
TOL_BF16 = 2e-3
ABS_FLOOR = 1e-3


@pytest.fixture(scope="module")
def scn():
    import sparseconvnet as s
    return s


def q(t, mode):
    """Make values bf16-representable for the bf16-operand modes (the 'inputs stated' of the bar)."""
    return t.bfloat16().float() if mode != "fp32" else t


def make_input(coords, c, seed, mode):
    g = torch.Generator().manual_seed(seed)
    feats = q(torch.randn(coords.shape[0], c, generator=g), mode)
    return torch.as_tensor(coords), feats


def copy_params(dst, src, mode):
    sd = {k: q(v.detach().clone().float(), mode) if v.dtype.is_floating_point else v.clone()
          for k, v in src.state_dict().items()}
    dst.load_state_dict(sd)
    src.load_state_dict(sd)


def check(a, b, mode, what):
    a = a.detach().float().cpu()
    b = b.detach().float().cpu()
    assert a.shape == b.shape, what
    if b.numel() == 0:
        return
    # Quantities whose exact value is 0 (e.g. the gradient of a conv bias that feeds a BatchNorm) carry
    # only rounding noise on both sides: the denominator is floored at ABS_FLOOR per element.
    if mode == "fp32":
        e = float((a - b).abs().max() / b.abs().max().clamp_min(ABS_FLOOR))
        assert e <= TOL_FP32, f"{what}: rel max err {e:.3e} > {TOL_FP32}"
    else:
        e = float((a - b).double().norm() / b.double().norm().clamp_min(ABS_FLOOR * b.numel() ** 0.5))
        assert e <= TOL_BF16, f"{what}: rel L2 err {e:.3e} > {TOL_BF16}"


# --------------------------------------------------------------------------- integer work: bit-exact


@pytest.mark.parametrize("dup", [0, 37])
@pytest.mark.parametrize("dtype", [torch.int64, torch.float64, torch.float32, torch.int32])
def test_input_layer_rows_bit_exact(scn, dup, dtype):
    coords = random_sites(500, (20, 12, 30), 3, seed=1, dup=dup)
    feats = torch.randn(coords.shape[0], 2)
    rows_ref, active_ref = O.input_layer_rules(coords)
    layer = scn.InputLayer(3, [20, 12, 30])
    out = layer((torch.as_tensor(coords).to(dtype).cuda(), feats.cuda(), 3))
    assert np.array_equal(out.metadata.row_of_input.cpu().numpy().astype(np.int64), rows_ref)
    assert np.array_equal(out.get_spatial_locations().numpy(), active_ref)
    ref = O.input_layer_forward(feats.double(), rows_ref, active_ref.shape[0], 3)
    assert rel_err(out.features, ref) < 1e-6
    assert out.batch_size() == 3


def test_input_layer_mean_mode_and_cpu_coords(scn):
    coords = random_sites(200, (9, 9, 9), 2, seed=2, dup=50)
    feats = torch.randn(coords.shape[0], 3)
    rows_ref, active_ref = O.input_layer_rules(coords)
    out = scn.InputLayer(3, 9, mode=4)((torch.as_tensor(coords), feats.cuda()))   # coords left on the host
    ref = O.input_layer_forward(feats.double(), rows_ref, active_ref.shape[0], 4)
    assert rel_err(out.features, ref) < 1e-6
    assert out.batch_size() == 2


def _gpu_rulebook_normal_form(scn, x, nbr, n_out, out_spatial=None):
    from sparseeventid_b200.scn import ops
    pairs = [p.cpu().numpy().astype(np.int64) for p in ops.rulebook_pairs(nbr, n_out)]
    return pairs


@pytest.mark.parametrize("filt", [(3, 3, 3), (1, 3, 3), (5, 5, 5), (1, 5, 5), (1, 1, 1), (3, 1, 5)])
def test_submanifold_rulebook_bit_exact(scn, filt):
    coords = blob_sites(700, (40, 30, 50), 3, seed=4)
    x = scn.InputLayer(3, [40, 30, 50])((torch.as_tensor(coords).cuda(), torch.ones(coords.shape[0], 1).cuda(), 3))
    md = x.metadata
    nbr = md.subm_table((40, 30, 50), filt)
    n = coords.shape[0]
    got = _gpu_rulebook_normal_form(scn, x, nbr, n)
    loc = x.get_spatial_locations().numpy()
    ref_rules = O.submanifold_rulebook(coords, filt)
    a = O.normalize_rulebook(got, loc, loc)
    b = O.normalize_rulebook(ref_rules, coords, coords)
    assert len(a) == len(b) == int(np.prod(filt))
    for k, (ra, rb) in enumerate(zip(a, b)):
        assert np.array_equal(ra, rb), f"offset {k}: rulebooks differ"
    # table-level invariants: identity centre, mirror symmetry, padding rows empty
    t = nbr.cpu().numpy()
    K = t.shape[0]
    assert np.array_equal(t[(K - 1) // 2, :n], np.arange(n))
    assert np.all(t[:, n:] == -1)
    for k in range(K):
        o = np.nonzero(t[k, :n] >= 0)[0]
        assert np.array_equal(t[K - 1 - k, t[k, o]], o)


def test_submanifold_rulebook_16bit_edges_and_empty(scn):
    edge = np.array([[0, 0, 65535, 0], [0, 1, 0, 0], [65535, 65535, 65535, 0], [0, 0, 0, 1], [0, 0, 1, 1]])
    x = scn.InputLayer(3, 65536)((torch.as_tensor(edge).cuda(), torch.ones(5, 1).cuda()))
    nbr = x.metadata.subm_table((65536,) * 3, (3, 3, 3))
    got = _gpu_rulebook_normal_form(scn, x, nbr, 5)
    ref = O.submanifold_rulebook(edge, (3, 3, 3))
    for ra, rb in zip(O.normalize_rulebook(got, edge, edge), O.normalize_rulebook(ref, edge, edge)):
        assert np.array_equal(ra, rb)
    assert sum(len(r) for r in got) == 7
    e = scn.InputLayer(3, 16)((torch.zeros(0, 4).long().cuda(), torch.zeros(0, 1).cuda(), 2))
    assert e.features.shape == (0, 1)
    y = scn.SubmanifoldConvolution(3, 1, 4, 3, True).cuda()(e)
    assert y.features.shape == (0, 4)


@pytest.mark.parametrize("filt,grid", [((2, 2, 2), (32, 24, 40)), ((1, 2, 2), (3, 48, 32))])
def test_strided_rulebook_bit_exact(scn, filt, grid):
    coords = blob_sites(600, grid, 2, seed=6)
    x = scn.InputLayer(3, list(grid))((torch.as_tensor(coords).cuda(), torch.ones(coords.shape[0], 1).cuda(), 2))
    md = x.metadata
    rule = md.strided_rule(grid, filt, filt)
    out_coords_ref, rules_ref, out_sp_ref = O.strided_rulebook(coords, filt, filt, grid)
    assert rule.out_spatial == out_sp_ref
    out_loc = md.coords(rule.out_spatial).cpu().numpy()
    # same set of output sites; the GPU numbers them in first-appearance order (SparseConvNet: created on first touch), the
    # oracle by ascending key -- the normal form below compares on coordinates
    assert np.array_equal(out_loc[np.lexsort(out_loc.T[::-1])], out_coords_ref[np.lexsort(out_coords_ref.T[::-1])])
    first, coarse = {}, coords.copy()
    coarse[:, :3] //= np.asarray(filt)
    for c in coarse:
        first.setdefault(tuple(int(v) for v in c), len(first))
    assert [first[tuple(int(v) for v in c)] for c in out_loc] == list(range(out_loc.shape[0]))   # first-appearance numbering
    got = _gpu_rulebook_normal_form(scn, x, rule.down, rule.n_out)
    a = O.normalize_rulebook(got, coords, out_loc)
    b = O.normalize_rulebook(rules_ref, coords, out_coords_ref)
    for k, (ra, rb) in enumerate(zip(a, b)):
        assert np.array_equal(ra, rb), f"offset {k}"
    # up table is the transpose of the down table
    got_up = _gpu_rulebook_normal_form(scn, x, rule.up, rule.n_in)
    for k in range(rule.K):
        d = set(map(tuple, got[k].tolist()))
        u = set((i, o) for o, i in got_up[k].tolist())
        assert d == u


# --------------------------------------------------------------------------- floating point layers


def run_pair(scn, mode, make_gpu, make_ref, coords, grid, batch, cin, seed=0, dense_out=False):
    scn.set_precision(mode)
    oscn.set_numerics(mode)
    try:
        torch.manual_seed(seed)
        ref_mods = make_ref()
        gpu_mods = make_gpu()
        for g, r in zip(gpu_mods, ref_mods):
            if len(list(r.state_dict())):
                copy_params(g, r, mode)
            g.cuda()
        c, f = make_input(coords, cin, seed + 1, mode)
        f_ref = f.clone().double().requires_grad_(True)
        for r in ref_mods:
            r.double()
        xr = oscn.InputLayer(3, list(grid))((c, f_ref, batch))
        f_gpu = f.clone().cuda().requires_grad_(True)
        xg = scn.InputLayer(3, list(grid))((c.cuda(), f_gpu, batch))
        if mode == "bf16":      # exercise the bf16-storage kernels: features enter the layer as bf16
            xg.features = xg.features.to(torch.bfloat16)
            xr.features = oscn.round_storage(xr.features)
        for r in ref_mods:
            xr = r(xr)
        for g in gpu_mods:
            xg = g(xg)
        yr = xr if dense_out else xr.features
        yg = xg if dense_out else xg.features
        perm = None
        if not dense_out:
            # a strided level is numbered in first-appearance order on the GPU and by ascending key in the oracle:
            # compare row r of the GPU with the oracle's row of the same site
            lg, lr = xg.get_spatial_locations().numpy(), xr.get_spatial_locations().numpy()
            if not np.array_equal(lg, lr):
                og, orr = np.lexsort(lg.T[::-1]), np.lexsort(lr.T[::-1])
                assert np.array_equal(lg[og], lr[orr]), "the two sides have different active sites"
                perm = np.empty_like(og)
                perm[og] = orr                                   # GPU row r <-> oracle row perm[r]
                perm = torch.as_tensor(perm)
        check(yg, yr if perm is None else yr[perm], mode, "forward")
        gen = torch.Generator().manual_seed(seed + 2)
        dout = q(torch.randn(yr.shape, generator=gen), mode)
        yr.backward(dout.double())
        yg.backward((dout if perm is None else dout[perm]).cuda().to(yg.dtype))
        check(f_gpu.grad, f_ref.grad, mode, "grad input")
        ref_norms = [float(p.grad.norm()) for r in ref_mods for p in r.parameters()]
        scale = max(ref_norms) if ref_norms else 1.0
        for g, r in zip(gpu_mods, ref_mods):
            for (n1, p1), (n2, p2) in zip(g.named_parameters(), r.named_parameters()):
                if float(p2.grad.norm()) < 1e-3 * scale:
                    # structurally zero gradient (a conv bias feeding a BatchNorm): only rounding noise on
                    # either side, so it is required to be small rather than relatively equal
                    assert float(p1.grad.float().norm()) < 1e-2 * scale, f"grad {n1} should be ~0"
                    continue
                check(p1.grad, p2.grad, mode, f"grad {n1}")
            for (n1, b1), (n2, b2) in zip(g.named_buffers(), r.named_buffers()):
                assert rel_err(b1, b2) < 1e-4, f"buffer {n1}"
    finally:
        scn.set_precision("bf16")
        oscn.set_numerics("fp32")


MODES = ["fp32", "mixed", "bf16"]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("cin,cout,filt", [(32, 32, (3, 3, 3)), (64, 96, (3, 3, 3)), (32, 64, (1, 3, 3)),
                                           (192, 128, (1, 1, 1)), (1, 32, (5, 5, 5)), (3, 5, (3, 3, 3)),
                                           (160, 160, (3, 3, 3))])
def test_submanifold_convolution(scn, mode, cin, cout, filt):
    grid, B = (24, 20, 28), 2
    coords = blob_sites(400, grid, B, seed=8)
    run_pair(scn, mode,
             lambda: [scn.SubmanifoldConvolution(3, cin, cout, list(filt), True)],
             lambda: [oscn.SubmanifoldConvolution(3, cin, cout, list(filt), True)],
             coords, grid, B, cin)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("cin,cout,filt", [(32, 64, (2, 2, 2)), (64, 96, (1, 2, 2)), (5, 7, (2, 2, 2))])
def test_strided_convolution(scn, mode, cin, cout, filt):
    grid, B = (24, 20, 28), 2
    coords = blob_sites(400, grid, B, seed=9)
    run_pair(scn, mode,
             lambda: [scn.Convolution(3, cin, cout, list(filt), list(filt), False)],
             lambda: [oscn.Convolution(3, cin, cout, list(filt), list(filt), False)],
             coords, grid, B, cin)


@pytest.mark.parametrize("mode", MODES)
def test_down_then_deconvolution(scn, mode):
    grid, B = (16, 16, 16), 2
    coords = blob_sites(300, grid, B, seed=10)
    run_pair(scn, mode,
             lambda: [scn.Convolution(3, 32, 64, 2, 2, False), scn.Deconvolution(3, 64, 32, 2, 2, True)],
             lambda: [oscn.Convolution(3, 32, 64, 2, 2, False), oscn.Deconvolution(3, 64, 32, 2, 2, True)],
             coords, grid, B, 32)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("c,leak", [(32, 1), (96, 0), (160, 0.333), (5, 1), (12, 0.333)])
def test_batchnorm_train(scn, mode, c, leak):
    grid, B = (16, 16, 16), 2
    coords = random_sites(777, grid, B, seed=11)
    run_pair(scn, mode,
             lambda: [scn.BatchNormalization(c, leakiness=leak)],
             lambda: [oscn.BatchNormalization(c, leakiness=leak)],
             coords, grid, B, c)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_batchnorm_eval(scn, mode):
    grid, B, c = (16, 16, 16), 2, 64
    coords = random_sites(500, grid, B, seed=12)

    def mk(mod):
        def f():
            m = mod.BatchNormalization(c, leakiness=0.333)
            m.running_mean.normal_()
            m.running_var.uniform_(0.5, 2.0)
            m.eval()
            return [m]
        return f
    run_pair(scn, mode, mk(scn), mk(oscn), coords, grid, B, c)


@pytest.mark.parametrize("mode", MODES)
def test_residual_block_chain(scn, mode):
    """conv -> BN -> LeakyReLU -> conv -> BN -> AddTable -> LeakyReLU (reference ResidualBlock,
    src/networks/sparse_building_blocks.py:61-100), then SparseToDense."""
    grid, B, c = (16, 12, 20), 2, 32
    coords = blob_sites(350, grid, B, seed=13)

    class Res(torch.nn.Module):
        def __init__(self, m):
            super().__init__()
            self.c1 = m.SubmanifoldConvolution(3, c, c, 3, True)
            self.n1 = m.BatchNormalization(c)
            self.a1 = m.LeakyReLU()
            self.c2 = m.SubmanifoldConvolution(3, c, c, 3, True)
            self.n2 = m.BatchNormalization(c)
            self.add = m.AddTable()
            self.relu = m.LeakyReLU()
            self.dense = m.SparseToDense(3, c)

        def forward(self, x):
            out = self.a1(self.n1(self.c1(x)))
            out = self.n2(self.c2(out))
            out = self.relu(self.add([out, x]))
            return self.dense(out)

    run_pair(scn, mode, lambda: [Res(scn)], lambda: [Res(oscn)], coords, grid, B, c, dense_out=True)


def test_output_layer_roundtrip(scn):
    scn.set_precision("fp32")
    try:
        coords = random_sites(300, (10, 10, 10), 2, seed=14, dup=40)
        feats = torch.randn(coords.shape[0], 4)
        f_gpu = feats.clone().cuda().requires_grad_(True)
        x = scn.InputLayer(3, 10)((torch.as_tensor(coords).cuda(), f_gpu, 2))
        y = scn.OutputLayer(3)(x)
        rows, active = O.input_layer_rules(coords)
        ref_in = O.input_layer_forward(feats.double(), rows, active.shape[0], 3)
        ref = O.output_layer_forward(ref_in, rows)
        assert rel_err(y, ref) < 1e-6
        dout = torch.randn(y.shape)
        y.backward(dout.cuda())
        g = O.input_layer_backward(O.output_layer_backward(dout.double(), rows, active.shape[0]), rows)
        assert rel_err(f_gpu.grad, g) < 1e-6
    finally:
        scn.set_precision("bf16")


def test_no_cpu_fallback(scn):
    with pytest.raises(RuntimeError):
        scn.InputLayer(3, 8)((torch.zeros(4, 4).long(), torch.zeros(4, 1)))


def test_large_property_checks(scn):
    """Size-independent properties at a BASELINE-sized level (5e5 sites): identity centre, mirror symmetry,
    pair count = N for filter==stride, linearity of the conv in its input."""
    from sparseeventid_b200 import synthetic
    from sparseeventid_b200.data_transforms import larcvsparse_to_scnsparse_3d
    arr = synthetic.larcv_batch_3d(16, seed=99)
    c, f, b = larcvsparse_to_scnsparse_3d(arr)
    x = scn.InputLayer(3, list(synthetic.GRID_3D))((torch.as_tensor(c).cuda(), torch.as_tensor(f).cuda(), b))
    n = x.features.shape[0]
    assert n == c.shape[0]
    nbr = x.metadata.subm_table(synthetic.GRID_3D, (3, 3, 3))
    assert torch.equal(nbr[13, :n], torch.arange(n, dtype=torch.int32, device="cuda"))
    for k in (0, 5, 12):
        o = torch.nonzero(nbr[k, :n] >= 0)[:, 0]
        assert torch.equal(nbr[26 - k, nbr[k, o].long()].long(), o)
    rule = x.metadata.strided_rule(synthetic.GRID_3D, (2, 2, 2), (2, 2, 2))
    assert int((rule.down >= 0).sum()) == n and int((rule.up >= 0).sum()) == n
    keys = x.metadata.levels[rule.out_spatial].keys
    assert int(torch.unique(keys).shape[0]) == int(keys.shape[0]) == rule.n_out
    scn.set_precision("bf16")
    conv = scn.SubmanifoldConvolution(3, 32, 32, 3, False).cuda()
    a = torch.randn(n, 32, device="cuda").bfloat16()
    ya = conv(scn.SparseConvNetTensor(a, x.metadata, x.spatial_size)).features.float()
    y2 = conv(scn.SparseConvNetTensor((2 * a), x.metadata, x.spatial_size)).features.float()
    assert rel_l2(y2, 2 * ya) < 1e-6          # scaling by 2 is exact in bf16


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_direct_gradient_accumulation_matches_autograd(scn, mode):
    """trainer.FlatGradArena lets the kernels accumulate parameter gradients in place (no dW temporaries, no
    AccumulateGrad adds).  The gradients must equal the plain autograd path's, and a second backward must add."""
    from sparseeventid_b200.trainer import FlatGradArena
    scn.set_precision(mode)
    coords = blob_sites(300, (24, 24, 24), 3, seed=5)
    c = 32

    def net():
        torch.manual_seed(3)
        return torch.nn.Sequential(
            scn.SubmanifoldConvolution(3, 1, c, 3, True), scn.BatchNormalization(c), scn.LeakyReLU(),
            scn.SubmanifoldConvolution(3, c, c, 3, True), scn.BatchNormLeakyReLU(c),
            scn.Convolution(3, c, 2 * c, 2, 2, False), scn.SparseToDense(3, 2 * c)).cuda()

    feats = torch.randn(coords.shape[0], 1).cuda()
    ct = torch.as_tensor(coords).cuda()
    a, b = net(), net()
    arena = FlatGradArena(list(b.parameters()))
    assert all(getattr(p, "_scn_direct_grad", False) for p in b.parameters())
    for rounds in (1, 2):
        for m in (a, b):
            x = scn.InputLayer(3, [24, 24, 24])((ct, feats, 3))
            m(x).float().square().sum().backward()
        for (n, pa), (_, pb) in zip(a.named_parameters(), b.named_parameters()):
            ga, gb = pa.grad.float(), pb.grad.float()
            scale = float(ga.abs().max()) + 1e-12
            # wgrad uses fp32 atomics: summation order differs between runs, values agree to fp32 round-off
            assert float((ga - gb).abs().max()) <= 2e-4 * scale + 1e-6, (mode, rounds, n)
    assert arena.flat.abs().sum() > 0
    scn.set_precision("bf16")


@pytest.mark.parametrize("dataset", ["dune3d", "dune2d"])
def test_device_input_transform_matches_host_transform(scn, dataset):
    """SURVEY 8f-2: the device-side larcv -> SCN tuple (order-preserving compaction of the -999-padded batch filler
    array) gives the same rows, in the same order, as the reference's numpy transform; InputLayer row numbering and
    features downstream are therefore identical."""
    from sparseeventid_b200 import data_transforms as T
    from sparseeventid_b200 import synthetic
    if dataset == "dune3d":
        arr = synthetic.larcv_batch_3d(5, seed=11)
        arr[2, 0, :, 3] = T.PAD_VALUE                  # an empty event
        ch, fh, bh = T.larcvsparse_to_scnsparse_3d(arr)
        cg, fg, bg = T.larcvsparse_to_scnsparse_3d_gpu(torch.from_numpy(arr).cuda())
        grid = list(synthetic.GRID_3D)
    else:
        arr = synthetic.larcv_batch_2d(4, seed=12)
        ch, fh, bh = T.larcvsparse_to_scnsparse_2d(arr)
        cg, fg, bg = T.larcvsparse_to_scnsparse_2d_gpu(torch.from_numpy(arr).cuda())
        grid = list(synthetic.GRID_2D)
    assert bg == bh
    assert np.array_equal(cg.cpu().numpy().astype(np.int64), np.asarray(ch).astype(np.int64))
    assert np.array_equal(fg.cpu().numpy(), np.asarray(fh, dtype=np.float32))
    xa = scn.InputLayer(3, grid)((torch.as_tensor(np.asarray(ch)).cuda(), torch.as_tensor(np.asarray(fh)).float().cuda(), bh))
    xb = scn.InputLayer(3, grid)((cg, fg, bg))
    assert torch.equal(xa.metadata.row_of_input, xb.metadata.row_of_input)
    assert torch.equal(xa.features, xb.features)


def test_rulebook_prefetch_gives_identical_results(scn):
    """scn.prefetch builds InputLayer rules + the recorded rulebook plan for the NEXT batch on the rulebook stream;
    a forward/backward that adopts them must be bit-identical to one that builds them itself, and a different
    tensor object must never pick them up."""
    from sparseeventid_b200.scn import core
    scn.set_precision("bf16")
    torch.manual_seed(1)
    c = 32
    net = torch.nn.Sequential(
        scn.SubmanifoldConvolution(3, 1, c, 3, True), scn.BatchNormLeakyReLU(c),
        scn.Convolution(3, c, 2 * c, 2, 2, False), scn.SubmanifoldConvolution(3, 2 * c, 2 * c, 3, False),
        scn.SparseToDense(3, 2 * c)).cuda()
    il = scn.InputLayer(3, [24, 24, 24])

    def run(coords, feats):
        net.zero_grad()
        y = net(il((coords, feats, 3)))
        y.float().square().sum().backward()
        return y.detach().clone(), [p.grad.clone() for p in net.parameters()]

    a = torch.as_tensor(blob_sites(300, (24, 24, 24), 3, seed=5)).cuda()
    b = torch.as_tensor(blob_sites(280, (24, 24, 24), 3, seed=6)).cuda()
    fa, fb = torch.randn(a.shape[0], 1).cuda(), torch.randn(b.shape[0], 1).cuda()
    run(a, fa)                                           # records the plan
    want_y, want_g = run(b, fb)
    run(a, fa)
    md = core.prefetch(b, 3, [24, 24, 24], il._last_plan)
    assert md is not None and len(md.subm) == 2 and len(md.strided) == 1
    assert core.take_prefetched(b.clone(), 3, (24, 24, 24)) is None       # another tensor object: not adopted
    core.prefetch(b, 3, [24, 24, 24], il._last_plan)
    got_y, got_g = run(b, fb)
    assert not core._prefetched                                            # it was consumed
    assert torch.equal(got_y, want_y)
    for g, w in zip(got_g, want_g):
        scale = float(w.abs().max()) + 1e-12
        assert float((g - w).abs().max()) <= 2e-4 * scale                  # wgrad atomics: fp32 summation order only


@pytest.mark.parametrize("fused", [True, False])
def test_forward_follows_optimizer_updates(scn, fused):
    """Regression: the re-laid weight images must track the parameters through optimizer steps.  Fused Adam updates
    parameters WITHOUT bumping Tensor._version, so a version-keyed image cache silently froze the forward weights."""
    scn.set_precision("bf16")
    torch.manual_seed(2)
    c = 32
    net = torch.nn.Sequential(scn.SubmanifoldConvolution(3, 1, c, 3, True), scn.BatchNormLeakyReLU(c),
                              scn.SubmanifoldConvolution(3, c, c, 3, True), scn.SparseToDense(3, c)).cuda()
    opt = torch.optim.Adam(net.parameters(), lr=5e-2, fused=fused)
    coords = torch.as_tensor(blob_sites(200, (16, 16, 16), 2, seed=9)).cuda()
    feats = torch.randn(coords.shape[0], 1).cuda()
    il = scn.InputLayer(3, [16, 16, 16])
    y0 = net(il((coords, feats, 2))).detach().clone()
    for _ in range(3):
        opt.zero_grad()
        net(il((coords, feats, 2))).float().square().mean().backward()
        opt.step()
    net.eval()
    y_trained = net(il((coords, feats, 2))).detach()
    fresh = torch.nn.Sequential(scn.SubmanifoldConvolution(3, 1, c, 3, True), scn.BatchNormLeakyReLU(c),
                                scn.SubmanifoldConvolution(3, c, c, 3, True), scn.SparseToDense(3, c)).cuda().eval()
    fresh.load_state_dict(net.state_dict())
    y_fresh = fresh(il((coords, feats, 2))).detach()
    assert torch.equal(y_trained, y_fresh)               # same parameters -> same output, whatever the history
    assert float((y_trained - y0).abs().max()) > 1e-3    # and the three steps did change the network
