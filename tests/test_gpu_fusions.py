"""GPU tests of the fused / batched forms that sit between the per-layer kernels and the training step:

  * scn_bn_backward_colsum: the column sums of dx produced by the BatchNorm backward's apply pass equal the sums of the
    dx it stored (they replace the bias-gradient pass of the convolution in front of the BatchNorm, SCN's Convolution
    backward as reached from src/networks/sparse_building_blocks.py:29-39),
  * conv -> BatchNorm: the bias gradient the convolution ends up with equals the column sums of its grad_output,
  * scn_conv_prep_weights_batched: every weight image built by the one-launch form is byte-identical to the image the
    per-module call builds (forward and dgrad images, every channel configuration of the default network).
"""
import copy

import pytest
import torch

from helpers import blob_sites

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def scn():
    import sparseconvnet as s
    return s


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("n,c", [(1, 32), (64, 192), (777, 96), (3000, 160), (5000, 32), (20000, 64), (9000, 128)])
def test_bn_backward_colsum_is_the_sum_of_the_stored_dx(scn, n, c, dtype):
    from sparseeventid_b200.scn import ops
    g = torch.Generator(device="cuda").manual_seed(n + c)
    x = (torch.randn(n, c, device="cuda", generator=g) * 2 + 0.5).to(dtype)
    d = torch.randn(n, c, device="cuda", generator=g).to(dtype)
    gamma = torch.rand(c, device="cuda", generator=g) + 0.5
    beta = torch.randn(c, device="cuda", generator=g) * 0.1
    rm, rv = torch.zeros(c, device="cuda"), torch.ones(c, device="cuda")
    out, stats = ops.bn_forward(x, gamma, beta, rm, rv, True, 1e-4, 0.9, 0.333)
    dx, dg, db, colsum = ops.bn_backward(x, d, gamma, beta, stats, True, 0.333, want_colsum=True)
    dx2, dg2, db2 = ops.bn_backward(x, d, gamma, beta, stats, True, 0.333)
    assert torch.equal(dx, dx2) and torch.allclose(dg, dg2, rtol=1e-5, atol=1e-5) and torch.allclose(db, db2, rtol=1e-5, atol=1e-5)
    want = dx.double().sum(0)
    scale = float(dx.double().abs().sum(0).max()) + 1e-12
    assert float((colsum.double() - want).abs().max()) <= 2e-6 * scale + 1e-7, (n, c, dtype)
    # and dx itself against the textbook formula in float64
    xd, dd = x.double(), d.double()
    mean, var = xd.mean(0), xd.var(0, unbiased=False)
    xh = (xd - mean) / torch.sqrt(var + 1e-4)
    y = xh * gamma.double() + beta.double()
    dl = torch.where(y > 0, dd, dd * 0.333)
    ref = gamma.double() / torch.sqrt(var + 1e-4) * (dl - dl.mean(0) - xh * (dl * xh).mean(0))
    err = float((dx.double() - ref).norm() / (ref.norm() + 1e-30))
    if n > 1:
        assert err <= (5e-3 if dtype == torch.bfloat16 else 2e-5), (n, c, dtype, err)


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_conv_bias_gradient_through_batchnorm(scn, mode):
    scn.set_precision(mode)
    try:
        torch.manual_seed(4)
        c = 32
        conv = scn.SubmanifoldConvolution(3, c, c, 3, True).cuda()
        bn = scn.BatchNormLeakyReLU(c).cuda()
        tail = scn.SubmanifoldConvolution(3, c, c, 3, True).cuda()
        coords = torch.as_tensor(blob_sites(400, (20, 20, 20), 3, seed=21)).cuda()
        feats = torch.randn(coords.shape[0], c).cuda()
        x = scn.InputLayer(3, [20, 20, 20])((coords, feats, 3))
        y = conv(x)
        kept = []
        y.features.register_hook(lambda gr: kept.append(gr.detach().clone()))
        z = tail(bn(y))
        z.features.float().square().sum().backward()
        dout = kept[0].double()
        want = dout.sum(0)
        scale = float(dout.abs().sum(0).max()) + 1e-12
        assert float((conv.bias.grad.double() - want).abs().max()) <= 2e-6 * scale + 1e-7
        # the tail convolution's grad_output does not come from a BatchNorm: its own column-sum pass
        assert conv.bias.grad.shape == tail.bias.grad.shape and float(tail.bias.grad.abs().max()) > 0
    finally:
        scn.set_precision("fp32")


def test_batched_weight_images_equal_per_module_images(scn):
    from sparseeventid_b200 import _lib as L
    from sparseeventid_b200.scn import config, functional as F, ops
    scn.set_precision("bf16")
    try:
        torch.manual_seed(7)
        mods = [scn.SubmanifoldConvolution(3, 32, 32, 3, True), scn.SubmanifoldConvolution(3, 64, 64, 3, False),
                scn.SubmanifoldConvolution(3, 96, 96, 3, True), scn.SubmanifoldConvolution(3, 160, 160, 3, True),
                scn.SubmanifoldConvolution(3, 192, 128, 1, True), scn.Convolution(3, 32, 64, 2, 2, False),
                scn.Convolution(3, 64, 96, 2, 2, True), scn.Deconvolution(3, 128, 96, 2, 2, False),
                scn.Convolution(3, 160, 192, 2, 2, False)]
        mods = [m.cuda() for m in mods]
        built = F.prepare_weight_images(mods)
        assert built == 2 * len(mods)
        prec, fdt = config.precision_code(), config.feature_dtype()
        for m in mods:
            w = m.weight
            K, cin, cout = w.shape[0], w.shape[-2], w.shape[-1]
            ws = m.workspace(K, cin, cout, prec, fdt, w.device)
            w3 = w.detach().reshape(K, cin, cout).contiguous()
            fwd = ops.prep_weights(w3, False, False, prec, fdt)
            bwd = ops.prep_weights(w3, True, m.mirror_dgrad, prec, fdt)
            assert torch.equal(ws.fwd[: fwd.numel()], fwd), (type(m).__name__, cin, cout, "forward image")
            assert torch.equal(ws.bwd[: bwd.numel()], bwd), (type(m).__name__, cin, cout, "dgrad image")
        F.release_weight_images()
    finally:
        scn.set_precision("fp32")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_batchnorm_calls_with_changing_channel_counts(scn, dtype):
    """The two-launch BatchNorm alternates between two sets of accumulators and each call's apply kernel clears the set
    the NEXT call will use -- as far as the PREVIOUS call wrote it.  A sequence whose channel count goes up and down
    (the backward pass of the encoder does) must give the textbook result at every call."""
    from sparseeventid_b200.scn import ops
    g = torch.Generator(device="cuda").manual_seed(5)
    for i, (n, c) in enumerate([(3000, 160), (5000, 32), (900, 192), (4000, 64), (7000, 32), (2500, 128), (6000, 96), (64, 32)]):
        x = (torch.randn(n, c, device="cuda", generator=g) * 1.5 - 0.3).to(dtype)
        d = torch.randn(n, c, device="cuda", generator=g).to(dtype)
        gamma = torch.rand(c, device="cuda", generator=g) + 0.5
        beta = torch.randn(c, device="cuda", generator=g) * 0.1
        rm, rv = torch.zeros(c, device="cuda"), torch.ones(c, device="cuda")
        out, stats = ops.bn_forward(x, gamma, beta, rm, rv, True, 1e-4, 0.9, 0.333)
        xd = x.double()
        mean, var = xd.mean(0), xd.var(0, unbiased=False)
        xh = (xd - mean) / torch.sqrt(var + 1e-4)
        y = xh * gamma.double() + beta.double()
        ref = torch.where(y > 0, y, y * 0.333)
        tol = 8e-3 if dtype == torch.bfloat16 else 2e-5
        assert float((out.double() - ref).norm() / ref.norm()) <= tol, ("forward", i, n, c)
        assert float((stats[0].double() - mean).abs().max()) <= 1e-5 * float(mean.abs().max() + 1), ("mean", i, n, c)
        assert float((stats[1].double() * torch.sqrt(var + 1e-4) - 1).abs().max()) <= 1e-5, ("invstd", i, n, c)
        if i % 2 == 0:                                   # odd / even mixes forward and backward calls on the two sets
            dx, dg, db = ops.bn_backward(x, d, gamma, beta, stats, True, 0.333)
            dl = torch.where(y > 0, d.double(), d.double() * 0.333)
            dref = gamma.double() / torch.sqrt(var + 1e-4) * (dl - dl.mean(0) - xh * (dl * xh).mean(0))
            assert float((dx.double() - dref).norm() / dref.norm()) <= tol, ("backward", i, n, c)
            assert float((db.double() - dl.sum(0)).abs().max()) <= 1e-4 * float(dl.abs().sum(0).max()), ("dbeta", i, n, c)


def test_second_consumer_of_a_fused_batchnorm_does_not_update_running_statistics_again(scn):
    """BatchNormalization -> LeakyReLU runs as one kernel; a second reader of the BatchNorm's own output makes the layer
    run once more as written.  The running statistics must have been updated exactly once (SCN: one module call)."""
    scn.set_precision("fp32")
    torch.manual_seed(1)
    c = 32
    coords = torch.as_tensor(blob_sites(300, (16, 16, 16), 2, seed=3)).cuda()
    feats = (torch.randn(coords.shape[0], c) * 2 + 1).cuda()
    x = scn.InputLayer(3, [16, 16, 16])((coords, feats, 2))
    bn = scn.BatchNormalization(c).cuda().train()
    y = bn(x)
    z = scn.LeakyReLU(0.333)(y)
    fused = z.features
    plain = y.features                        # second consumer: the BatchNorm as written
    want_mean = 0.1 * x.features.float().mean(0)
    assert torch.allclose(bn.running_mean, want_mean, rtol=1e-5, atol=1e-6)
    assert torch.allclose(torch.where(plain > 0, plain, plain * 0.333), fused, rtol=1e-5, atol=1e-6)


def test_graphed_head_and_loss_match_eager(scn):
    """Trainer replays the dense heads + focal loss as CUDA graphs; with dropout off (head.eval()) loss, gradients and
    the parameters after two optimizer steps must equal the eager path's."""
    import numpy as np
    from sparseeventid_b200 import synthetic
    from sparseeventid_b200.data_transforms import larcvsparse_to_scnsparse_3d
    from sparseeventid_b200.trainer import Trainer
    scn.set_precision("bf16")
    try:
        c, f, bs = larcvsparse_to_scnsparse_3d(synthetic.larcv_batch_3d(4, seed=77))
        batch = (torch.from_numpy(np.ascontiguousarray(c, dtype=np.float64)).cuda(),
                 torch.from_numpy(np.ascontiguousarray(f, dtype=np.float32)).cuda(), bs)
        labels = {k: torch.from_numpy(v).cuda() for k, v in synthetic.make_labels(4, seed=77).items()}
        trainers = []
        for graph in (True, False):
            tr = Trainer(scn, "dune3d", device="cuda", seed=0)
            tr.graph_head = graph
            tr.model.head.eval()
            trainers.append(tr)
        tg, te = trainers
        la, lb = [], []
        for _ in range(2):
            # the encoder's gradients carry order-dependent sums (bounded below), and Adam turns their last bits into
            # parameter differences of the order of the learning rate: the eager trainer starts every step from the
            # graphed one's state, so that the head's parameters compare the head alone
            te.model.load_state_dict(tg.model.state_dict())
            te.opt.load_state_dict(copy.deepcopy(tg.opt.state_dict()))     # its own moments, not views of tg's
            la.append(float(tg.step(batch, labels)))
            lb.append(float(te.step(batch, labels)))
        assert bool(tg._head_graphs) and not te._head_graphs
        (pa, ga), (pb, gb) = [([p.detach().clone() for p in tr.model.head.parameters()], tr.arena.flat.detach().clone())
                              for tr in trainers]
        assert np.allclose(la, lb, rtol=1e-5, atol=1e-7), (la, lb)
        for x, y in zip(pa, pb):
            assert torch.allclose(x, y, rtol=1e-4, atol=1e-6)
        scale = float(gb.abs().max())
        assert float((ga - gb).abs().max()) <= 2e-3 * scale          # encoder gradients: bf16 kernels with atomics-free but order-dependent sums
    finally:
        scn.set_precision("fp32")


@pytest.mark.parametrize("n,K", [(5000, 125), (333, 125), (2048, 25), (17, 9)])
def test_stem_tensor_core_kernels(scn, n, K):
    """csrc/stem_tc.cu: the one-input-channel stem as dense GEMMs over the neighbour table (bf16 hi/lo splits of the fp32
    input and weights, fp32 accumulation) against float64: the forward within bf16 output rounding, the weight gradient
    within 1e-5 of its scale."""
    from sparseeventid_b200 import _lib as L
    from sparseeventid_b200.scn import ops
    g = torch.Generator(device="cuda").manual_seed(n * 7 + K)
    n_pad = ops.pad128(n)
    nbr = torch.full((K, n_pad), -1, dtype=torch.int32, device="cuda")
    live = torch.rand(K, n, device="cuda", generator=g) < 0.16
    idx = torch.randint(0, n, (K, n), device="cuda", generator=g, dtype=torch.int32)
    nbr[:, :n] = torch.where(live, idx, torch.full_like(idx, -1))
    nbr[K // 2, :n] = torch.arange(n, device="cuda", dtype=torch.int32)
    x = torch.randn(n, 1, device="cuda", generator=g) * 3 + 1
    w = torch.randn(K, 1, 32, device="cuda", generator=g) * 0.2
    bias = torch.randn(32, device="cuda", generator=g)
    dout = torch.randn(n, 32, device="cuda", generator=g).bfloat16()
    prec = L.PREC_BF16
    assert ops.conv_path(K, 1, 32, prec, torch.bfloat16) == 0            # not a tcgen05 shape: the stem path decides
    bp = ops.prep_weights(w.reshape(K, 1, 32).contiguous(), False, False, prec, torch.bfloat16)
    out = ops.conv_forward(x, nbr, n, 1, 32, bp, bias, prec, torch.bfloat16)
    j = nbr[:, :n].long()
    xg = torch.where(j >= 0, x.double()[:, 0][j.clamp_min(0)], torch.zeros((), dtype=torch.float64, device="cuda"))   # [K, n]
    ref = bias.double()[None, :] + torch.einsum("kn,kc->nc", xg, w.double()[:, 0, :])
    err = float((out.double() - ref).abs().max() / ref.abs().max())
    assert err <= 6e-3, ("forward", n, K, err)                           # bf16 output: half an ulp = 2^-9
    assert float((out.double() - ref).norm() / ref.norm()) <= 3e-3
    dw = ops.conv_wgrad(x, dout, nbr, n, 1, 32, prec)
    dref = torch.einsum("kn,nc->kc", xg, dout.double())
    derr = float((dw.double()[:, 0, :] - dref).abs().max() / dref.abs().max())
    assert derr <= 1e-5, ("wgrad", n, K, derr)
