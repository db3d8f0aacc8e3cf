"""Legacy reference networks (SURVEY §8 a11: src/networks/torch/sparseresnet3d.py, src/networks/torch/sparseresnet.py)
replayed against the committed fixtures tests/golden/legacy*.npz, which tests/golden/make_golden_legacy.py generated
by importing the reference files VERBATIM on the oracle shim.

  * CPU: the repo's mirror (sparseeventid_b200/legacy_networks.py) on the oracle reproduces the fixture.
  * GPU: the mirror on the product kernels, "fp32" mode within 2e-3 of the fixture (north-star bar); "bf16" mode
    within the deep-network bf16 noise floor (see tests/test_golden_network.py for why that is not 2e-3).
"""
import os

import numpy as np
import pytest
import torch

from helpers import LEGACY_CASES, init_deterministic, legacy_batch
from oracle import sparseconvnet_oracle as oscn
from sparseeventid_b200 import legacy_networks as legacy
from sparseeventid_b200 import networks, synthetic

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL = 2e-3


def run(scn_mod, case, device):
    spec = LEGACY_CASES[case]
    cls = legacy.LegacyResNet3D if spec["kind"] == "3d" else legacy.LegacyResNet2D
    torch.manual_seed(0)
    model = cls(scn_mod, legacy.LEGACY_OUTPUT_SHAPE, legacy.LegacyNetworkConfig(**spec["cfg"]))
    init_deterministic(model)
    model.to(device).train()
    coords, feats, bs = legacy_batch(case)
    labels = {k: torch.as_tensor(v).to(device) for k, v in synthetic.make_labels(2, seed=11).items()}
    logits = model((torch.as_tensor(coords).to(device), torch.as_tensor(feats).to(device), bs))
    loss = networks.focal_loss(labels, logits)
    loss.backward()
    return model, logits, loss


def errors(model, logits, loss, want):
    def rel(a, b):
        a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
        return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-6))
    errs = {"loss": rel(float(loss), want["loss"])}
    for k, v in logits.items():
        errs["logits_" + k] = rel(v.detach().double().cpu().numpy(), want["logits_" + k])
    gn = np.asarray([float(p.grad.double().norm()) for _, p in model.named_parameters()])
    wn = np.asarray(want["grad_norms"], dtype=np.float64)
    big = wn > 1e-3 * wn.max()
    errs["grad_norms"] = float((np.abs(gn - wn)[big] / wn[big]).max())
    return errs


@pytest.mark.parametrize("case", sorted(LEGACY_CASES))
def test_oracle_mirror_reproduces_legacy_fixture(case):
    want = np.load(os.path.join(GOLDEN, case + ".npz"))
    oscn.set_numerics("fp32")
    # the fixtures were recorded with 8 intra-op threads: the oracle's fp32 gradient sums are split by thread, so the
    # replay reproduces them bit for bit only with the same count, whatever the host's core count
    threads = torch.get_num_threads()
    torch.set_num_threads(8)
    try:
        model, logits, loss = run(oscn, case, "cpu")
    finally:
        torch.set_num_threads(threads)
    assert [n for n, _ in model.named_parameters()] == [str(n) for n in want["param_names"]]
    assert sum(p.numel() for p in model.parameters()) == int(want["n_params"][0])
    errs = errors(model, logits, loss, want)
    assert max(errs.values()) <= 1e-9, errs


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("case", sorted(LEGACY_CASES))
def test_gpu_legacy_network_matches_fixture(case, mode):
    """fp32 mode: within 2e-3 of the fixture (truth).  bf16 mode: no further from truth than 1.5x the distance of the
    ORACLE run under the same stated precision (+ a floor of 2e-3; 1e-2 for the worst gradient norm): the bar a wrong
    kernel fails and a kernel that merely rounds differently passes (see tests/test_golden_network.py)."""
    import sparseconvnet as scn
    want = np.load(os.path.join(GOLDEN, case + ".npz"))
    scn.set_precision(mode)
    try:
        model, logits, loss = run(scn, case, "cuda")
        errs = errors(model, logits, loss, want)
        print(case, mode, {k: f"{v:.2e}" for k, v in errs.items()})
        if mode == "fp32":
            assert max(errs.values()) <= TOL, errs
        else:
            oscn.set_numerics(mode)
            try:
                o_model, o_logits, o_loss = run(oscn, case, "cpu")
                o_errs = errors(o_model, o_logits, o_loss, want)
            finally:
                oscn.set_numerics("fp32")
            print(case, "oracle[" + mode + "]", {k: f"{v:.2e}" for k, v in o_errs.items()})
            for k, e in errs.items():
                floor = 1e-2 if k == "grad_norms" else 2e-3
                assert e <= 1.5 * o_errs[k] + floor, (k, e, o_errs[k])
    finally:
        scn.set_precision("bf16")
