"""bench.py --dump-outputs (CPU, oracle modules, a small encoder): the timed loop starts from the trainer's initial state
whatever ran before it, so the dumped results of its last step are a function of the arguments alone."""
import numpy as np
import torch

CFG = dict(depth=2, n_initial_filters=8, n_output_filters=8, blocks_per_layer=1)


def _trainer():
    from oracle import sparseconvnet_oracle as oscn
    from sparseeventid_b200 import networks
    from sparseeventid_b200.trainer import Trainer
    oscn.set_numerics("fp32")
    return Trainer(oscn, "dune3d", device="cpu", cfg=networks.EncoderConfig(**CFG), seed=0)


def _batches():
    out = []
    for seed in (5, 6):
        rng = np.random.default_rng(seed)
        rows = []
        for b in range(2):
            pts = np.unique(rng.integers(8, 24, size=(60, 3)), axis=0)
            rows.append(np.concatenate([pts, np.full((pts.shape[0], 1), b)], 1))
        coords = np.concatenate(rows, 0).astype(np.int64)
        feats = rng.normal(size=(coords.shape[0], 1)).astype(np.float32)
        labels = {k: torch.as_tensor(rng.integers(0, 2, size=2)) for k in
                  ("labelneutID", "labelprotID", "labelnpiID", "labelcpiID")}
        out.append(((torch.as_tensor(coords), torch.as_tensor(feats), 2), labels))
    return out


def _run(trainer, batches, steps):
    loss = None
    for i in range(steps):
        batch, labels = batches[i % len(batches)]
        loss = trainer.step(batch, labels).detach()
    return loss


def test_reset_then_steps_reproduce_a_fresh_trainer():
    import bench
    batches = _batches()

    fresh = _trainer()
    torch.manual_seed(0)
    want = bench.step_outputs(fresh, _run(fresh, batches, 3))

    tr = _trainer()
    reset = bench.training_state_reset(tr)
    _run(tr, batches, 5)                                   # set-up steps of any number: Adam moments, lr schedule, BN stats
    reset()
    got = bench.step_outputs(tr, _run(tr, batches, 3))

    assert set(got) == set(want) == {"loss", "grad_sample", "param_sample", "bn_running_stats"}
    for k in want:
        assert got[k].dtype == np.float32 and got[k].shape == want[k].shape, k
        assert np.array_equal(got[k], want[k]), k
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
