"""Parity at the BENCHMARKED configuration (bench.py's first batch: 64 synthetic dune3d events, ~5e5 active sites).

  * rulebooks: the neighbour tables of all six levels (3^3), the 5^3 stem and the five stride-2 maps are compared
    BIT-EXACT with the oracle's rulebooks.  Level-0 rows are the input order on both sides (checked); deeper levels are
    numbered in first-appearance order on the GPU and by ascending key in the oracle, so the GPU tables are translated
    row by row through the coordinate-matched permutation before the comparison: the table form nbr[k][out] = in,
    in one numbering, IS the order-normalised rulebook.
  * one training step (forward, focal loss, backward) of the default encoder + heads on that batch:
      - "fp32" mode against the oracle in float64 ("truth"): loss / logits / encoder output / gradient norms within
        2e-3 relative (BASELINE.json north_star bar); element-wise, a gradient tensor may differ from truth by 2e-2
        in relative L2 with cosine >= 0.9999 (measured on B200: median 3.6e-3, max 7.9e-3 -- the fp32 ORACLE is just
        as far from float64: the network amplifies fp32 rounding ~1e4-fold at this initialisation);
      - "bf16" mode (what bench.py times: bf16 storage, tcgen05 kernels on multi-group, double-buffered, 148-CTA
        launches): loss / logits within 2e-3 of truth.  The network amplifies a rounding error ~1e4-fold at this
        initialisation (fp32 vs fp64 gradients already differ by up to ~1.5e-3), so NO bf16 pipeline can hold the
        gradients to 2e-3 end to end; the falsifiable bar is relative to truth: the GPU's distance from truth may not
        exceed 1.5x the distance of the oracle run under the same stated precision (+ a floor of 5e-2 in relative L2:
        a wrong kernel is off by O(1)), per tensor.
"""
import numpy as np
import pytest
import torch

from helpers import BENCH_BATCH as BATCH
from helpers import BENCH_SEED as SEED
from helpers import bench_batch, init_deterministic
from oracle import scn_oracle as O
from oracle import sparseconvnet_oracle as oscn
from sparseeventid_b200 import networks, synthetic

TOL = 2e-3


def rules_to_table(rules, n_out):
    t = np.full((len(rules), n_out), -1, dtype=np.int64)
    for k, r in enumerate(rules):
        r = np.asarray(r, dtype=np.int64).reshape(-1, 2)
        assert np.unique(r[:, 1]).shape[0] == r.shape[0], "an output row appears twice under one offset"
        t[k, r[:, 1]] = r[:, 0]
    return t


@pytest.mark.gpu
def test_bench_batch_rulebooks_bit_exact():
    import sparseconvnet as scn
    coords, feats, bs = bench_batch()
    ci = coords.astype(np.int64)
    assert np.unique(O.pack_keys(ci)).shape[0] == ci.shape[0], "the synthetic batch has no duplicate sites"
    x = scn.InputLayer(3, list(synthetic.GRID_3D))((torch.as_tensor(coords).cuda(), torch.as_tensor(feats).cuda(), bs))
    md = x.metadata
    sp = tuple(synthetic.GRID_3D)
    assert np.array_equal(md.coords(sp).cpu().numpy(), ci)               # level 0 rows == input order
    cur = ci                                     # oracle rows of the level
    gmap = np.arange(ci.shape[0])                # GPU row -> oracle row (level 0: identical numbering)

    def to_oracle(table, rows_map, vals_map):
        """GPU table [K, n] (rows / entries in GPU numbering) -> the same table in the oracle's numbering."""
        out = np.full_like(table, -1)
        out[:, rows_map] = np.where(table >= 0, vals_map[np.maximum(table, 0)], -1)
        return out

    for level in range(6):
        n = cur.shape[0]
        for filt in ([(5, 5, 5)] if level == 0 else []) + [(3, 3, 3)]:
            got = md.subm_table(sp, filt)[:, :n].cpu().numpy().astype(np.int64)
            want = rules_to_table(O.submanifold_rulebook(cur, filt), n)
            assert np.array_equal(to_oracle(got, gmap, gmap), want), f"level {level} filter {filt}: neighbour table differs from the oracle rulebook"
            assert bool((md.subm_table(sp, filt)[:, n:] == -1).all())
        if level == 5:
            break
        rule = md.strided_rule(sp, (2, 2, 2), (2, 2, 2))
        out_coords, rules, out_sp = O.strided_rulebook(cur, (2, 2, 2), (2, 2, 2), sp)
        assert rule.out_spatial == out_sp and rule.n_out == out_coords.shape[0]
        # same output sites; the GPU numbers them in first-appearance order, the oracle by ascending key
        gloc = md.coords(out_sp).cpu().numpy()
        gkeys, okeys = O.pack_keys(gloc), O.pack_keys(out_coords)
        assert np.array_equal(np.sort(gkeys), okeys)
        gmap_next = np.searchsorted(okeys, gkeys)
        down = rule.down[:, :rule.n_out].cpu().numpy().astype(np.int64)
        assert np.array_equal(to_oracle(down, gmap_next, gmap), rules_to_table(rules, rule.n_out)), f"level {level}: stride-2 map differs"
        up = rule.up[:, :n].cpu().numpy().astype(np.int64)
        want_up = rules_to_table([r[:, ::-1] for r in rules], n)
        assert np.array_equal(to_oracle(up, gmap, gmap_next), want_up), f"level {level}: transposed stride-2 map differs"
        cur, sp, gmap = out_coords, out_sp, gmap_next
    assert cur.shape[0] > 1000


def _step(scn_mod, device, dtype, coords, feats, bs, labels):
    enc, head = networks.build_networks(scn_mod, "dune3d")
    model = networks.EventIDModel(enc, head)
    init_deterministic(model)
    model.to(device)
    if dtype == torch.float64:
        model.double()
    model.train()
    head.eval()
    lab = {k: torch.as_tensor(v).to(device) for k, v in labels.items()}
    x = (torch.as_tensor(coords).to(device), torch.as_tensor(feats).to(device).to(dtype), bs)
    encoded = enc(x)
    logits = head(encoded)
    loss = networks.focal_loss(lab, logits)
    loss.backward()
    pooled = torch.as_tensor(encoded).double().mean(dim=(2, 3, 4)).cpu()
    return {"loss": float(loss.detach()), "pooled": pooled.detach(),
            "logits": {k: v.detach().double().cpu() for k, v in logits.items()},
            "grads": {n: p.grad.detach().double().cpu() for n, p in model.named_parameters()}}


def _dist(a, truth):
    """Per-tensor distances from truth: logits (max-norm relative), pooled encoder output and gradients (relative L2,
    cosine); parameters whose true gradient is ~0 (conv biases feeding a BatchNorm) are left out of the relative bars."""
    out = {"loss": abs(a["loss"] - truth["loss"]) / abs(truth["loss"]),
           "logits": max(float((a["logits"][k] - v).abs().max() / v.abs().max()) for k, v in truth["logits"].items()),
           "pooled": float((a["pooled"] - truth["pooled"]).norm() / truth["pooled"].norm())}
    gmax = max(float(g.norm()) for g in truth["grads"].values())
    rel, cos, nrm = {}, {}, {}
    for n, g in truth["grads"].items():
        if float(g.norm()) < 1e-3 * gmax:
            assert float(a["grads"][n].norm()) < 1e-2 * gmax, f"gradient of {n} should be ~0"
            continue
        d = a["grads"][n]
        rel[n] = float((d - g).norm() / g.norm())
        cos[n] = float((d.flatten() @ g.flatten()) / (d.norm() * g.norm()))
        nrm[n] = abs(float(d.norm()) - float(g.norm())) / float(g.norm())
    out["grad_rel"], out["grad_cos"], out["grad_norm"] = rel, cos, nrm
    return out


@pytest.mark.gpu
def test_bench_batch_training_step_vs_oracle():
    import sparseconvnet as scn
    coords, feats, bs = bench_batch()
    labels = synthetic.make_labels(BATCH, seed=SEED)
    torch.set_num_threads(max(1, torch.get_num_threads()))
    oscn.set_numerics("fp32")
    truth = _step(oscn, "cpu", torch.float64, coords, feats, bs, labels)
    oscn.set_numerics("bf16")
    try:
        o_bf16 = _dist(_step(oscn, "cpu", torch.float32, coords, feats, bs, labels), truth)
    finally:
        oscn.set_numerics("fp32")
    try:
        scn.set_precision("fp32")
        g32 = _dist(_step(scn, "cuda", torch.float32, coords, feats, bs, labels), truth)
        scn.set_precision("bf16")
        g16 = _dist(_step(scn, "cuda", torch.float32, coords, feats, bs, labels), truth)
    finally:
        scn.set_precision("bf16")

    def summary(d):
        r, c = np.asarray(list(d["grad_rel"].values())), np.asarray(list(d["grad_cos"].values()))
        return (f"loss {d['loss']:.1e} logits {d['logits']:.1e} pooled {d['pooled']:.1e} grad rel-L2 median {np.median(r):.1e} "
                f"max {r.max():.1e} cos min {c.min():.5f} grad-norm max {max(d['grad_norm'].values()):.1e}")
    print(f"\nbatch-{BATCH} step vs float64 oracle:\n  gpu fp32 : {summary(g32)}\n  gpu bf16 : {summary(g16)}\n  oracle bf16: {summary(o_bf16)}")

    # fp32 mode: the north-star bar
    assert g32["loss"] <= TOL and g32["logits"] <= TOL and g32["pooled"] <= TOL
    assert max(g32["grad_norm"].values()) <= TOL, "fp32 gradient norms"
    r32 = np.asarray(list(g32["grad_rel"].values()))
    assert r32.max() <= 2e-2 and min(g32["grad_cos"].values()) >= 0.9999
    # bf16 mode: loss / logits at the north-star bar; everything else relative to truth
    assert g16["loss"] <= TOL and g16["logits"] <= TOL
    assert g16["pooled"] <= 1.5 * o_bf16["pooled"] + 1e-3
    for n, e in g16["grad_rel"].items():
        assert e <= 1.5 * o_bf16["grad_rel"][n] + 5e-2, f"bf16 gradient of {n}: {e:.3e} vs oracle[bf16] {o_bf16['grad_rel'][n]:.3e}"
        assert g16["grad_cos"][n] >= o_bf16["grad_cos"][n] - 0.05, f"bf16 gradient direction of {n}"
