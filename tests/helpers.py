"""Shared test helpers (seeded random sparse inputs)."""
import numpy as np
import torch


def random_sites(n, grid, batch, seed, dup=0):
    """int64 [n(+dup), 4] rows (x, y, z, b), unique unless dup > 0; batch index last."""
    rng = np.random.default_rng(seed)
    g = np.asarray(grid)
    total = int(np.prod(g)) * batch
    flat = rng.choice(total, size=min(n, total), replace=False)
    b, r = np.divmod(flat, int(np.prod(g)))
    x, r = np.divmod(r, g[1] * g[2])
    y, z = np.divmod(r, g[2])
    c = np.stack([x, y, z, b], 1).astype(np.int64)
    if dup:
        c = np.concatenate([c, c[rng.integers(0, c.shape[0], size=dup)]], 0)
        c = c[rng.permutation(c.shape[0])]
    return c


def blob_sites(n, grid, batch, seed):
    """Clustered sites (random walk) so that neighbourhoods are dense like tracks."""
    rng = np.random.default_rng(seed)
    g = np.asarray(grid)
    out = []
    for b in range(batch):
        p = (g // 2).astype(np.int64)
        pts = []
        for _ in range(n):
            p = np.clip(p + rng.integers(-1, 2, size=3), 0, g - 1)
            pts.append(p.copy())
        pts = np.unique(np.asarray(pts), axis=0)
        pts = pts[rng.permutation(pts.shape[0])]
        out.append(np.concatenate([pts, np.full((pts.shape[0], 1), b)], 1))
    return np.concatenate(out, 0).astype(np.int64)


# bench.py's first batch: host_batch(64, 1234 + 100000 * rank + 1000 * i) with rank = i = 0
BENCH_BATCH, BENCH_SEED = 64, 1234


def bench_batch(batch=BENCH_BATCH, seed=BENCH_SEED):
    """The benchmark's first batch (64 synthetic dune3d events, ~5e5 active sites): float64 coordinates, float32 features,
    batch size."""
    from sparseeventid_b200 import synthetic
    from sparseeventid_b200.data_transforms import larcvsparse_to_scnsparse_3d
    c, f, bs = larcvsparse_to_scnsparse_3d(synthetic.larcv_batch_3d(batch, seed=seed))
    return np.ascontiguousarray(c, dtype=np.float64), np.ascontiguousarray(f, dtype=np.float32), bs


def rel_err(a, b):
    a = torch.as_tensor(a).detach().double().cpu()
    b = torch.as_tensor(b).detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def rel_l2(a, b):
    a = torch.as_tensor(a).detach().double().cpu()
    b = torch.as_tensor(b).detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def init_deterministic(model, seed=7):
    """Fills every parameter/buffer from numpy PCG64 keyed by its name: identical on any box, any torch
    (used by tests/golden/make_golden.py and by the tests that replay the fixtures)."""
    import zlib
    with torch.no_grad():
        for name, p in list(model.named_parameters()) + list(model.named_buffers()):
            rng = np.random.default_rng([seed, zlib.crc32(name.encode())])
            if name.endswith("running_var"):
                v = rng.uniform(0.5, 1.5, size=tuple(p.shape))
            elif name.endswith("running_mean"):
                v = rng.normal(0, 0.1, size=tuple(p.shape))
            elif p.dim() >= 3:                         # conv weight [K,1,Cin,Cout]
                fan = p.shape[0] * p.shape[-2]
                v = rng.normal(0, np.sqrt(2.0 / fan), size=tuple(p.shape))
            elif p.dim() == 2:                         # Linear
                v = rng.normal(0, np.sqrt(1.0 / p.shape[1]), size=tuple(p.shape))
            elif name.endswith("norm.weight"):
                v = rng.uniform(0.8, 1.2, size=tuple(p.shape))
            else:
                v = rng.normal(0, 0.05, size=tuple(p.shape))
            p.copy_(torch.as_tensor(v, dtype=p.dtype))


def small_batch(dataset, batch=2, seed=4321, max_voxels=6000):
    """The seeded synthetic mini-batch the golden fixtures were generated on."""
    from sparseeventid_b200 import synthetic
    from sparseeventid_b200.data_transforms import larcvsparse_to_scnsparse_2d, larcvsparse_to_scnsparse_3d
    if dataset == "dune3d":
        return larcvsparse_to_scnsparse_3d(synthetic.larcv_batch_3d(batch, seed=seed, max_voxels=max_voxels))
    return larcvsparse_to_scnsparse_2d(synthetic.larcv_batch_2d(batch, seed=seed, max_voxels=max_voxels))


# Legacy networks (SURVEY §8 a11): reduced-depth instances of the reference's torch/sparseresnet3d.py and
# torch/sparseresnet.py used for the committed fixtures (tests/golden/make_golden_legacy.py).
LEGACY_CASES = {
    "legacy3d_nf32_d2": {"kind": "3d", "cfg": dict(n_initial_filters=32, network_depth=2, depth_pre_merge=0,
                                                   res_blocks_per_layer=1, batch_norm=True, leaky_relu=False)},
    "legacy2d_nf32_d3_pre2": {"kind": "2d", "cfg": dict(n_initial_filters=32, network_depth=3, depth_pre_merge=2,
                                                        res_blocks_per_layer=1, batch_norm=True, leaky_relu=True)},
}


def legacy_batch(case, batch=2, seed=2468, max_voxels=3000):
    """The seeded synthetic mini-batch of a legacy fixture: SCN input tuple on the legacy grids."""
    from sparseeventid_b200 import synthetic
    from sparseeventid_b200.data_transforms import larcvsparse_to_scnsparse_2d, larcvsparse_to_scnsparse_3d
    if LEGACY_CASES[case]["kind"] == "3d":
        return larcvsparse_to_scnsparse_3d(
            synthetic.larcv_batch_3d(batch, seed=seed, grid=(1536, 1536, 1536), max_voxels=max_voxels))
    return larcvsparse_to_scnsparse_2d(synthetic.larcv_batch_2d(batch, seed=seed, max_voxels=max_voxels))
