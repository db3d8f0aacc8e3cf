"""Checks against what the REFERENCE'S OWN FILES produce, recorded in tests/golden/reference_files.json
(tests/golden/make_reference_files.py says how; the reference tree is not part of this repository).  No GPU needed:
transforms are numpy, and constructing a network only allocates parameters.

  * the host input transforms == the reference's torch_geometric-free twins
    (src/utils/core/larcvio/data_transforms.py:50-142; src/io/data_transforms.py:21-49,198-252 are the same functions
    behind an unconditional `import torch_geometric`) on the same seeded synthetic batches;
  * the reference's `build_networks` (src/networks/classification_head.py:30-55 -> src/networks/resnet.py:10-161,
    sparse_building_blocks.py) constructed on the PRODUCT `sparseconvnet` package: the repo's mirror
    (sparseeventid_b200/networks.py) built on the product package has its state_dict keys, shapes, dtypes and
    parameter counts, and every sparse layer is the product's class.
"""
import hashlib
import json
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_files.json")


def _record(dataset):
    with open(GOLDEN) as f:
        return json.load(f)[dataset]


@pytest.mark.parametrize("dataset", ["dune3d", "dune2d"])
def test_host_transform_matches_reference_twin(dataset):
    from sparseeventid_b200 import data_transforms as mine
    from sparseeventid_b200 import synthetic
    want = _record(dataset)["transform"]
    if dataset == "dune3d":
        arr = synthetic.larcv_batch_3d(5, seed=77, max_voxels=4000)
        got = mine.larcvsparse_to_scnsparse_3d(arr)
    else:
        arr = synthetic.larcv_batch_2d(5, seed=77, max_voxels=4000)
        got = mine.larcvsparse_to_scnsparse_2d(arr)
    assert type(got).__name__ == want["type"] and len(got) == 3
    rows = np.asarray(want["sample_rows"])
    for a, name in zip(got[:2], ("coords", "feats")):
        w = want[name]
        assert str(a.dtype) == w["dtype"] and list(a.shape) == w["shape"], name
        assert np.array_equal(a[rows], np.asarray(want["sample_" + name], dtype=a.dtype)), name
        assert hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest() == w["sha256"], name
    assert got[2] == want["batch_size"]
    assert got[0].shape[0] > 1000


@pytest.mark.parametrize("dataset", ["dune3d", "dune2d"])
def test_product_networks_match_reference_layout(dataset):
    import sparseconvnet as product
    from sparseeventid_b200 import networks as mirror
    assert product.__name__ == "sparseconvnet" and "sparseeventid_b200" in product.SubmanifoldConvolution.__module__
    want = _record(dataset)["layout"]
    encoder, head = mirror.build_networks(product, dataset)
    model = mirror.EventIDModel(encoder, head)
    got = [[k, list(v.shape), str(v.dtype)] for k, v in model.state_dict().items()]
    assert [e[0] for e in got] == [e[0] for e in want["state_dict"]]
    for g, w in zip(got, want["state_dict"]):
        assert g == w, g[0]
    n = sum(p.numel() for p in model.parameters())
    assert n == want["n_params"] == {"dune3d": 20881994, "dune2d": 7173578}[dataset]      # SURVEY.md App. B census
    # every sparse layer of the encoder is the product's class (nothing fell back to a stub)
    leaves = [m for m in encoder.modules() if not list(m.children()) and list(m.parameters(recurse=False))]
    assert len(leaves) > 50, len(leaves)
    assert {type(m).__module__ for m in leaves} == {"sparseeventid_b200.scn.modules"}
