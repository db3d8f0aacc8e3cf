"""Generates tests/golden/reference_files.json, the record tests/test_reference_files.py compares against:

  * the output of the reference's larcv -> SCN transform (src/utils/core/larcvio/data_transforms.py:108-142 and
    its 2-D twin) on seeded synthetic batches: type, dtypes, shapes, batch size, the sha256 of the coordinate and
    feature bytes, and a fixed sample of rows;
  * the state_dict layout (keys, shapes, dtypes) and parameter count of the reference's `build_networks`
    (src/networks/classification_head.py:30-55) constructed on this repository's `sparseconvnet` package.

The reference tree is not part of this repository.  While it was at hand, tests/test_reference_files.py imported
those files and held them equal to this repository's twins (`sparseeventid_b200.data_transforms` and the mirror
`sparseeventid_b200.networks.build_networks`), so the record is taken from the twins:

    python tests/golden/make_reference_files.py

The parameter names and counts are cross-checked against tests/golden/*_default_encoder.npz, which
tests/golden/make_golden.py generated from the reference's own model files.
"""
import hashlib
import json
import os
import re
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
OUT = os.path.join(HERE, "reference_files.json")
SAMPLE_ROWS = 64


def transform_input(dataset):
    from sparseeventid_b200 import synthetic
    if dataset == "dune3d":
        return synthetic.larcv_batch_3d(5, seed=77, max_voxels=4000)
    return synthetic.larcv_batch_2d(5, seed=77, max_voxels=4000)


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def sample_rows(n):
    return np.sort(np.random.default_rng(0).choice(n, SAMPLE_ROWS, replace=False))


def transform_record(dataset):
    from sparseeventid_b200 import data_transforms as T
    arr = transform_input(dataset)
    out = T.larcvsparse_to_scnsparse_3d(arr) if dataset == "dune3d" else T.larcvsparse_to_scnsparse_2d(arr)
    coords, feats, bs = out
    rows = sample_rows(coords.shape[0])
    return {"type": type(out).__name__, "batch_size": bs,
            "coords": {"dtype": str(coords.dtype), "shape": list(coords.shape), "sha256": sha256(coords)},
            "feats": {"dtype": str(feats.dtype), "shape": list(feats.shape), "sha256": sha256(feats)},
            "sample_rows": rows.tolist(), "sample_coords": coords[rows].tolist(),
            "sample_feats": feats[rows].astype(np.float64).tolist()}


def layout_record(dataset):
    import sparseconvnet as product
    from sparseeventid_b200 import networks
    model = networks.EventIDModel(*networks.build_networks(product, dataset))
    fx = np.load(os.path.join(HERE, f"{dataset}_default_encoder.npz"))
    assert [n for n, _ in model.named_parameters()] == [str(s) for s in fx["param_names"]], dataset
    n_params = sum(p.numel() for p in model.parameters())
    assert n_params == int(fx["n_params"][0]), dataset
    return {"n_params": n_params,
            "state_dict": [[k, list(v.shape), str(v.dtype)] for k, v in model.state_dict().items()]}


def main():
    rec = {ds: {"transform": transform_record(ds), "layout": layout_record(ds)} for ds in ("dune3d", "dune2d")}
    text = json.dumps(rec, indent=1)
    # innermost lists on one line each (a state_dict entry, a sampled row): a reviewable diff when the record changes
    text = re.sub(r"\[([^\[\]{}]*)\]", lambda m: "[" + ", ".join(x.strip() for x in m.group(1).split(",")) + "]", text)
    with open(OUT, "w") as f:
        f.write(text + "\n")
    print("->", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
