"""CPU checks of the drop-in boundary: the C-ABI library builds/loads and exports exactly the symbols
include/scn_b200.h declares (no compute calls without a GPU); the Python veneer keeps SCN's module surface."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "scn_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(scn_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from sparseeventid_b200 import _lib, build
    path = build.build()
    lib = _lib.load(path)
    names = declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/scn_b200.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature"
    assert set(_lib.SIGNATURES) == set(names), set(_lib.SIGNATURES) ^ set(names)
    assert lib.scn_version().decode().endswith("sm_100a")
    assert lib.scn_hash_capacity(1000) == 2048 and lib.scn_hash_capacity(0) == 1024


def test_header_is_plain_c_and_a_c_caller_links(tmp_path):
    """include/scn_b200.h is valid pedantic C99 (no C++/torch types at the boundary) and tools/abi_harness.c -- a
    caller that is plain C + the CUDA runtime -- compiles and links against the library without torch."""
    import subprocess
    from sparseeventid_b200 import build
    build.build()
    probe = tmp_path / "h.c"
    probe.write_text('#include "scn_b200.h"\nint main(void) { return scn_version() == 0; }\n')
    inc = os.path.join(ROOT, "include")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-fsyntax-only", "-I", inc, str(probe)],
                   check=True)
    exe = tmp_path / "abi_harness"
    subprocess.run(["gcc", "-std=c99", "-O1", "-Wall", "-Werror", "-I", inc, "-I/usr/local/cuda/include",
                    os.path.join(ROOT, "tools", "abi_harness.c"), "-L", os.path.dirname(build.LIB), "-lscn_b200",
                    "-L/usr/local/cuda/lib64", "-lcudart", "-lm", "-o", str(exe)], check=True)
    out = subprocess.run(["ldd", str(exe)], capture_output=True, text=True).stdout
    assert "libscn_b200.so" in out and "libtorch" not in out and "libpython" not in out and "libc10" not in out


def test_library_is_sm100a_only_and_native():
    import subprocess
    from sparseeventid_b200 import build
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "--list-elf", build.LIB], capture_output=True, text=True)
    assert "sm_100a" in out.stdout and "sm_90" not in out.stdout and "sm_80" not in out.stdout


def test_module_surface_matches_reference_usage():
    """Constructor forms / parameter names the reference uses (SURVEY.md 2.3, App. A)."""
    import sparseconvnet as scn
    c = scn.SubmanifoldConvolution(dimension=3, nIn=1, nOut=32, filter_size=[5, 5, 5], bias=True)
    assert tuple(c.weight.shape) == (125, 1, 1, 32) and tuple(c.bias.shape) == (32,)
    c2 = scn.SubmanifoldConvolution(3, 1, 32, filter_size=5, bias=False)
    assert c2.bias is None and tuple(c2.weight.shape) == (125, 1, 1, 32)
    assert scn.SubmanifoldConvolution(3, 192, 128, filter_size=1, bias=True).filter_volume == 1
    assert scn.SubmanifoldConvolution(2, 4, 4, 3, False).filter_volume == 9
    d = scn.Convolution(dimension=3, nIn=32, nOut=64, filter_size=[1, 2, 2], filter_stride=[1, 2, 2], bias=False)
    assert tuple(d.weight.shape) == (4, 1, 32, 64)
    scn.Deconvolution(dimension=3, nIn=64, nOut=32, filter_size=[2, 2, 2], filter_stride=[2, 2, 2], bias=True)
    bn = scn.BatchNormalization(32)
    assert set(dict(bn.named_buffers())) == {"running_mean", "running_var"} and bn.eps == 1e-4 and bn.momentum == 0.9
    assert scn.BatchNormReLU(8).leakiness == 0 and abs(scn.BatchNormLeakyReLU(8).leakiness - 0.333) < 1e-9
    assert abs(scn.LeakyReLU().leak - 1 / 3) < 1e-9
    il = scn.InputLayer(dimension=3, spatial_size=torch.tensor([1024, 512, 1280]))
    assert il.spatial_size.tolist() == [1024, 512, 1280]
    assert scn.InputLayer(3, (1536, 1536, 1536)).spatial_size.tolist() == [1536] * 3
    seq = torch.nn.Sequential(scn.SparseToDense(dimension=3, nPlanes=128))
    assert isinstance(seq[0], torch.nn.Module)
    ap = scn.AveragePooling(dimension=3, pool_size=[2, 2, 2], pool_stride=[2, 2, 2])      # sparse_building_blocks.py:150-154
    assert ap.pool_volume == 8 and not list(ap.parameters()) and scn.AveragePooling(3, 2, 2, 1).nFeaturesToDrop == 1
    act = scn.Identity
    assert isinstance(act(), torch.nn.Module) and isinstance(scn.AddTable(), torch.nn.Module)
    # 3-D (2018-19 SCN) conv weights load into the 4-D parameter
    sd = {"weight": torch.zeros(27, 32, 32), "bias": torch.zeros(32)}
    scn.SubmanifoldConvolution(3, 32, 32, 3, True).load_state_dict(sd)


def test_product_path_has_no_cpu_fallback():
    import sparseconvnet as scn
    with pytest.raises(RuntimeError):
        scn.InputLayer(3, 8)((torch.zeros(4, 4).long(), torch.zeros(4, 1)))
    import sparseeventid_b200
    pkg = os.path.dirname(sparseeventid_b200.__file__)
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f"{f} imports the oracle"


def test_state_dict_keys_match_reference_layout():
    import sparseconvnet as scn
    from sparseeventid_b200 import networks
    enc, head = networks.build_networks(scn, "dune3d")
    keys = list(networks.EventIDModel(enc, head).state_dict())
    assert "encoder.network_layers.0.block_0.convolution_1.conv1.weight" in keys
    assert "encoder.network_layers.1.conv.weight" in keys and "encoder.network_layers.1.norm.running_var" in keys
    assert "encoder.bottleneck.bias" in keys and "head.classification_head.labelneutID.2.weight" in keys
    assert sum(p.numel() for p in enc.parameters()) == 20747328
    assert sum(p.numel() for p in head.parameters()) == 134666
    enc2, _ = networks.build_networks(scn, "dune2d")
    assert sum(p.numel() for p in enc2.parameters()) == 7038912
    assert enc.output_shape == [128, 32, 16, 40] and enc2.output_shape == [128, 3, 48, 32]


def test_torch_extension_builds_and_exports_the_module_functions():
    """The thin PyTorch C++ layer (csrc_torch/scn_torch.cpp) builds in-tree on a CPU-only box and exposes the autograd
    functions the modules call (no compute here: they need a GPU)."""
    from sparseeventid_b200 import build
    from sparseeventid_b200.scn import _ext
    path = build.build_torch_ext()
    assert os.path.exists(path) and os.path.dirname(path).endswith("build_torch")
    ext = _ext.get()
    assert ext is not None
    for name in ("conv", "batch_norm", "add_leaky", "leaky", "set_grad_ready_callback"):
        assert hasattr(ext, name), name


def test_missing_torch_extension_fails_at_first_forward_not_at_import(tmp_path):
    """The C++ autograd layer is required but loaded on first use: with it missing, importing the package and building
    a module work, and the first convolution forward raises a RuntimeError that names the build command."""
    import subprocess
    import sys
    code = f"""
import torch
from sparseeventid_b200 import build
build.TORCH_EXT_SO = {str(tmp_path / "scn_b200_torch.so")!r}
import sparseconvnet as scn
from sparseeventid_b200.scn import core
conv = scn.SubmanifoldConvolution(3, 1, 4, 3, True)
md, sp = core.Metadata(3, "cpu"), (4, 4, 4)       # a level and its neighbour table, as if already built
md.levels[sp] = core.Level(torch.zeros(2, dtype=torch.int64), 2, None, None, 0)
md.subm[(sp, (3, 3, 3))] = torch.full((27, 128), -1, dtype=torch.int32)
try:
    conv(core.SparseConvNetTensor(torch.zeros(2, 1), md, torch.LongTensor(list(sp))))
except RuntimeError as e:
    print("raised:", e)
"""
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "raised: scn_b200_torch.so not found" in r.stdout and "`python -m sparseeventid_b200.build`" in r.stdout, r.stdout


@pytest.mark.gpu
def test_plain_c_caller_runs_on_the_gpu(tmp_path):
    """tools/abi_harness.c -- a C99 program with no Python / torch in the process -- drives the hot path through
    include/scn_b200.h on the device and checks its results itself (InputLayer rules, convolutions, pooling)."""
    import subprocess
    from sparseeventid_b200 import build
    exe = tmp_path / "abi_harness"
    subprocess.run(["gcc", "-std=c99", "-O2", "-I", os.path.join(ROOT, "include"), "-I/usr/local/cuda/include",
                    os.path.join(ROOT, "tools", "abi_harness.c"), "-L", os.path.dirname(build.LIB), "-lscn_b200",
                    "-L/usr/local/cuda/lib64", "-lcudart", "-lm", "-o", str(exe)], check=True)
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.dirname(build.LIB) + ":/usr/local/cuda/lib64:" + os.environ.get("LD_LIBRARY_PATH", ""))
    r = subprocess.run([str(exe)], capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
    assert "all checks passed" in r.stdout
