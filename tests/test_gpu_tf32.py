"""The "tf32" precision mode: fp32 features, TF32 operands on the tcgen05 convolution kernels, fp32 accumulation.

Kernel level, through the entry points the layers call, against the float64 references of test_gpu_kernels.py:
  * probe: what the tensor cores do with the low 13 bits of an fp32 feature (x = 1 + 2^-11 + 2^-12, W = 1);
  * exact arm: integer operands in {-2..2} (exact in TF32, every partial sum exact in fp32): outputs, dx, dW and dbias
    must equal the float64 reference bit for bit;
  * rounding arm: N(0,1) values rounded to bf16 (exact in TF32): the bars of fp32 accumulation;
  * TF32-operand arm: full fp32 N(0,1) operands: each element within the TF32 operand error, and in aggregate at most
    half the error of float64 arithmetic on bf16-rounded operands -- the check that fails if an operand is narrowed to
    bf16 anywhere.
Every launch runs twice and must give identical bits (the stem's atomic weight gradient with non-integer operands
excepted).  The cases: the benchmark batch's six levels, a forced launch-configuration sweep for 1..8 channel chunks,
tile / wave row edges, rectangular tables and every TF32 k_wgrad_tc instantiation in its three wave regimes; a final
test checks that they reached every launcher branch.

Network level: the default dune3d encoder + heads against truth (the fp32 fixture) with the same-precision bars as
test_golden_network.py, closer to truth than the "mixed" mode; one benchmark-scale training step against the float64
oracle; 20 Trainer steps with finite losses.

The oracle's stated-numerics emulation knows "fp32", "mixed" and "bf16"; tf32_numerics() below adds the TF32 operand
rounding to it for the duration of a test: weights rounded to nearest (the weight image is built with cvt.rna), x and
dout as the probe pins the hardware (TF32_FEATURES).
"""
import ctypes
import math
import os
from contextlib import contextmanager

import numpy as np
import pytest
import torch

from helpers import bench_batch, blob_sites, init_deterministic, small_batch
from oracle import sparseconvnet_oracle as oscn
from test_gpu_kernels import (CHANNELS, EDGE_ROWS, assert_repeat, assert_sums, module_backward, module_forward,
                              rand_table, ref_dgrad, ref_forward, ref_wgrad)

# what the tcgen05 tensor cores do with the 13 mantissa bits of an fp32 operand below TF32's 10: "truncate" (ignore
# them) or "round" (to nearest); pinned by test_probe_feature_rounding on a B200
TF32_FEATURES = "truncate"

ARMS = ["exact", "rounding", "tf32"]


# ==================================================================================== TF32 rounding (bit level)


def _bits(t):
    return t.detach().to(torch.float32).contiguous().view(torch.int32)


def tf32_truncate(t):
    """fp32 value with the low 13 mantissa bits cleared (toward zero)."""
    return (_bits(t) & ~0x1FFF).view(torch.float32).to(t.dtype)


def tf32_round(t):
    """Round to the nearest TF32 value, ties away from zero (cvt.rna.tf32.f32; finite values)."""
    return ((_bits(t) + 0x1000) & ~0x1FFF).view(torch.float32).to(t.dtype)


def tf32_features(t):
    return tf32_truncate(t) if TF32_FEATURES == "truncate" else tf32_round(t)


@contextmanager
def tf32_numerics():
    """The oracle as the "tf32" mode computes: operands of tensor-core convolution shapes rounded to TF32 (the weight,
    the only 3-D operand, to nearest; x and dout as the hardware reads them), nothing stored rounded."""
    saved_ro = oscn._ro

    def ro(t, k, n_in, n_out):
        if not oscn._tensor_core_shape(k, n_in, n_out):
            return t
        return tf32_round(t) if t.dim() == 3 else tf32_features(t)

    oscn.set_numerics("fp32")
    oscn._ro = ro
    try:
        yield
    finally:
        oscn._ro = saved_ro
        oscn.set_numerics("fp32")


def test_tf32_rounding_matches_bit_definition():
    """Hand-picked values: ties, the 2^-11 / 2^-12 bits, negatives, subnormals."""
    one = 1.0
    u = 2.0 ** -10                       # TF32 ulp at 1
    cases = [  # value, truncated, rounded to nearest (ties away)
        (one, one, one),
        (one + 2 ** -11, one, one + u),                      # exact tie -> away from zero
        (one + 2 ** -12, one, one),                          # below half
        (one + 2 ** -11 + 2 ** -12, one, one + u),           # above half
        (one + u + 2 ** -11, one + u, one + 2 * u),          # tie at an odd TF32 mantissa -> away as well (not even)
        (-(one + 2 ** -11), -one, -(one + u)),
        (-(one + 2 ** -12), -one, -one),
        (2.0 - 2 ** -23, 2.0 - u, 2.0),                      # rounds up into the next binade
        # subnormals: the TF32 grid is 2^-136 there
        (3 * 2.0 ** -136, 3 * 2.0 ** -136, 3 * 2.0 ** -136),
        (2.0 ** -149, 0.0, 0.0),                             # smallest subnormal
        (2.0 ** -137, 0.0, 2.0 ** -136),                     # tie -> away from zero
        (2.0 ** -137 + 2.0 ** -138, 0.0, 2.0 ** -136),
        (-(2.0 ** -136 + 2.0 ** -138), -(2.0 ** -136), -(2.0 ** -136)),
        (2.0 ** -127 + 2.0 ** -137, 2.0 ** -127, 2.0 ** -127 + 2.0 ** -136),
    ]
    v = torch.tensor([c[0] for c in cases], dtype=torch.float32)
    assert torch.equal(tf32_truncate(v), torch.tensor([c[1] for c in cases], dtype=torch.float32))
    assert torch.equal(tf32_round(v), torch.tensor([c[2] for c in cases], dtype=torch.float32))
    # integers of the exact arm and bf16 values of the rounding arm are TF32 values
    w = torch.randn(4096, generator=torch.Generator().manual_seed(1)).bfloat16().float()
    assert torch.equal(tf32_truncate(w), w) and torch.equal(tf32_round(w), w)
    # a float64 tensor is rounded through its fp32 value
    assert torch.equal(tf32_round(v.double()), tf32_round(v).double())


def test_tf32_mode_is_accepted():
    import subprocess
    import sys
    from sparseeventid_b200 import _lib as L
    from sparseeventid_b200.scn import config
    saved = config.get_precision()
    try:
        config.set_precision("tf32")
        assert config.get_precision() == "tf32"
        assert config.feature_dtype() == torch.float32 and config.precision_code() == L.PREC_TF32 == 2
        for mode in ("fp32", "mixed", "bf16"):
            config.set_precision(mode)
            assert config.precision_code() == {"fp32": L.PREC_FP32, "mixed": L.PREC_BF16, "bf16": L.PREC_BF16}[mode]
        for bad in ("TF32", "fp16", "", None):
            with pytest.raises(ValueError):
                config.set_precision(bad)
    finally:
        config.set_precision(saved)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = "from sparseeventid_b200.scn import config; print(config.get_precision(), config.precision_code())"
    for env, want in (("tf32", "tf32 2"), ("bogus", None)):
        r = subprocess.run([sys.executable, "-c", code], cwd=root, capture_output=True, text=True,
                           env=dict(os.environ, SCN_B200_PRECISION=env))
        if want is None:
            assert r.returncode != 0 and "SCN_B200_PRECISION" in r.stderr
        else:
            assert r.returncode == 0 and r.stdout.split() == want.split(), r.stderr


# ==================================================================================== GPU plumbing

LAUNCH_FIELDS = ("grid", "T", "NM", "nbuf", "ksplit", "SA", "SB", "min_tiles", "max_tiles")
WG_FIELDS = ("grid", "s_other", "s_centre", "pairs", "slots", "nca", "ncb")
_LAUNCHES = []          # (n_in, {LAUNCH_FIELDS}) of every TF32 k_conv_tc launch of this file
_WG_LAUNCHES = []       # (K, Cin, Cout, {WG_FIELDS}) of every TF32 k_wgrad_tc launch
_DONE = {}


def _done(name):
    _DONE[name] = _DONE.get(name, 0) + 1


def _lib():
    from sparseeventid_b200 import _lib as L
    lib = L.lib()
    lib.scn_tc_debug_knobs.argtypes = [ctypes.c_int] * 4
    lib.scn_tc_debug_knobs.restype = None
    lib.scn_tc_debug_last_launch.argtypes = [ctypes.POINTER(ctypes.c_int32)]
    lib.scn_tc_debug_last_launch.restype = None
    lib.scn_wgrad_debug_last_launch.argtypes = [ctypes.POINTER(ctypes.c_int32)]
    lib.scn_wgrad_debug_last_launch.restype = None
    return lib


def _last_launch(n_in):
    buf = (ctypes.c_int32 * len(LAUNCH_FIELDS))()
    _lib().scn_tc_debug_last_launch(buf)
    cfg = dict(zip(LAUNCH_FIELDS, list(buf)))
    _LAUNCHES.append((n_in, cfg))
    return cfg


def _last_wgrad_launch(K, cin, cout):
    buf = (ctypes.c_int32 * len(WG_FIELDS))()
    _lib().scn_wgrad_debug_last_launch(buf)
    cfg = dict(zip(WG_FIELDS, list(buf)))
    _WG_LAUNCHES.append((K, cin, cout, cfg))
    return cfg


@pytest.fixture
def knobs():
    lib = _lib()
    yield lambda grid, t, sa, sb: lib.scn_tc_debug_knobs(grid, t, sa, sb)
    lib.scn_tc_debug_knobs(0, 0, 0, 0)


def _prec():
    from sparseeventid_b200 import _lib as L
    return L.PREC_TF32


def draw(shape, arm, gen):
    """fp32 operands: integers {-2..2} (exact), N(0,1) rounded to bf16 (rounding) or full fp32 N(0,1) (tf32)."""
    if arm == "exact":
        return torch.randint(-2, 3, shape, device="cuda", generator=gen).float()
    v = torch.randn(shape, device="cuda", generator=gen)
    return v.bfloat16().float() if arm == "rounding" else v


def _report(bad, got, ref, mag, what):
    idx = torch.nonzero(bad)[:6].tolist()
    rows = [f"  at {tuple(i)}: A={float(mag[tuple(i)]):.6g} ref={float(ref[tuple(i)]):.9g} got={float(got[tuple(i)]):.9g}"
            for i in idx]
    return f"{what}: {int(bad.sum())} of {bad.numel()} elements wrong\n" + "\n".join(rows)


def _rel_l2(a, ref):
    n = float(ref.norm())
    return float((a.double() - ref).norm()) / n if n > 0 else 0.0


def check_values(got, ref, mag, arm, what, sums=False, bf16_ref=None):
    """fp32 outputs / dx (sums=False) or dW (sums=True) against the float64 reference of the unrounded operands.
    bf16_ref: the float64 result on bf16-rounded operands (tf32 arm: the aggregate bar).  Arm "split": full fp32
    operands through the stem's hi/lo bf16 split (x = hi + lo to 2^-17, no lo.lo term): 2^-14 A throughout."""
    assert got.shape == ref.shape, what
    assert got.dtype == torch.float32, what
    if ref.numel() == 0:
        return
    if arm == "exact":
        assert float(mag.max()) < 2 ** 24, f"{what}: precondition A < 2^24 broken ({float(mag.max())})"
        bad = got.double() != ref
    else:
        acc = 2 ** -14 if sums or arm == "split" else 2 ** -16
        bar = acc * mag + (2 ** -9 * mag if arm == "tf32" else 0)
        bad = (got.double() - ref).abs() > bar
    assert not bool(bad.any()), _report(bad, got, ref, mag, what)
    if arm == "tf32" and bf16_ref is not None and float(ref.norm()) > 0:
        e_got, e_bf16 = _rel_l2(got, ref), _rel_l2(bf16_ref, ref)
        assert e_got <= 0.5 * e_bf16, f"{what}: relative L2 error {e_got:.3e} > half of bf16 operands' {e_bf16:.3e}"


def _bf(t):
    return t.bfloat16().double()


def check_layer(x, w, bias, dout, nbr_fwd, nbr_bwd, n_out_rows, mirror, arm, what, need_dx=True, atomic_wgrad=False):
    """Forward, dgrad, wgrad and dbias of one layer through the module entry points in the tf32 mode, twice each."""
    from sparseeventid_b200.scn import ops
    prec = _prec()
    K, cin, cout = w.shape
    f32 = torch.float32
    out, again = module_forward(x, w, bias, nbr_fwd, n_out_rows, prec, f32), module_forward(x, w, bias, nbr_fwd, n_out_rows, prec, f32)
    if ops.conv_path(K, cin, cout, prec, f32) == 2:
        _last_launch(cin)
    ref, mag = ref_forward(x, w, bias, nbr_fwd, n_out_rows)
    bref = ref_forward(_bf(x), _bf(w), bias, nbr_fwd, n_out_rows)[0] if arm == "tf32" else None
    check_values(out, ref, mag, arm, what + " forward", bf16_ref=bref)
    assert_repeat(out, again, what + " forward")
    del ref, mag, bref
    first = module_backward(x, dout, w, nbr_fwd, nbr_bwd, n_out_rows, mirror, prec, need_dx)
    second = module_backward(x, dout, w, nbr_fwd, nbr_bwd, n_out_rows, mirror, prec, need_dx)
    dx, dw, db = first
    if need_dx:
        if ops.conv_path(K, cout, cin, prec, f32) == 2:
            _last_launch(cout)
        ref, mag = ref_dgrad(dout, w, nbr_fwd, n_out_rows, x.shape[0])
        bref = ref_dgrad(_bf(dout), _bf(w), nbr_fwd, n_out_rows, x.shape[0])[0] if arm == "tf32" else None
        check_values(dx, ref, mag, arm, what + " dgrad", bf16_ref=bref)
        del ref, mag, bref
    ref, mag = ref_wgrad(x, dout, nbr_fwd, n_out_rows)
    bref = ref_wgrad(_bf(x), _bf(dout), nbr_fwd, n_out_rows)[0] if arm == "tf32" else None
    check_values(dw, ref, mag, arm, what + " wgrad", sums=True, bf16_ref=bref)
    d64 = dout.double()
    assert_sums(db, d64.sum(0), d64.abs().sum(0), "exact" if arm == "exact" else "rounding", what + " dbias")
    if atomic_wgrad and arm != "exact":          # fp32 atomics: a repeated weight gradient may differ in the last bits
        first, second = first[:1], second[:1]
    assert_repeat(first, second, what + " backward")


# ==================================================================================== probe


@pytest.mark.gpu
def test_probe_feature_rounding():
    """One live pair, W = 1 (exact in TF32), x = 1 + 2^-11 + 2^-12: 1 if the tensor cores drop the low 13 bits of an
    fp32 operand, 1 + 2^-10 if they round it to nearest, x itself if they used all of it."""
    from sparseeventid_b200.scn import ops
    prec = _prec()
    x = torch.zeros((1, 32), device="cuda")
    x[0, 0] = 1 + 2 ** -11 + 2 ** -12
    w = torch.zeros((1, 32, 32), device="cuda")
    w[0, 0, 0] = 1.0
    nbr = torch.full((1, 128), -1, dtype=torch.int32, device="cuda")
    nbr[0, 0] = 0
    assert ops.conv_path(1, 32, 32, prec, torch.float32) == 2
    out = module_forward(x, w, None, nbr, 1, prec, torch.float32)
    got = float(out[0, 0])
    seen = {1.0: "truncate", 1 + 2 ** -10: "round"}.get(got, f"other ({got!r})")
    print(f"\ntcgen05 kind::tf32 reads x = 1 + 2^-11 + 2^-12 as {got!r}: {seen}")
    assert seen == TF32_FEATURES
    # dout of the weight gradient goes through the same operand path
    dout = torch.zeros((1, 32), device="cuda")
    dout[0, 0] = 1 + 2 ** -11 + 2 ** -12
    xw = torch.zeros((1, 32), device="cuda")
    xw[0, 0] = 1.0
    dw = ops.conv_wgrad(xw, dout, nbr, 1, 32, 32, prec)
    assert float(dw[0, 0, 0]) == float(tf32_features(torch.tensor(1 + 2 ** -11 + 2 ** -12)))


# ==================================================================================== the benchmark's own tables


@pytest.fixture(scope="module")
def bench_tables():
    import sparseconvnet as scn
    from sparseeventid_b200 import synthetic
    coords, feats, bs = bench_batch()
    x = scn.InputLayer(3, list(synthetic.GRID_3D))((torch.as_tensor(coords).cuda(), torch.as_tensor(feats).cuda(), bs))
    md = x.metadata
    sp = tuple(synthetic.GRID_3D)
    levels = []
    for level in range(6):
        e = {"n": md.levels[sp].n, "subm": md.subm_table(sp, (3, 3, 3))}
        if level == 0:
            e["stem"] = md.subm_table(sp, (5, 5, 5))
        if level == 5:
            e["one"] = md.subm_table(sp, (1, 1, 1))
        else:
            e["rule"] = md.strided_rule(sp, (2, 2, 2), (2, 2, 2))
            sp = e["rule"].out_spatial
        levels.append(e)
    return levels


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("level", range(6))
def test_bench_level_submanifold(bench_tables, level, arm):
    e, c = bench_tables[level], CHANNELS[level]
    g = torch.Generator(device="cuda").manual_seed(100 + level)
    n = e["n"]
    x, dout = draw((n, c), arm, g), draw((n, c), arm, g)
    w, b = draw((27, c, c), arm, g), draw((c,), arm, g)
    check_layer(x, w, b, dout, e["subm"], e["subm"], n, True, arm, f"tf32 level {level} ({n} x {c}) 3^3")
    _done("bench")


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("level", range(5))
def test_bench_level_downsample(bench_tables, level, arm):
    e = bench_tables[level]
    rule, cin, cout = e["rule"], CHANNELS[level], CHANNELS[level + 1]
    g = torch.Generator(device="cuda").manual_seed(200 + level)
    x, dout = draw((e["n"], cin), arm, g), draw((rule.n_out, cout), arm, g)
    w = draw((8, cin, cout), arm, g)
    check_layer(x, w, None, dout, rule.down, rule.up, rule.n_out, False, arm,
                f"tf32 downsample {level} ({e['n']} -> {rule.n_out} rows, {cin} -> {cout})")
    _done("bench")


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ARMS)
def test_bench_stem(bench_tables, arm):
    """5^3 stem, one fp32 input channel -> 32 fp32 outputs (stem_tc.cu, hi/lo split of x, W and the fp32 dout): fp32
    accuracy, so the TF32-operand arm is held to the rounding arm's bars."""
    from sparseeventid_b200.scn import ops
    e = bench_tables[0]
    g = torch.Generator(device="cuda").manual_seed(300)
    n = e["n"]
    x, dout = draw((n, 1), arm, g), draw((n, 32), arm, g)
    w, b = draw((125, 1, 32), arm, g), draw((32,), arm, g)
    assert ops.conv_path(125, 1, 32, _prec(), torch.float32) == 0
    check_layer(x, w, b, dout, e["stem"], e["stem"], n, True, {"tf32": "split"}.get(arm, arm),
                f"tf32 stem 5^3 ({arm} operands)", need_dx=False, atomic_wgrad=True)


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ARMS)
def test_bench_bottleneck(bench_tables, arm):
    e = bench_tables[5]
    g = torch.Generator(device="cuda").manual_seed(400)
    n = e["n"]
    x, dout = draw((n, 192), arm, g), draw((n, 128), arm, g)
    w, b = draw((1, 192, 128), arm, g), draw((128,), arm, g)
    check_layer(x, w, b, dout, e["one"], e["one"], n, True, arm, "tf32 bottleneck 1^3 192 -> 128")


# ==================================================================================== forced launch configurations

# n_in = 32 c for c = 1..8 channel chunks per offset
SWEEP = [(32, 64, "subm"), (64, 32, "down"), (96, 96, "subm"), (128, 160, "down"), (160, 160, "subm"),
         (192, 224, "down"), (224, 96, "subm"), (256, 256, "subm")]
SA_SB = [(sa, sb) for sa in (4, 8, 12) for sb in (2, 3, 0)]


@pytest.fixture(scope="module")
def blob_tables():
    import sparseconvnet as scn
    grid = (64, 64, 64)
    coords = blob_sites(2000, grid, 2, seed=11)
    x = scn.InputLayer(3, list(grid))((torch.as_tensor(coords).cuda(), torch.ones(coords.shape[0], 1).cuda(), 2))
    md = x.metadata
    n = md.levels[grid].n
    rule = md.strided_rule(grid, (2, 2, 2), (2, 2, 2))
    return {"subm": (md.subm_table(grid, (3, 3, 3)), n, n), "down": (rule.down, rule.n_out, n)}


@pytest.mark.gpu
@pytest.mark.parametrize("n_in,n_out,table", SWEEP)
def test_forced_launch_configurations(blob_tables, knobs, n_in, n_out, table):
    """Every forced (grid, T) with one of the nine (SA, SB) each, exact arm; the other arms at grid 2."""
    from sparseeventid_b200.scn import ops
    prec = _prec()
    nbr, n_rows, n_src = blob_tables[table]
    K = nbr.shape[0]
    for arm in ARMS:
        g = torch.Generator(device="cuda").manual_seed(n_in * 1000 + n_out)
        x = draw((n_src, n_in), arm, g)
        w, b = draw((K, n_in, n_out), arm, g), draw((n_out,), arm, g)
        bimg = ops.prep_weights(w, False, False, prec, torch.float32)
        ref, mag = ref_forward(x, w, b, nbr, n_rows)
        bref = ref_forward(_bf(x), _bf(w), b, nbr, n_rows)[0] if arm == "tf32" else None
        i = 0
        for grid in ((1, 2, 3, 7) if arm == "exact" else (2,)):
            for t in range(1, 9):
                sa, sb = SA_SB[i % len(SA_SB)]
                knobs(grid, t, sa, sb)
                out = ops.conv_forward(x, nbr, n_rows, n_in, n_out, bimg, b, prec, torch.float32)
                again = ops.conv_forward(x, nbr, n_rows, n_in, n_out, bimg, b, prec, torch.float32)
                cfg = _last_launch(n_in)
                what = f"tf32 {n_in} -> {n_out}, K {K}, {n_rows} rows, forced grid {grid} T {t} SA {sa} SB {sb}: launched {cfg}"
                check_values(out, ref, mag, arm, what, bf16_ref=bref)
                assert_repeat(out, again, what)
                i += 1
    knobs(0, 0, 0, 0)
    _done("sweep")


# ==================================================================================== row-count edges, rectangles


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("c", [32, 96, 160])
@pytest.mark.parametrize("n", EDGE_ROWS)
def test_row_count_edges(n, c, arm):
    from sparseeventid_b200.scn import ops
    prec = _prec()
    g = torch.Generator(device="cuda").manual_seed(n + c)
    nbr = rand_table(27, n, n, 0.3, g)
    x, dout = draw((n, c), arm, g), draw((n, c), arm, g)
    w, b = draw((27, c, c), arm, g), draw((c,), arm, g)
    bimg = ops.prep_weights(w, False, False, prec, torch.float32)
    what = f"tf32 {n} rows x {c}"
    out = ops.conv_forward(x, nbr, n, c, c, bimg, b, prec, torch.float32)
    again = ops.conv_forward(x, nbr, n, c, c, bimg, b, prec, torch.float32)
    cfg = _last_launch(c)
    ref, mag = ref_forward(x, w, b, nbr, n)
    bref = ref_forward(_bf(x), _bf(w), b, nbr, n)[0] if arm == "tf32" else None
    check_values(out, ref, mag, arm, f"{what} forward, launched {cfg}", bf16_ref=bref)
    assert_repeat(out, again, what + " forward")
    dw, again = ops.conv_wgrad(x, dout, nbr, n, c, c, prec), ops.conv_wgrad(x, dout, nbr, n, c, c, prec)
    wcfg = _last_wgrad_launch(27, c, c)
    ref, mag = ref_wgrad(x, dout, nbr, n)
    bref = ref_wgrad(_bf(x), _bf(dout), nbr, n)[0] if arm == "tf32" else None
    check_values(dw, ref, mag, arm, f"{what} wgrad, launched {wcfg}", sums=True, bf16_ref=bref)
    assert_repeat(dw, again, what + " wgrad")
    _done("edges")


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("n_src,n_out", [(5000, 1300), (1300, 5000)])
@pytest.mark.parametrize("K,cin,cout", [(8, 64, 96), (27, 160, 64), (8, 32, 192), (27, 224, 128)])
def test_rectangular_tables(n_src, n_out, K, cin, cout, arm):
    from sparseeventid_b200.scn import ops
    prec = _prec()
    g = torch.Generator(device="cuda").manual_seed(n_src + 3 * n_out + K + cin)
    nbr = rand_table(K, n_out, n_src, 0.4, g)
    x, dout = draw((n_src, cin), arm, g), draw((n_out, cout), arm, g)
    w, b = draw((K, cin, cout), arm, g), draw((cout,), arm, g)
    bimg = ops.prep_weights(w, False, False, prec, torch.float32)
    what = f"tf32 {n_src} -> {n_out} rows, K {K}, {cin} -> {cout}"
    out = ops.conv_forward(x, nbr, n_out, cin, cout, bimg, b, prec, torch.float32)
    again = ops.conv_forward(x, nbr, n_out, cin, cout, bimg, b, prec, torch.float32)
    _last_launch(cin)
    ref, mag = ref_forward(x, w, b, nbr, n_out)
    bref = ref_forward(_bf(x), _bf(w), b, nbr, n_out)[0] if arm == "tf32" else None
    check_values(out, ref, mag, arm, what + " forward", bf16_ref=bref)
    assert_repeat(out, again, what + " forward")
    dw, again = ops.conv_wgrad(x, dout, nbr, n_out, cin, cout, prec), ops.conv_wgrad(x, dout, nbr, n_out, cin, cout, prec)
    _last_wgrad_launch(K, cin, cout)
    ref, mag = ref_wgrad(x, dout, nbr, n_out)
    bref = ref_wgrad(_bf(x), _bf(dout), nbr, n_out)[0] if arm == "tf32" else None
    check_values(dw, ref, mag, arm, what + " wgrad", sums=True, bf16_ref=bref)
    assert_repeat(dw, again, what + " wgrad")


# ==================================================================================== every TF32 k_wgrad_tc instantiation

# (Cin, Cout) -> 32-channel blocks (nca, ncb) and pairs per stage (64 up to 4 blocks, 32 up to 9, 16 beyond); Cin
# covers M blocks of 1..4 blocks (the partial last M block of 96, 160, 192 and 224 channels)
WG_CHANNELS = [(32, 32), (64, 64), (96, 32), (32, 128), (96, 96), (160, 64), (128, 160), (96, 192), (160, 160),
               (224, 96), (64, 256), (192, 128), (256, 256), (224, 224)]
WG_K = [1, 8, 27]
WG_REGIMES = ["one CTA per offset", "one wave", "two waves"]


def _wg_rows(K, regime):
    if regime == WG_REGIMES[0]:
        return 300
    per_cta = 200 if regime == WG_REGIMES[1] else 300
    return int(math.ceil(per_cta * 512 / (0.3 * K)))


WG_CASES = [(cc, K, WG_REGIMES[(i + j) % 3]) for i, cc in enumerate(WG_CHANNELS) for j, K in enumerate(WG_K)]


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("cc,K,regime", WG_CASES)
def test_wgrad_instantiations(cc, K, regime, arm):
    from sparseeventid_b200.scn import ops
    prec = _prec()
    cin, cout = cc
    n = _wg_rows(K, regime)
    g = torch.Generator(device="cuda").manual_seed(cin * 7 + cout + K + n)
    nbr = rand_table(K, n, n, 0.3, g)
    x, dout = draw((n, cin), arm, g), draw((n, cout), arm, g)
    what = f"tf32 wgrad {cin} x {cout}, K {K}, {n} rows ({regime})"
    dw, again = ops.conv_wgrad(x, dout, nbr, n, cin, cout, prec), ops.conv_wgrad(x, dout, nbr, n, cin, cout, prec)
    cfg = _last_wgrad_launch(K, cin, cout)
    assert (cfg["nca"], cfg["ncb"]) == (cin // 32, cout // 32), f"{what}: launched {cfg}"
    ref, mag = ref_wgrad(x, dout, nbr, n)
    bref = ref_wgrad(_bf(x), _bf(dout), nbr, n)[0] if arm == "tf32" else None
    check_values(dw, ref, mag, arm, f"{what}: launched {cfg}", sums=True, bf16_ref=bref)
    assert_repeat(dw, again, what)
    _done("wgrad")


# ==================================================================================== batched weight images


@pytest.mark.gpu
def test_batched_images_match_per_module_images():
    """scn_conv_prep_weights_batched builds byte-identical TF32 images (forward and mirrored / plain dgrad)."""
    import sparseconvnet as scn
    from sparseeventid_b200 import _lib as L
    from sparseeventid_b200.scn import functional as F
    from sparseeventid_b200.scn import ops
    scn.set_precision("tf32")
    prec = _prec()
    torch.manual_seed(3)
    mods = [scn.SubmanifoldConvolution(3, 32, 64, 3, True), scn.Convolution(3, 64, 96, 2, 2, False),
            scn.SubmanifoldConvolution(3, 160, 160, 3, False), scn.Convolution(3, 224, 256, 2, 2, False),
            scn.SubmanifoldConvolution(3, 1, 32, 5, True), scn.SubmanifoldConvolution(3, 256, 32, 1, False)]
    for m in mods:
        m.cuda()
    try:
        assert F.prepare_weight_images(mods) == 2 * 5          # the stem has no tcgen05 image
        for m in mods:
            w = m.weight
            K, cin, cout = w.shape[0], w.shape[-2], w.shape[-1]
            ws = m.workspace(K, cin, cout, prec, torch.float32, w.device)
            if ws.path != 2:
                continue
            w3 = w.detach().view(K, cin, cout)
            want_f = ops.prep_weights(w3, False, False, prec, torch.float32)
            want_b = ops.prep_weights(w3, True, m.mirror_dgrad, prec, torch.float32)
            assert want_f.numel() == K * cin * cout * 4
            assert torch.equal(ws.fwd, want_f), f"{m}: forward image"
            assert torch.equal(ws.bwd_buffer(K, cin, cout, prec, torch.float32, w.device), want_b), f"{m}: dgrad image"
            # the image holds TF32 values: W rounded to nearest
            assert torch.equal(torch.sort(want_f.view(torch.float32))[0], torch.sort(tf32_round(w3).flatten())[0])
    finally:
        F.release_weight_images()
        scn.set_precision("bf16")


# ==================================================================================== coverage of the launchers


@pytest.mark.gpu
def test_launches_reached_every_launcher_branch():
    want = {"bench": 3 * 11, "sweep": len(SWEEP), "edges": 3 * 3 * len(EDGE_ROWS), "wgrad": 3 * len(WG_CASES)}
    if any(_DONE.get(k, 0) < v for k, v in want.items()):
        pytest.skip(f"needs the whole file to have passed first: {_DONE} of {want}")
    cfgs = [c for _, c in _LAUNCHES]

    def groups(c):
        return -(-c["max_tiles"] // c["T"])

    plain = [c for c in cfgs if not c["ksplit"]]
    assert {1, 2, 4} <= {c["NM"] for c in cfgs}, "NM"
    for nbuf in (1, 2):
        assert any(c["nbuf"] == nbuf and groups(c) >= 3 for c in plain), f"nbuf {nbuf} with >= 3 groups per CTA"
    assert any(c["max_tiles"] % c["T"] or c["min_tiles"] % c["T"] for c in plain), "a partial last group"
    assert any(c["ksplit"] and c["min_tiles"] == 1 and c["max_tiles"] == 2 for c in cfgs), "a mixed K-split launch"
    assert any(c["SB"] == 2 for c in cfgs), "SB = 2"
    assert set(range(1, 9)) <= {n_in // 32 for n_in, _ in _LAUNCHES}, "chunks per offset 1..8"
    wg = _WG_LAUNCHES
    assert {16, 32, 64} <= {c["pairs"] for *_, c in wg}, "every TF32 wgrad instantiation"
    for pairs in (16, 32, 64):
        mine = [(K, c) for K, _, _, c in wg if c["pairs"] == pairs]
        assert any(K > 1 and c["grid"] == K for K, c in mine), f"{pairs} pairs: one CTA per offset"
        assert any(K < c["grid"] <= 148 for K, c in mine), f"{pairs} pairs: one wave"
        assert any(c["grid"] > 148 for _, c in mine), f"{pairs} pairs: two waves"
    assert set(range(1, 9)) <= {c["nca"] for *_, c in wg} and set(range(1, 9)) <= {c["ncb"] for *_, c in wg}


# ==================================================================================== whole network


GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _run_network(scn_mod, device):
    from sparseeventid_b200 import networks, synthetic
    enc, head = networks.build_networks(scn_mod, "dune3d")
    model = networks.EventIDModel(enc, head)
    init_deterministic(model)
    model.to(device)
    model.train()
    head.eval()
    coords, feats, bs = small_batch("dune3d")
    labels = {k: torch.as_tensor(v).to(device) for k, v in synthetic.make_labels(2, seed=11).items()}
    encoded = enc((torch.as_tensor(coords).to(device), torch.as_tensor(feats).to(device), bs))
    logits = head(encoded)
    loss = networks.focal_loss(labels, logits)
    loss.backward()
    out = {"loss": float(loss.detach()), "enc_pooled": encoded.detach().double().mean(dim=(2, 3, 4)).cpu().numpy(),
           "grad_norms": np.asarray([float(p.grad.double().norm()) for _, p in model.named_parameters()])}
    for k, v in logits.items():
        out["logits_" + k] = v.detach().double().cpu().numpy()
    return out


@pytest.mark.gpu
def test_network_tf32_vs_truth_and_mixed():
    """dune3d default encoder + heads: loss / logits within 2e-3 of truth; encoder output and gradient norms no further
    from truth than 1.5 x the oracle under TF32 operands (+ the floors of test_golden_network.py); and closer to truth
    than the "mixed" mode (bf16 operands) on the encoder output and the median gradient-norm error."""
    import sparseconvnet as scn
    fx = np.load(os.path.join(GOLDEN, "dune3d_default_encoder.npz"), allow_pickle=False)
    try:
        scn.set_precision("tf32")
        got = _run_network(scn, "cuda")
        scn.set_precision("mixed")
        mixed = _run_network(scn, "cuda")
    finally:
        scn.set_precision("bf16")
    with tf32_numerics():
        want = _run_network(oscn, "cpu")

    def rel(a, b):
        a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
        return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-6))

    errs = {"loss": rel(got["loss"], fx["loss"])}
    errs.update({k: rel(got[k], fx[k]) for k in fx.files if k.startswith("logits_")})
    for k, e in errs.items():
        assert e <= 2e-3, f"tf32 vs truth: {k} relative error {e:.3e}"
    d_gpu, d_or, d_mixed = (rel(r["enc_pooled"], fx["enc_pooled"]) for r in (got, want, mixed))
    assert d_gpu <= 1.5 * d_or + 2e-3, f"tf32: encoder output {d_gpu:.3e} from truth, oracle[tf32] {d_or:.3e}"
    wn = np.asarray(fx["grad_norms"], dtype=np.float64)
    big = wn > 1e-3 * wn.max()
    e_gpu, e_or, e_mixed = (np.abs(np.asarray(r["grad_norms"]) - wn)[big] / wn[big] for r in (got, want, mixed))
    assert np.all(np.asarray(got["grad_norms"])[~big] < 1e-2 * wn.max()), "near-zero gradients are not near zero"
    assert e_gpu.max() <= 1.5 * e_or.max() + 1e-2, f"tf32: worst grad norm {e_gpu.max():.3e} vs oracle {e_or.max():.3e}"
    assert np.median(e_gpu) <= 1.5 * np.median(e_or) + 2e-3, f"tf32: median grad norm {np.median(e_gpu):.3e}"
    print(f"\n[dune3d] distance from truth, tf32 gpu / oracle[tf32] / mixed gpu: encoder output {d_gpu:.2e} / {d_or:.2e} / "
          f"{d_mixed:.2e}; median grad norm {np.median(e_gpu):.2e} / {np.median(e_or):.2e} / {np.median(e_mixed):.2e}; "
          f"loss/logits {errs}")
    assert d_gpu < d_mixed, f"tf32 encoder output {d_gpu:.3e} not closer to truth than mixed {d_mixed:.3e}"
    assert np.median(e_gpu) < np.median(e_mixed), "tf32 median gradient-norm error not below mixed"


@pytest.mark.gpu
def test_bench_batch_training_step_tf32():
    """One step on the benchmark batch against the float64 oracle (bars relative to the oracle under TF32 operands),
    then 20 Trainer steps in the tf32 mode with finite losses."""
    import sparseconvnet as scn
    from test_bench_scale_parity import BATCH, SEED, TOL, _dist, _step
    from sparseeventid_b200 import synthetic
    from sparseeventid_b200.trainer import Trainer
    coords, feats, bs = bench_batch()
    labels = synthetic.make_labels(BATCH, seed=SEED)
    oscn.set_numerics("fp32")
    truth = _step(oscn, "cpu", torch.float64, coords, feats, bs, labels)
    with tf32_numerics():
        o_tf32 = _dist(_step(oscn, "cpu", torch.float32, coords, feats, bs, labels), truth)
    try:
        scn.set_precision("tf32")
        g = _dist(_step(scn, "cuda", torch.float32, coords, feats, bs, labels), truth)
        r = np.asarray(list(g["grad_rel"].values()))
        print(f"\nbatch-{BATCH} tf32 step vs float64 oracle: loss {g['loss']:.1e} logits {g['logits']:.1e} pooled "
              f"{g['pooled']:.1e} grad rel-L2 median {np.median(r):.1e} max {r.max():.1e}; oracle[tf32] pooled "
              f"{o_tf32['pooled']:.1e} grad rel-L2 max {max(o_tf32['grad_rel'].values()):.1e}")
        assert g["loss"] <= TOL and g["logits"] <= TOL
        assert g["pooled"] <= 1.5 * o_tf32["pooled"] + 1e-3
        for n, e in g["grad_rel"].items():
            assert e <= 1.5 * o_tf32["grad_rel"][n] + 5e-2, f"tf32 gradient of {n}: {e:.3e} vs oracle {o_tf32['grad_rel'][n]:.3e}"
            assert g["grad_cos"][n] >= o_tf32["grad_cos"][n] - 0.05, f"tf32 gradient direction of {n}"
        trainer = Trainer(scn, "dune3d", device=torch.device("cuda"), seed=0)
        batch = (torch.as_tensor(coords).cuda(), torch.as_tensor(feats).cuda(), bs)
        lab = {k: torch.as_tensor(v).cuda() for k, v in labels.items()}
        losses = [float(trainer.step(batch, lab)) for _ in range(20)]
        assert all(math.isfinite(v) for v in losses), losses
    finally:
        scn.set_precision("bf16")
