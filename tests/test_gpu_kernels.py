"""Direct checks of the convolution kernels through the C ABI.

The first two tests compare the tcgen05 kernels (`scn_conv_forward`, csrc/conv_tc.cu; `scn_conv_wgrad`,
csrc/wgrad_tc.cu) with a plain torch fp32 gather + matmul of the SAME bf16 operands at shapes the layer tests do not
reach: row counts that are not multiples of 128, a single offset, tables without any pair, Cin != Cout, 160 / 192 / 256
channels, several CTAs per offset.  Tolerance 2e-3 relative to the largest element.

The rest hold every convolution kernel to a float64 reference of the same operation (gather / mm / index_add_ over the
pairs of the FORWARD table; dgrad is checked against the true transpose) in two arms:
  * exact: x, dout, W and bias are small integers held in bf16, so every product and partial sum is an integer far below
    2^24 and fp32 adds it exactly in any order or split.  dW must equal the reference bit for bit; bf16 outputs must
    equal the reference rounded once to nearest even.  One dropped pair, wrong row, stale accumulator or lost partial
    group fails, where a tolerance relative to the largest element would hide it.  The precondition A < 2^24 (A = the
    sum of the magnitudes of an element's terms) is asserted, not assumed.  (Tensor-core fp32 accumulation is taken to
    be exact on such integers; if a case fails, compare with the exact FMA path "fp32" before suspecting the kernel.)
  * rounding: N(0,1) values rounded to bf16, element by element
        forward / dx:  |got - ref| <= 2^-8 |ref| + 2^-16 A        dW:  |got - ref| <= 2^-14 A
    (one bf16 output rounding plus fp32 accumulation; catches operands narrowed below bf16, which integers cannot).
Cases: the benchmark batch's real tables at all six levels (3^3 submanifold, the five 2^3 downsamples, the 5^3 stem, the
K = 1 bottleneck) through the entry points the layers call; a forced launch-configuration sweep (scn_tc_debug_knobs);
row counts at the tile and wave edges; rectangular tables; every k_wgrad_tc instantiation; the mma.sync and exact FMA
paths.  Every launch runs twice and must be bit-identical (DESIGN 4.1, 4.2), except the weight gradients that finish
with fp32 atomics (stem, mma.sync and FMA paths) in the rounding arm.  The last test asserts that the launches reached
every launcher branch they are meant to pin (scn_tc_debug_last_launch / scn_wgrad_debug_last_launch).
"""
import ctypes
import math

import pytest
import torch

from helpers import bench_batch, blob_sites

SHAPES = [(1, 1, 32, 32), (200, 1, 64, 64), (129, 3, 64, 32), (1000, 27, 32, 32), (3000, 27, 64, 96), (2500, 27, 96, 96),
          (2000, 27, 128, 128), (1500, 27, 160, 160), (1500, 27, 192, 192), (1200, 8, 160, 192), (900, 27, 256, 256),
          (70000, 27, 64, 64), (40000, 8, 32, 64)]


def make(n, K, cin, cout, density, seed):
    from sparseeventid_b200.scn import ops
    g = torch.Generator(device="cuda").manual_seed(seed)
    n_pad = ops.pad128(n)
    nbr = torch.full((K, n_pad), -1, dtype=torch.int32, device="cuda")
    mask = torch.rand(K, n, device="cuda", generator=g) < density
    idx = torch.randint(0, n, (K, n), device="cuda", dtype=torch.int32, generator=g)
    nbr[:, :n] = torch.where(mask, idx, torch.full_like(idx, -1))
    x = torch.randn(n, cin, device="cuda", generator=g).bfloat16()
    d = torch.randn(n, cout, device="cuda", generator=g).bfloat16()
    w = (torch.randn(K, cin, cout, device="cuda", generator=g) / cin ** 0.5).bfloat16().float().contiguous()
    return nbr, x, d, w


@pytest.mark.gpu
@pytest.mark.parametrize("density", [0.3, 0.0, 1.0])
@pytest.mark.parametrize("n,K,cin,cout", SHAPES)
def test_wgrad_kernel_matches_torch(n, K, cin, cout, density):
    from sparseeventid_b200 import _lib as L
    from sparseeventid_b200.scn import ops
    if density == 1.0 and n > 5000:
        pytest.skip("dense large case adds nothing")
    nbr, x, d, _ = make(n, K, cin, cout, density, seed=n + K)
    dw = ops.conv_wgrad(x, d, nbr, n, cin, cout, L.PREC_BF16)
    ref = torch.zeros(K, cin, cout, device="cuda")
    xf, df = x.float(), d.float()
    for k in range(K):
        j = nbr[k, :n].long()
        m = j >= 0
        if bool(m.any()):
            ref[k] = xf[j[m]].t() @ df[m]
    scale = float(ref.abs().max())
    if scale == 0.0:
        assert float(dw.abs().max()) == 0.0
    else:
        assert float((dw - ref).abs().max()) <= 2e-3 * scale


@pytest.mark.gpu
@pytest.mark.parametrize("density", [0.3, 0.0])
@pytest.mark.parametrize("n,K,cin,cout", SHAPES)
def test_forward_kernel_matches_torch(n, K, cin, cout, density):
    from sparseeventid_b200 import _lib as L
    from sparseeventid_b200.scn import ops
    nbr, x, _, w = make(n, K, cin, cout, density, seed=7 * n + K)
    bias = torch.randn(cout, device="cuda")
    bp = ops.prep_weights(w, False, False, L.PREC_BF16, torch.bfloat16)
    out = ops.conv_forward(x, nbr, n, cin, cout, bp, bias, L.PREC_BF16, torch.bfloat16)
    ref = bias.expand(n, cout).clone()
    xf = x.float()
    for k in range(K):
        j = nbr[k, :n].long()
        m = j >= 0
        if bool(m.any()):
            ref[m] += xf[j[m]] @ w[k]
    ref = ref.bfloat16().float()                     # the kernel stores bf16
    scale = float(ref.abs().max())
    # one bf16 ulp (2^-8 relative to the element) where fp32 summation order flips a rounding
    assert float((out.float() - ref).abs().max()) <= 2 ** -7 * scale
    assert float((out.float() - ref).norm() / ref.norm().clamp_min(1e-20)) <= 2e-3


# ==================================================================================== float64 references (CPU or GPU)


def _pairs(nbr, k, n_rows):
    """(input rows, output rows) of offset k of a [K, n_pad] table, as int64 index tensors."""
    j = nbr[k, :n_rows].long()
    o = torch.nonzero(j >= 0).squeeze(1)
    return j[o], o


def ref_forward(x, w, bias, nbr, n_out_rows):
    """out[o] = bias + sum_k x[nbr[k][o]] @ W[k] in float64, and A[o] = |bias| + sum_k |x[nbr[k][o]]| @ |W[k]|."""
    x64, w64 = x.double(), w.double()
    out = torch.zeros(n_out_rows, w.shape[2], dtype=torch.float64, device=x.device)
    mag = torch.zeros_like(out)
    if bias is not None:
        out += bias.double()
        mag += bias.double().abs()
    for k in range(nbr.shape[0]):
        i, o = _pairs(nbr, k, n_out_rows)
        g = x64[i]
        out.index_add_(0, o, g @ w64[k])
        mag.index_add_(0, o, g.abs() @ w64[k].abs())
    return out, mag


def ref_dgrad(dout, w, nbr, n_out_rows, n_in_rows):
    """dx[i] = sum over the pairs (i, o) of offset k of the FORWARD table of dout[o] @ W[k]^T, in float64, and A."""
    d64, w64 = dout.double(), w.double()
    dx = torch.zeros(n_in_rows, w.shape[1], dtype=torch.float64, device=dout.device)
    mag = torch.zeros_like(dx)
    for k in range(nbr.shape[0]):
        i, o = _pairs(nbr, k, n_out_rows)
        g = d64[o]
        dx.index_add_(0, i, g @ w64[k].t())
        mag.index_add_(0, i, g.abs() @ w64[k].abs().t())
    return dx, mag


def ref_wgrad(x, dout, nbr, n_out_rows):
    """dW[k] = sum over the pairs (i, o) of offset k of x[i]^T dout[o], in float64, and A."""
    x64, d64 = x.double(), dout.double()
    K = nbr.shape[0]
    dw = torch.zeros(K, x.shape[1], dout.shape[1], dtype=torch.float64, device=x.device)
    mag = torch.zeros_like(dw)
    for k in range(K):
        i, o = _pairs(nbr, k, n_out_rows)
        dw[k] = x64[i].t() @ d64[o]
        mag[k] = x64[i].abs().t() @ d64[o].abs()
    return dw, mag


def _report(bad, got, ref, mag, what):
    idx = torch.nonzero(bad)[:6].tolist()
    rows = [f"  at {tuple(i)}: A={float(mag[tuple(i)]):.6g} ref={float(ref[tuple(i)]):.9g} got={float(got[tuple(i)]):.9g}"
            for i in idx]
    return f"{what}: {int(bad.sum())} of {bad.numel()} elements wrong\n" + "\n".join(rows)


def assert_features(got, ref, mag, arm, what):
    """Forward output / dx (bf16 or fp32) against the float64 reference."""
    assert got.shape == ref.shape, what
    if ref.numel() == 0:
        return
    if arm == "exact":
        assert float(mag.max()) < 2 ** 24, f"{what}: precondition A < 2^24 broken ({float(mag.max())})"
        bad = got != ref.float().to(got.dtype)
    else:
        bad = (got.double() - ref).abs() > 2 ** -8 * ref.abs() + 2 ** -16 * mag
    assert not bool(bad.any()), _report(bad, got, ref, mag, what)


def assert_sums(got, ref, mag, arm, what):
    """Weight / bias gradient (fp32) against the float64 reference."""
    assert got.shape == ref.shape, what
    if ref.numel() == 0:
        return
    if arm == "exact":
        assert float(mag.max()) < 2 ** 24, f"{what}: precondition A < 2^24 broken ({float(mag.max())})"
        bad = got.double() != ref
    else:
        bad = (got.double() - ref).abs() > 2 ** -14 * mag
    assert not bool(bad.any()), _report(bad, got, ref, mag, what)


def test_references_match_a_literal_triple_loop():
    """The float64 references above, pinned on a 7-row, K = 3 table against the definition written out as loops."""
    g = torch.Generator().manual_seed(5)
    n_in, n_out, K, cin, cout = 7, 5, 3, 3, 2
    nbr = torch.full((K, 128), -1, dtype=torch.int32)
    nbr[:, :n_out] = torch.tensor([[0, -1, 6, 2, -1], [1, 1, -1, 6, 0], [-1, 3, 4, 5, 6]], dtype=torch.int32)
    x = torch.randint(-3, 4, (n_in, cin), generator=g).double()
    d = torch.randint(-3, 4, (n_out, cout), generator=g).double()
    w = torch.randint(-3, 4, (K, cin, cout), generator=g).double()
    b = torch.randint(-3, 4, (cout,), generator=g).double()
    out, dx, dw = torch.zeros(n_out, cout), torch.zeros(n_in, cin), torch.zeros(K, cin, cout)
    aout, adx, adw = torch.zeros(n_out, cout), torch.zeros(n_in, cin), torch.zeros(K, cin, cout)
    for o in range(n_out):
        for n in range(cout):
            out[o, n], aout[o, n] = b[n], abs(b[n])
    for k in range(K):
        for o in range(n_out):
            i = int(nbr[k, o])
            if i < 0:
                continue
            for c in range(cin):
                for n in range(cout):
                    t = float(x[i, c] * w[k, c, n])
                    out[o, n] += t
                    aout[o, n] += abs(t)
                    t = float(d[o, n] * w[k, c, n])
                    dx[i, c] += t
                    adx[i, c] += abs(t)
                    t = float(x[i, c] * d[o, n])
                    dw[k, c, n] += t
                    adw[k, c, n] += abs(t)
    for (got, a), (want, wa) in ((ref_forward(x, w, b, nbr, n_out), (out, aout)),
                                 (ref_dgrad(d, w, nbr, n_out, n_in), (dx, adx)),
                                 (ref_wgrad(x, d, nbr, n_out), (dw, adw))):
        assert torch.equal(got, want.double()) and torch.equal(a, wa.double())
    # the bars themselves: one wrong element fails either arm; a bf16-rounded exact result passes
    ref, mag = ref_forward(x, w, b, nbr, n_out)
    assert_features(ref.float().bfloat16(), ref, mag, "exact", "self")
    assert_features(ref.float().bfloat16(), ref, mag, "rounding", "self")
    wrong = ref.float().clone()
    wrong[3, 1] += 1.0
    for arm in ("exact", "rounding"):
        with pytest.raises(AssertionError):
            assert_features(wrong, ref, mag, arm, "self")
        with pytest.raises(AssertionError):
            assert_sums(wrong, ref, mag, arm, "self")


# ==================================================================================== GPU plumbing

ARMS = ["exact", "rounding"]
LAUNCH_FIELDS = ("grid", "T", "NM", "nbuf", "ksplit", "SA", "SB", "min_tiles", "max_tiles")
WG_FIELDS = ("grid", "s_other", "s_centre", "pairs", "slots", "nca", "ncb")
_LAUNCHES = []          # (n_in, {LAUNCH_FIELDS}) of every k_conv_tc launch of this file
_WG_LAUNCHES = []       # (K, Cin, Cout, {WG_FIELDS}) of every k_wgrad_tc launch
_DONE = {}              # feeding test -> completed cases (the coverage test needs the whole file)


def _done(name):
    _DONE[name] = _DONE.get(name, 0) + 1


def _lib():
    from sparseeventid_b200 import _lib as L
    lib = L.lib()
    # developer entries outside include/scn_b200.h (like tools/tc_sweep.py): declared here
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
    """Sets the (documented result-preserving) launch knobs of k_conv_tc; always back to automatic afterwards."""
    lib = _lib()
    yield lambda grid, t, sa, sb: lib.scn_tc_debug_knobs(grid, t, sa, sb)
    lib.scn_tc_debug_knobs(0, 0, 0, 0)


def draw(shape, arm, gen, dtype=torch.bfloat16):
    """Small integers {-2..2} (exact arm) or N(0,1) values, rounded to bf16; returned as `dtype`."""
    if arm == "exact":
        v = torch.randint(-2, 3, shape, device="cuda", generator=gen).float()
    else:
        v = torch.randn(shape, device="cuda", generator=gen)
    return v.bfloat16().to(dtype)


def rand_table(K, n_out, n_in, density, gen):
    """[K, pad128(n_out)] table of random input rows (-1 padded) whose last input row is referenced."""
    from sparseeventid_b200.scn import ops
    nbr = torch.full((K, ops.pad128(n_out)), -1, dtype=torch.int32, device="cuda")
    live = torch.rand(K, n_out, device="cuda", generator=gen) < density
    idx = torch.randint(0, n_in, (K, n_out), device="cuda", dtype=torch.int32, generator=gen)
    nbr[:, :n_out] = torch.where(live, idx, torch.full_like(idx, -1))
    nbr[K - 1, n_out - 1] = n_in - 1
    return nbr


def _twice(fn):
    """Runs fn twice on the same inputs: (first result, second result)."""
    return fn(), fn()


def assert_repeat(a, b, what):
    """The second launch on the same inputs gave the same bits (checked after the values, so a wrong kernel whose
    repeats differ is reported by what it got wrong)."""
    for u, v in zip(a if isinstance(a, tuple) else (a,), b if isinstance(b, tuple) else (b,)):
        if u is not None:
            assert torch.equal(u, v), f"{what}: a repeated launch gave different bits"


def module_forward(x, w, bias, nbr, n_out_rows, prec, dtype):
    from sparseeventid_b200.scn import ops
    K, cin, cout = w.shape
    wimg = torch.zeros((ops.conv_prep_bytes(K, cin, cout, prec, dtype),), dtype=torch.uint8, device="cuda")
    return ops.conv_module_forward(x, w, bias, nbr, n_out_rows, K, cin, cout, prec, dtype, wimg, False)


def module_backward(x, dout, w, nbr_fwd, nbr_bwd, n_out_rows, mirror, prec, need_dx=True):
    """-> (dx or None, dW, dbias) through the layers' one-call backward; dW / dbias start as NaN (zeroed by the call)."""
    from sparseeventid_b200.scn import ops
    K, cin, cout = w.shape
    wimg_t = None
    if need_dx:
        wimg_t = torch.zeros((ops.conv_prep_bytes(K, cout, cin, prec, x.dtype),), dtype=torch.uint8, device="cuda")
    dw = torch.full((K, cin, cout), float("nan"), device="cuda")
    db = torch.full((cout,), float("nan"), device="cuda")
    dx = ops.conv_module_backward(x, dout, w, nbr_fwd, nbr_bwd, n_out_rows, K, cin, cout, mirror, prec, wimg_t, False,
                                  need_dx, dw, True, db, False)
    return dx, dw, db


def check_layer(x, w, bias, dout, nbr_fwd, nbr_bwd, n_out_rows, mirror, arm, what, prec=None, need_dx=True,
                wgrad_atomics=False):
    """Forward, dgrad, wgrad and dbias of one layer through the module entry points, each launched twice."""
    from sparseeventid_b200 import _lib as L
    from sparseeventid_b200.scn import ops
    prec = L.PREC_BF16 if prec is None else prec
    dtype = dout.dtype
    K, cin, cout = w.shape
    tc = ops.conv_path(K, cin, cout, prec, dtype) == 2
    out, again = _twice(lambda: module_forward(x, w, bias, nbr_fwd, n_out_rows, prec, dtype))
    if tc:
        _last_launch(cin)
    ref, mag = ref_forward(x, w, bias, nbr_fwd, n_out_rows)
    assert_features(out, ref, mag, arm, what + " forward")
    assert_repeat(out, again, what + " forward")
    del ref, mag
    first, second = _twice(lambda: module_backward(x, dout, w, nbr_fwd, nbr_bwd, n_out_rows, mirror, prec, need_dx))
    dx, dw, db = first
    if need_dx:
        if ops.conv_path(K, cout, cin, prec, dtype) == 2:
            _last_launch(cout)                     # the dgrad (the weight gradient has its own kernel)
        ref, mag = ref_dgrad(dout, w, nbr_fwd, n_out_rows, x.shape[0])
        assert_features(dx, ref, mag, arm, what + " dgrad")
        del ref, mag
    ref, mag = ref_wgrad(x, dout, nbr_fwd, n_out_rows)
    assert_sums(dw, ref, mag, arm, what + " wgrad")
    d64 = dout.double()
    assert_sums(db, d64.sum(0), d64.abs().sum(0), arm, what + " dbias")
    if wgrad_atomics and arm == "rounding":       # fp32 atomics: a repeated weight gradient may differ in the last bits
        first, second = first[:1], second[:1]
    assert_repeat(first, second, what + " backward")


# ==================================================================================== the benchmark's own tables

CHANNELS = [32, 64, 96, 128, 160, 192]        # the default encoder's levels (n_initial_filters 32, additive growth)


@pytest.fixture(scope="module")
def bench_tables():
    """Level row counts and the real neighbour tables of the benchmark's first batch (test_bench_scale_parity holds
    them bit-exact against the oracle's rulebooks)."""
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
    """3^3 submanifold forward / dgrad (mirrored weights, same table) / wgrad / dbias at the level's real table."""
    e, c = bench_tables[level], CHANNELS[level]
    g = torch.Generator(device="cuda").manual_seed(100 + level)
    n = e["n"]
    x, dout = draw((n, c), arm, g), draw((n, c), arm, g)
    w, b = draw((27, c, c), arm, g, torch.float32), draw((c,), arm, g, torch.float32)
    check_layer(x, w, b, dout, e["subm"], e["subm"], n, True, arm, f"level {level} ({n} x {c}) 3^3")
    _done("bench")


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("level", range(5))
def test_bench_level_downsample(bench_tables, level, arm):
    """2^3 stride-2 convolution: forward over `down`, dgrad over `up` (W[k]^T), wgrad; no bias, like the encoder."""
    e = bench_tables[level]
    rule, cin, cout = e["rule"], CHANNELS[level], CHANNELS[level + 1]
    g = torch.Generator(device="cuda").manual_seed(200 + level)
    x, dout = draw((e["n"], cin), arm, g), draw((rule.n_out, cout), arm, g)
    w = draw((8, cin, cout), arm, g, torch.float32)
    check_layer(x, w, None, dout, rule.down, rule.up, rule.n_out, False, arm,
                f"downsample {level} ({e['n']} -> {rule.n_out} rows, {cin} -> {cout})")
    _done("bench")


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ARMS)
def test_bench_stem(bench_tables, arm):
    """5^3 stem, one fp32 input channel -> 32 (stem_tc.cu: hi/lo bf16 split of x and W): forward and wgrad."""
    e = bench_tables[0]
    g = torch.Generator(device="cuda").manual_seed(300)
    n = e["n"]
    x, dout = draw((n, 1), arm, g, torch.float32), draw((n, 32), arm, g)
    w, b = draw((125, 1, 32), arm, g, torch.float32), draw((32,), arm, g, torch.float32)
    check_layer(x, w, b, dout, e["stem"], e["stem"], n, True, arm, "stem 5^3", need_dx=False, wgrad_atomics=True)


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ARMS)
def test_bench_bottleneck(bench_tables, arm):
    """K = 1 bottleneck 192 -> 128 at the deepest level."""
    e = bench_tables[5]
    g = torch.Generator(device="cuda").manual_seed(400)
    n = e["n"]
    x, dout = draw((n, 192), arm, g), draw((n, 128), arm, g)
    w, b = draw((1, 192, 128), arm, g, torch.float32), draw((128,), arm, g, torch.float32)
    check_layer(x, w, b, dout, e["one"], e["one"], n, True, arm, "bottleneck 1^3 192 -> 128")


# ==================================================================================== forced launch configurations

# (n_in, n_out, table): "subm" = 3^3 submanifold table of ~3200 blob sites (K = 27, odd: PAIR's last stage holds one
# offset), "down" = its stride-2 table (K = 8, even; fewer output rows than input rows)
SWEEP = [(32, 32, "subm"), (32, 64, "down"), (32, 256, "subm"), (64, 64, "subm"), (64, 224, "down"), (96, 96, "subm"),
         (96, 32, "subm"), (128, 128, "subm"), (128, 160, "down"), (160, 160, "subm"), (160, 192, "subm"),
         (192, 192, "subm"), (192, 128, "down"), (224, 224, "subm"), (224, 96, "subm"), (256, 256, "subm"),
         (256, 64, "down")]
SA_SB = [(sa, sb) for sa in (4, 8, 12) for sb in (2, 3, 0)]     # SB 0: as deep as shared memory allows


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


def _sweep(blob_tables, knobs, n_in, n_out, table):
    """Every forced (grid, T) with three of the nine (SA, SB) each, exact arm, plus the rounding arm at grid 2."""
    from sparseeventid_b200 import _lib as L
    from sparseeventid_b200.scn import ops
    nbr, n_rows, n_src = blob_tables[table]
    K = nbr.shape[0]
    for arm in ARMS:
        g = torch.Generator(device="cuda").manual_seed(n_in * 1000 + n_out)
        x = draw((n_src, n_in), arm, g)
        w, b = draw((K, n_in, n_out), arm, g, torch.float32), draw((n_out,), arm, g, torch.float32)
        bimg = ops.prep_weights(w, False, False, L.PREC_BF16, torch.bfloat16)
        ref, mag = ref_forward(x, w, b, nbr, n_rows)
        i = 0
        for grid in ((1, 2, 3, 7) if arm == "exact" else (2,)):
            for t in range(1, 9):
                for j in range(3 if arm == "exact" else 1):
                    sa, sb = SA_SB[(i + 3 * j) % len(SA_SB)]
                    knobs(grid, t, sa, sb)
                    out, again = _twice(lambda: ops.conv_forward(x, nbr, n_rows, n_in, n_out, bimg, b, L.PREC_BF16,
                                                                 torch.bfloat16))
                    cfg = _last_launch(n_in)
                    what = f"{n_in} -> {n_out}, K {K}, {n_rows} rows, forced grid {grid} T {t} SA {sa} SB {sb}: launched {cfg}"
                    assert_features(out, ref, mag, arm, what)
                    assert_repeat(out, again, what)
                i += 1
    knobs(0, 0, 0, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("n_in,n_out,table", SWEEP)
def test_forced_launch_configurations(blob_tables, knobs, n_in, n_out, table):
    _sweep(blob_tables, knobs, n_in, n_out, table)
    _done("sweep")


# ==================================================================================== row-count edges, rectangles

EDGE_ROWS = [1, 127, 128, 129, 18944, 18945, 37888, 37889]      # 18 945 rows = 149 tiles: a mixed K-split launch at 160


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("c", [32, 96, 160])
@pytest.mark.parametrize("n", EDGE_ROWS)
def test_row_count_edges(n, c, arm):
    """Automatic configuration at the tile (128 rows) and wave (148 tiles) edges: forward and wgrad, square table."""
    from sparseeventid_b200 import _lib as L
    from sparseeventid_b200.scn import ops
    g = torch.Generator(device="cuda").manual_seed(n + c)
    nbr = rand_table(27, n, n, 0.3, g)
    x, dout = draw((n, c), arm, g), draw((n, c), arm, g)
    w, b = draw((27, c, c), arm, g, torch.float32), draw((c,), arm, g, torch.float32)
    bimg = ops.prep_weights(w, False, False, L.PREC_BF16, torch.bfloat16)
    what = f"{n} rows x {c}"
    out, again = _twice(lambda: ops.conv_forward(x, nbr, n, c, c, bimg, b, L.PREC_BF16, torch.bfloat16))
    cfg = _last_launch(c)
    ref, mag = ref_forward(x, w, b, nbr, n)
    assert_features(out, ref, mag, arm, f"{what} forward, launched {cfg}")
    assert_repeat(out, again, what + " forward")
    dw, again = _twice(lambda: ops.conv_wgrad(x, dout, nbr, n, c, c, L.PREC_BF16))
    wcfg = _last_wgrad_launch(27, c, c)
    ref, mag = ref_wgrad(x, dout, nbr, n)
    assert_sums(dw, ref, mag, arm, f"{what} wgrad, launched {wcfg}")
    assert_repeat(dw, again, what + " wgrad")
    _done("edges")


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("n_src,n_out", [(5000, 1300), (1300, 5000)])
@pytest.mark.parametrize("K,cin,cout", [(8, 64, 96), (27, 160, 64), (8, 32, 192), (27, 224, 128)])
def test_rectangular_tables(n_src, n_out, K, cin, cout, arm):
    """n_out != n_in (strided forward and deconvolution shapes), random table referencing the last input row."""
    from sparseeventid_b200 import _lib as L
    from sparseeventid_b200.scn import ops
    g = torch.Generator(device="cuda").manual_seed(n_src + 3 * n_out + K + cin)
    nbr = rand_table(K, n_out, n_src, 0.4, g)
    x, dout = draw((n_src, cin), arm, g), draw((n_out, cout), arm, g)
    w, b = draw((K, cin, cout), arm, g, torch.float32), draw((cout,), arm, g, torch.float32)
    bimg = ops.prep_weights(w, False, False, L.PREC_BF16, torch.bfloat16)
    what = f"{n_src} -> {n_out} rows, K {K}, {cin} -> {cout}"
    out, again = _twice(lambda: ops.conv_forward(x, nbr, n_out, cin, cout, bimg, b, L.PREC_BF16, torch.bfloat16))
    _last_launch(cin)
    ref, mag = ref_forward(x, w, b, nbr, n_out)
    assert_features(out, ref, mag, arm, what + " forward")
    assert_repeat(out, again, what + " forward")
    dw, again = _twice(lambda: ops.conv_wgrad(x, dout, nbr, n_out, cin, cout, L.PREC_BF16))
    _last_wgrad_launch(K, cin, cout)
    ref, mag = ref_wgrad(x, dout, nbr, n_out)
    assert_sums(dw, ref, mag, arm, what + " wgrad")
    assert_repeat(dw, again, what + " wgrad")


# ==================================================================================== every k_wgrad_tc instantiation

# (nca, ncb) = 64-channel blocks of Cin / Cout -> channels; includes the product's 128 -> 160 downsample (2, 3), the
# 192 -> 128 bottleneck (3, 2) and the legacy network's 192 -> 224 (3, 4); (0, 0) is the 32 x 32 pair instance
WG_CHANNELS = {(0, 0): (32, 32), (1, 1): (64, 64), (1, 2): (32, 128), (1, 3): (64, 160), (1, 4): (64, 256),
               (2, 1): (128, 32), (2, 2): (96, 96), (2, 3): (128, 160), (2, 4): (96, 224),
               (3, 1): (160, 64), (3, 2): (192, 128), (3, 3): (160, 192), (3, 4): (192, 224),
               (4, 1): (256, 32), (4, 2): (224, 96), (4, 3): (256, 160), (4, 4): (224, 256)}
WG_K = [1, 4, 8, 9, 27]
WG_REGIMES = ["one CTA per offset", "one wave", "two waves"]


def _wg_rows(K, regime):
    """Rows of a density-0.3 table for which the launcher picks K CTAs / one wave of 148 / two waves (wgrad_tc.cu:
    ~0.3 K n / 512 pairs per CTA, one wave from 148 CTAs' worth, two from 0.85 x 296)."""
    if regime == WG_REGIMES[0]:
        return 300
    per_cta = 200 if regime == WG_REGIMES[1] else 300
    return int(math.ceil(per_cta * 512 / (0.3 * K)))


WG_CASES = [(ab, K, WG_REGIMES[(i + j) % 3]) for i, ab in enumerate(WG_CHANNELS) for j, K in enumerate(WG_K)]


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("ab,K,regime", WG_CASES)
def test_wgrad_instantiations(ab, K, regime, arm):
    from sparseeventid_b200 import _lib as L
    from sparseeventid_b200.scn import ops
    cin, cout = WG_CHANNELS[ab]
    n = _wg_rows(K, regime)
    g = torch.Generator(device="cuda").manual_seed(cin * 7 + cout + K + n)
    nbr = rand_table(K, n, n, 0.3, g)
    x, dout = draw((n, cin), arm, g), draw((n, cout), arm, g)
    what = f"wgrad {cin} x {cout}, K {K}, {n} rows ({regime})"
    dw, again = _twice(lambda: ops.conv_wgrad(x, dout, nbr, n, cin, cout, L.PREC_BF16))
    cfg = _last_wgrad_launch(K, cin, cout)
    assert (cfg["nca"], cfg["ncb"]) == ((1, 1) if ab == (0, 0) else ab), f"{what}: launched {cfg}"
    ref, mag = ref_wgrad(x, dout, nbr, n)
    assert_sums(dw, ref, mag, arm, f"{what}: launched {cfg}")
    assert_repeat(dw, again, what)
    _done("wgrad")


# ==================================================================================== mma.sync and exact FMA paths


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("mode", ["mixed", "fp32"])
@pytest.mark.parametrize("cin,cout", [(32, 64), (96, 96), (160, 32), (256, 128)])
def test_other_paths(blob_tables, cin, cout, mode, arm):
    """fp32 features: "mixed" runs mma.sync on bf16 operands, "fp32" the exact FMA kernels (submanifold table, mirrored
    dgrad).  Their weight gradients finish with fp32 atomics."""
    from sparseeventid_b200 import _lib as L
    from sparseeventid_b200.scn import ops
    prec = L.PREC_FP32 if mode == "fp32" else L.PREC_BF16
    assert ops.conv_path(27, cin, cout, prec, torch.float32) == (0 if mode == "fp32" else 1)
    nbr, n, _ = blob_tables["subm"]
    g = torch.Generator(device="cuda").manual_seed(cin + 5 * cout)
    x, dout = draw((n, cin), arm, g, torch.float32), draw((n, cout), arm, g, torch.float32)
    w, b = draw((27, cin, cout), arm, g, torch.float32), draw((cout,), arm, g, torch.float32)
    check_layer(x, w, b, dout, nbr, nbr, n, True, arm, f"{mode} 3^3 {cin} -> {cout}", prec=prec, wgrad_atomics=True)


# ==================================================================================== coverage of the launchers


@pytest.mark.gpu
def test_launches_reached_every_launcher_branch():
    """The launches above reached each configuration the kernels' group / buffer / class / K-split logic has."""
    want = {"bench": 22, "sweep": len(SWEEP), "edges": 2 * 3 * len(EDGE_ROWS), "wgrad": 2 * len(WG_CASES)}
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
    assert {4, 8, 12} <= {c["SA"] for c in cfgs}, "SA"
    nch = {(-(-n_in // 64), n_in == 32) for n_in, _ in _LAUNCHES}
    assert {(1, True), (1, False), (2, False), (3, False), (4, False)} <= nch, f"NCH with / without pairing: {nch}"
    wg = _WG_LAUNCHES
    assert {(a, b) for a in range(1, 5) for b in range(1, 5)} <= {(c["nca"], c["ncb"]) for *_, c in wg}
    assert any(K > 1 and c["grid"] == K for K, *_, c in wg), "one CTA per offset"
    assert any(K < c["grid"] <= 148 for K, *_, c in wg), "one wave"
    assert any(c["grid"] > 148 for *_, c in wg), "two waves"
    assert {32, 64} <= {c["pairs"] for *_, c in wg}, "32- and 64-pair stages"
