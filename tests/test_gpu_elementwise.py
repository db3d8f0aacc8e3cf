"""Direct checks of the bandwidth-bound kernels of csrc/elementwise.cu through the C ABI, against float64 references.

BatchNorm (forward, backward, fused column sums of dx) and the column sums (`scn_col_sum`) run in two arms.  Every bar
is per element, or per channel for statistics and sums; none is relative to the largest element or to a norm.
  * exact: x and dout are integers in [-8, 8] (exact in bf16 and fp32), gamma in {0.5, 1, 2}, beta = 0, leak in
    {1, 0.5}.  Preconditions, asserted from the grid and rows per block of the launch record: every fp32 partial sum
    of (x - pivot), (x - pivot)^2 and of the masked dout stays below 2^24 (so the fp64 accumulators hold the exact sums),
    and with leak != 1 no channel's mean lies within 1e-3 of an integer (so the leaky mask, the sign of
    fmaf(x, sc, sh), is the float64 sign).  Then save_mean, save_invstd, running_mean and running_var equal the float64
    values within 1 fp32 ulp (this checks that the Newton-refined rsqrt is correct to fp32 rounding), dbeta is bit-exact,
    and a repeated call gives identical bits.
  * rounding: N(mu, sigma^2) with mu / sigma in {0, 10, 100}, and a case whose pivot (row 0) sits 30 sigma from the mean;
    leak 0.333, generic gamma and beta.  With u = 2^-24, L the length of the longest fp32 addition chain a column sum
    goes through (rows per thread + block partials, read from the launch record) and gamma_L = (L + 4) u:
        sums (dbeta, dgamma, column sums):  |got - ref| <= gamma_L sum|terms| (+ the error of xhat for dgamma)
        statistics: Sum d and Sum d^2 (d = x - pivot) carry gamma_L sum|d| and gamma_L sum d^2, so
            |mean err| <= gamma_L sum|d| / n,  |var err| <= gamma_L (sum d^2 + 2 |s1| sum|d|) / n;
            sum d^2 / n = var + (pivot - mean)^2: the pivot's distance enters the variance bar squared
        forward out:  |got - ref| <= 2^-21 (|x sc| + |m sc| + |beta|) + one output rounding
        dx:           |got - ref| <= 2^-21 A + |sc| (dbeta bar + |xhat| dgamma bar) / n + one output rounding,
                      A = |sc d| + |x e2| + |m e2| + |sc s1|  (sc = gamma invstd, e2 = sc s2 invstd)
    Elements whose y = xhat gamma + beta lies within the fold error of 0 may take either side of the leaky mask; the
    bars add what that flip changes.  The references use the kernel's own saved mean / invstd, so the forward and the
    backward are checked apart from the statistics.
Data movement is bit-exact: LeakyReLU, AddTable + LeakyReLU (8-, 4- and 1-wide paths), the fp32 -> bf16 convert (ties,
+-0, subnormals, the largest finite value, overflow; NaN stays NaN), scatter-add and the InputLayer (integer features,
duplicates; the mean is a correctly rounded fp32 division), AveragePooling rows (integer features, scales 1/8 and
1/4, V = 4 and V = 1) and SparseToDense (sites outside the volume dropped forward, zero backward).  Deterministic
kernels must repeat bit for bit.  The last test asserts that the launches reached every launcher branch
(scn_ew_debug_last_launch).
"""
import ctypes
import math

import numpy as np
import pytest
import torch

from helpers import bench_batch

U = 2.0 ** -24
EPS = float(np.float32(1e-4))
MOM = float(np.float32(0.9))
LEAK_R = float(np.float32(0.333))

# ==================================================================================== float64 references (CPU or GPU)


def ref_bn_stats(x, training, rm, rv, eps=EPS, momentum=MOM):
    """-> dict(mean, var (biased), invstd, running_mean, running_var) in float64, SCN conventions (unbiased running
    variance with divisor max(n - 1, 1); running = momentum * running + (1 - momentum) * batch)."""
    rm64, rv64 = rm.double(), rv.double()
    if not training:
        return dict(mean=rm64, var=rv64, invstd=1.0 / torch.sqrt(rv64 + eps), running_mean=rm64, running_var=rv64)
    n = x.shape[0]
    x64 = x.double()
    mean = x64.mean(0)
    var = ((x64 - mean) ** 2).mean(0)
    unbiased = var * n / max(n - 1, 1)
    return dict(mean=mean, var=var, invstd=1.0 / torch.sqrt(var + eps),
                running_mean=momentum * rm64 + (1 - momentum) * mean,
                running_var=momentum * rv64 + (1 - momentum) * unbiased)


def ref_bn_forward(x, mean, invstd, gamma, beta, leak):
    """-> (out, y) in float64 from the given statistics: y = (x - mean) invstd gamma + beta, out = leaky(y)."""
    y = (x.double() - mean.double()) * invstd.double() * gamma.double() + beta.double()
    return torch.where(y > 0, y, y * leak), y


def ref_bn_backward(x, dout, mean, invstd, gamma, beta, leak, training):
    """-> dict(dx, dgamma, dbeta, dd, xh, y) in float64 from the given (saved) statistics."""
    n = x.shape[0]
    m, s = mean.double(), invstd.double()
    g = gamma.double()
    xh = (x.double() - m) * s
    y = xh * g + beta.double()
    dd = torch.where(y > 0, dout.double(), dout.double() * leak)
    dbeta, dgamma = dd.sum(0), (dd * xh).sum(0)
    if training:
        dx = g * s * (dd - dbeta / n - xh * dgamma / n)
    else:
        dx = g * s * dd
    return dict(dx=dx, dgamma=dgamma, dbeta=dbeta, dd=dd, xh=xh, y=y)


def ulp32(v):
    """fp32 ulp of float64 values (2^-149 floor)."""
    _, e = torch.frexp(v.double().abs())
    return torch.ldexp(torch.ones_like(v, dtype=torch.float64), (e - 24).clamp_min(-149))


def out_unit(dtype):
    """Bound on one rounding to `dtype` relative to the value: half a bf16 ulp, or a whole fp32 ulp."""
    return 2.0 ** -8 if dtype == torch.bfloat16 else 2.0 ** -23


def _report(bad, got, ref, bar, what):
    idx = torch.nonzero(bad)[:6].tolist()
    rows = [f"  at {tuple(i)}: ref={float(ref[tuple(i)]):.9g} got={float(got[tuple(i)]):.9g} bar={float(bar[tuple(i)]):.3g}"
            for i in idx]
    return f"{what}: {int(bad.sum())} of {bad.numel()} wrong\n" + "\n".join(rows)


def assert_within(got, ref, bar, what):
    assert got.shape == ref.shape, what
    bad = ~((got.double() - ref).abs() <= bar)          # NaN fails
    assert not bool(bad.any()), _report(bad, got, ref, bar, what)


def assert_exact(got, ref, what):
    assert got.shape == ref.shape, what
    bad = ~(got.double() == ref)
    assert not bool(bad.any()), _report(bad, got, ref, torch.zeros_like(ref), what)


def fold_error(x, mean, invstd, gamma, beta):
    """Bound on the fp32 error of y = fmaf(x, sc, sh) (or ((x - m) is) g + b) against float64 at the same statistics."""
    sc = invstd.double() * gamma.double()
    return 2.0 ** -21 * ((x.double() * sc).abs() + (mean.double() * sc).abs() + beta.double().abs())


def chain_length(rec, n, C):
    """Longest fp32 addition chain of a column sum of the launch `rec` (fields of scn_ew_debug_last_launch) over n rows."""
    if rec["slices"]:                                     # k_col_reduce2: kRedRows = 256 rows per block
        cv = -(-(C // rec["vec"]) // rec["slices"])
        ry = 256 // cv
        return -(-256 // ry) + ry
    ry = 256 // (C // 8)                                  # two-launch kernels and k_col_sum_fused
    g = rec["grid"]
    return -(-n // (g * ry)) + max(8, ry) + 5


def rows_per_block(rec, n, C):
    if rec["slices"]:
        return 256
    ry = 256 // (C // 8)
    return -(-n // (rec["grid"] * ry)) * ry


def test_references_match_literal_loops():
    """The float64 references and bars above, pinned on a 5 x 3 case against the definitions written out as loops."""
    g = torch.Generator().manual_seed(3)
    n, C, leak = 5, 3, 0.5
    x = torch.randint(-4, 5, (n, C), generator=g).double()
    d = torch.randint(-4, 5, (n, C), generator=g).double()
    gamma, beta = torch.tensor([0.5, 1.0, 2.0]), torch.tensor([0.25, -0.5, 0.0])
    rm, rv = torch.tensor([0.1, -0.2, 0.3]), torch.tensor([1.5, 0.5, 2.0])
    st = ref_bn_stats(x, True, rm, rv)
    for c in range(C):
        col = [float(x[r, c]) for r in range(n)]
        mu = sum(col) / n
        var = sum((v - mu) ** 2 for v in col) / n
        assert math.isclose(float(st["mean"][c]), mu, rel_tol=1e-15, abs_tol=1e-15)
        assert math.isclose(float(st["var"][c]), var, rel_tol=1e-14)
        assert math.isclose(float(st["running_var"][c]), MOM * float(rv[c]) + (1 - MOM) * var * n / (n - 1), rel_tol=1e-14)
        inv = 1 / math.sqrt(var + EPS)
        out, _ = ref_bn_forward(x, st["mean"], st["invstd"], gamma, beta, leak)
        bw = ref_bn_backward(x, d, st["mean"], st["invstd"], gamma, beta, leak, True)
        xh = [(v - mu) * inv for v in col]
        y = [h * float(gamma[c]) + float(beta[c]) for h in xh]
        dd = [float(d[r, c]) if y[r] > 0 else float(d[r, c]) * leak for r in range(n)]
        db, dg = sum(dd), sum(a * h for a, h in zip(dd, xh))
        for r in range(n):
            assert math.isclose(float(out[r, c]), y[r] if y[r] > 0 else y[r] * leak, rel_tol=1e-13, abs_tol=1e-13)
            want = float(gamma[c]) * inv * (dd[r] - db / n - xh[r] * dg / n)
            assert math.isclose(float(bw["dx"][r, c]), want, rel_tol=1e-12, abs_tol=1e-12)
        assert math.isclose(float(bw["dbeta"][c]), db, abs_tol=1e-12)
        assert math.isclose(float(bw["dgamma"][c]), dg, rel_tol=1e-12, abs_tol=1e-12)
    one = ref_bn_stats(x[:1], True, rm, rv)                   # n = 1: divisor max(n - 1, 1)
    assert torch.equal(one["var"], torch.zeros(C, dtype=torch.float64))
    assert torch.allclose(one["running_var"], MOM * rv.double())
    ev = ref_bn_stats(x, False, rm, rv)
    assert torch.equal(ev["mean"], rm.double())
    # ulp32 and the bar helpers
    assert float(ulp32(torch.tensor([1.0]))) == 2.0 ** -23 and float(ulp32(torch.tensor([-3.0]))) == 2.0 ** -22
    ref = torch.tensor([1.0, 2.0], dtype=torch.float64)
    assert_within(torch.tensor([1.0, 2.0]), ref, torch.zeros(2, dtype=torch.float64), "self")
    with pytest.raises(AssertionError):
        assert_within(torch.tensor([1.0, float("nan")]), ref, torch.ones(2, dtype=torch.float64), "self")
    with pytest.raises(AssertionError):
        assert_exact(torch.tensor([1.0, 2.0 + 2 ** -20]), ref, "self")
    rec2 = {"slices": 0, "grid": 592, "vec": 8}
    assert chain_length(rec2, 495518, 32) == 14 + 64 + 5 and rows_per_block(rec2, 495518, 32) == 14 * 64
    assert chain_length({"slices": 2, "grid": 1, "vec": 8}, 10, 2056) == 256 + 1   # 129 groups per slice: RY = 1


# ==================================================================================== GPU plumbing

EW_RECORDS = ("bn_fwd", "bn_bwd", "col_sum", "elem", "pool")
EW_FIELDS = ("path", "vec", "apply", "avec", "grid", "grid2", "slices", "colsum")
_LAUNCHES = {k: [] for k in EW_RECORDS}     # (shape info, record) of every launch of this file
_DONE = {}


def _done(name):
    _DONE[name] = _DONE.get(name, 0) + 1


def _lib():
    from sparseeventid_b200 import _lib as L
    lib = L.lib()
    # developer entry outside include/scn_b200.h: declared here
    lib.scn_ew_debug_last_launch.argtypes = [ctypes.POINTER(ctypes.c_int32)]
    lib.scn_ew_debug_last_launch.restype = None
    return lib


def last_launch(kind, info=None):
    buf = (ctypes.c_int32 * (len(EW_RECORDS) * len(EW_FIELDS)))()
    _lib().scn_ew_debug_last_launch(buf)
    i = EW_RECORDS.index(kind) * len(EW_FIELDS)
    rec = dict(zip(EW_FIELDS, list(buf)[i:i + len(EW_FIELDS)]))
    _LAUNCHES[kind].append((info, rec))
    return rec


def exact_data(n, C, dtype, gen, leak):
    """x, dout integers in [-8, 8]; with leak != 1 no channel mean within 1e-3 of an integer (moved off by raising a
    seventh of the channel's entries below 8 by one; asserted by the caller's precondition)."""
    x = torch.randint(-8, 9, (n, C), device="cuda", generator=gen).float()
    if leak != 1.0 and n >= 3:
        k = n // 7 + 1
        for step in range(16):
            m = x.double().mean(0)
            bad = (m - m.round()).abs() <= 1.5e-3
            if not bool(bad.any()):
                break
            rows = torch.arange(step * k, (step + 1) * k, device="cuda") % n
            blk = x[rows]
            blk[:, bad] = torch.where(blk[:, bad] < 8, blk[:, bad] + 1, blk[:, bad])
            x[rows] = blk
    d = torch.randint(-8, 9, (n, C), device="cuda", generator=gen).float()
    gamma = torch.tensor([0.5, 1.0, 2.0], device="cuda")[torch.randint(0, 3, (C,), device="cuda", generator=gen)]
    return x.to(dtype), d.to(dtype), gamma, torch.zeros(C, device="cuda")


DISTS = {"mu0": (0.0, 0.0), "mu10": (10.0, 0.0), "mu100": (100.0, 0.0), "pivot30": (0.0, 30.0)}


def rounding_data(n, C, dtype, gen, dist):
    mu_s, pivot_s = DISTS[dist]
    sigma = 1.5
    x = torch.randn(n, C, device="cuda", generator=gen) * sigma + mu_s * sigma
    if pivot_s:
        x[0] = mu_s * sigma + pivot_s * sigma
    d = torch.randn(n, C, device="cuda", generator=gen).to(dtype)
    gamma = torch.rand(C, device="cuda", generator=gen) + 0.5
    beta = torch.randn(C, device="cuda", generator=gen) * 0.3
    return x.to(dtype), d, gamma, beta


def check_bn_forward(x, gamma, beta, rm, rv, training, leak, arm, what):
    """One forward call (twice in the exact arm) against the float64 reference; -> (stats [2, C], forward record)."""
    from sparseeventid_b200.scn import ops
    n, C = x.shape
    rm1, rv1 = rm.clone(), rv.clone()
    out, stats = ops.bn_forward(x, gamma, beta, rm1, rv1, training, EPS, MOM, leak)
    rec = last_launch("bn_fwd", (n, C, training, x.dtype))
    what = f"{what} forward [{rec}]"
    ref = ref_bn_stats(x, training, rm, rv)
    m, s = stats[0], stats[1]
    if not training:
        assert torch.equal(m, rm), what + ": eval save_mean is the running mean"
        assert_within(s, ref["invstd"], ulp32(ref["invstd"]), what + " eval save_invstd")
        assert torch.equal(rm1, rm) and torch.equal(rv1, rv), what + ": eval changed the running statistics"
    elif arm == "exact":
        rpb = rows_per_block(rec, n, C)
        assert 256 * rpb < 2 ** 24, f"{what}: precondition: a partial sum of (x - pivot)^2 can reach 2^24"
        for name, got, want in (("save_mean", m, ref["mean"]), ("save_invstd", s, ref["invstd"]),
                                ("running_mean", rm1, ref["running_mean"]), ("running_var", rv1, ref["running_var"])):
            assert_within(got, want, ulp32(want), f"{what} {name}")
    else:
        gam = (chain_length(rec, n, C) + 4) * U
        x64 = x.double()
        dlt = x64 - x64[0]
        s1 = dlt.sum(0) / n
        e_mean = gam * dlt.abs().sum(0) / n
        e_var = gam * ((dlt * dlt).sum(0) + 2 * s1.abs() * dlt.abs().sum(0)) / n
        var_eps = ref["var"] + EPS
        assert_within(m, ref["mean"], e_mean + ulp32(ref["mean"]), what + " save_mean")
        assert_within(s, ref["invstd"], ref["invstd"] * (0.51 * e_var / var_eps + 2.0 ** -22), what + " save_invstd")
        assert_within(rm1, ref["running_mean"], (1 - MOM) * e_mean + ulp32(ref["running_mean"]), what + " running_mean")
        assert_within(rv1, ref["running_var"], (1 - MOM) * e_var * n / max(n - 1, 1) + ulp32(ref["running_var"]),
                      what + " running_var")
    want, y = ref_bn_forward(x, m, s, gamma, beta, leak)
    err = fold_error(x, m, s, gamma, beta)
    amb = y.abs() <= err
    if arm == "exact" and leak != 1.0:
        assert not bool(amb.any()), f"{what}: precondition: an element's y is within the fold error of 0"
    bar = 1.01 * err + out_unit(x.dtype) * want.abs() + torch.where(amb, y.abs(), torch.zeros_like(y))
    assert_within(out, want, bar, what + " out")
    if arm == "exact":
        rm2, rv2 = rm.clone(), rv.clone()
        out2, stats2 = ops.bn_forward(x, gamma, beta, rm2, rv2, training, EPS, MOM, leak)
        for a, b, name in ((out, out2, "out"), (stats, stats2, "stats"), (rm1, rm2, "running_mean"), (rv1, rv2, "running_var")):
            assert torch.equal(a, b), f"{what}: a repeated call gave different bits ({name})"
    return stats, rec


def check_bn_backward(x, dout, gamma, beta, stats, training, leak, arm, what, colsum, acc_init=None):
    """One backward call (twice in the exact arm) against the float64 reference at the saved statistics.
    acc_init: (dgamma, dbeta) to accumulate into (accumulate = 1)."""
    from sparseeventid_b200.scn import ops
    n, C = x.shape
    kw = {}
    if acc_init is not None:
        kw = dict(dgamma=acc_init[0].clone(), dbeta=acc_init[1].clone())
    res = ops.bn_backward(x, dout, gamma, beta, stats, training, leak, want_colsum=colsum, **kw)
    rec = last_launch("bn_bwd", (n, C, training, x.dtype, colsum))
    what = f"{what} backward{' + colsum' if colsum else ''}{' accumulate' if acc_init is not None else ''} [{rec}]"
    crec = last_launch("col_sum", (n, C, x.dtype)) if rec["colsum"] == 2 else dict(rec, grid=rec["grid2"])
    dx, dg, db = res[:3]
    m, s = stats[0], stats[1]
    r = ref_bn_backward(x, dout, m, s, gamma, beta, leak, training)
    err = fold_error(x, m, s, gamma, beta)
    amb = r["y"].abs() <= err
    if arm == "exact" and leak != 1.0:
        assert not bool(amb.any()), f"{what}: precondition: an element's y is within the fold error of 0"
    flip = torch.where(amb, (1 - leak) * dout.double().abs(), torch.zeros_like(r["dd"]))   # what a flipped mask moves
    gam = (chain_length(rec, n, C) + 4) * U
    x64, m64, s64 = x.double(), m.double(), s.double()
    xh_err = 2.0 ** -22 * (x64.abs() + m64.abs()) * s64
    e_db = gam * r["dd"].abs().sum(0) + flip.sum(0)
    e_dg = gam * (r["dd"] * r["xh"]).abs().sum(0) + (r["dd"].abs() * xh_err).sum(0) + (flip * r["xh"].abs()).sum(0)
    want_db, want_dg = r["dbeta"], r["dgamma"]
    if acc_init is not None:
        want_db, want_dg = want_db + acc_init[1].double(), want_dg + acc_init[0].double()
    if arm == "exact":
        assert 16 * 8 * rows_per_block(rec, n, C) < 2 ** 24 and 16 * n < 2 ** 24, \
            f"{what}: precondition: a partial sum of the masked dout can reach 2^24"
        assert_exact(db, want_db, what + " dbeta")
    else:
        assert_within(db, want_db, e_db + ulp32(want_db), what + " dbeta")
    assert_within(dg, want_dg, e_dg + ulp32(want_dg), what + " dgamma")
    sc = s64 * gamma.double()
    s1, s2 = r["dbeta"] / n, r["dgamma"] / n
    if training:
        e2 = sc * s2 * s64
        A = (sc * r["dd"]).abs() + (x64 * e2).abs() + (m64 * e2).abs() + (sc * s1).abs()
        stat_term = sc.abs() * (e_db + r["xh"].abs() * e_dg) / n
    else:
        A = (sc * r["dd"]).abs()
        stat_term = torch.zeros_like(A)
    bar = 2.0 ** -21 * A + stat_term + sc.abs() * flip
    bar = 1.01 * bar + out_unit(x.dtype) * r["dx"].abs()
    assert_within(dx, r["dx"], bar, what + " dx")
    if colsum:
        cs = res[3]
        stored = dx.double()
        cg = (chain_length(crec, n, C) + 4) * U
        assert_within(cs, stored.sum(0), cg * stored.abs().sum(0) + ulp32(stored.sum(0)), what + " column sums of dx")
    if arm == "exact":
        res2 = ops.bn_backward(x, dout, gamma, beta, stats, training, leak, want_colsum=colsum,
                               **({} if acc_init is None else dict(dgamma=acc_init[0].clone(), dbeta=acc_init[1].clone())))
        for i, (a, b) in enumerate(zip(res, res2)):
            assert torch.equal(a, b), f"{what}: a repeated call gave different bits (output {i})"
    return rec


def check_bn(x, dout, gamma, beta, training, leak, arm, what, rm=None, rv=None):
    """Forward, then the backward with and without the fused column sums."""
    C = x.shape[1]
    g = torch.Generator(device="cuda").manual_seed(C)
    if rm is None:
        rm = torch.randn(C, device="cuda", generator=g) * 0.1
        rv = torch.rand(C, device="cuda", generator=g) + 0.5
    stats, _ = check_bn_forward(x, gamma, beta, rm, rv, training, leak, arm, what)
    for colsum in (True, False):
        check_bn_backward(x, dout, gamma, beta, stats, training, leak, arm, what, colsum)


def bn_inputs(n, C, dtype, case, seed):
    """case: "exact-<leak>" or a DISTS key -> (x, dout, gamma, beta, leak, arm)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    if case.startswith("exact"):
        leak = float(case.split("-")[1])
        x, d, gamma, beta = exact_data(n, C, dtype, g, leak)
        return x, d, gamma, beta, leak, "exact"
    x, d, gamma, beta = rounding_data(n, C, dtype, g, case)
    return x, d, gamma, beta, LEAK_R, "rounding"


def check_col_sum(x, what, accumulate=None):
    """scn_col_sum (or scn_col_sum_acc with `accumulate` as the initial value) against float64."""
    from sparseeventid_b200 import _lib as L
    from sparseeventid_b200.scn import ops
    n, C = x.shape
    if accumulate is None:
        out = ops.col_sum(x)
        base = torch.zeros(C, dtype=torch.float64, device="cuda")
    else:
        out = accumulate.clone()
        ws = torch.empty(2 * C, dtype=torch.float64, device="cuda")
        L.check(L.lib().scn_col_sum_acc(x.data_ptr(), L.dtype_code(x), n, C, ws.data_ptr(), out.data_ptr(), 1,
                                        L.stream()), "scn_col_sum_acc")
        base = accumulate.double()
    rec = last_launch("col_sum", (n, C, x.dtype))
    x64 = x.double()
    want = x64.sum(0) + base
    gam = (chain_length(rec, n, C) + 4) * U
    assert_within(out, want, gam * x64.abs().sum(0) + ulp32(want), f"{what} column sums [{rec}]")
    return rec


# ==================================================================================== BatchNorm at the benchmark's shapes

CHANNELS = [32, 64, 96, 128, 160, 192]
BN_CASES = ["exact-0.5", "exact-1", "mu0", "mu10", "mu100", "pivot30"]
DTYPES = [torch.bfloat16, torch.float32]


@pytest.fixture(scope="module")
def bench_rows():
    """Active sites per level of the benchmark's first batch (InputLayer, then the stride-2 rules)."""
    import sparseconvnet as scn
    from sparseeventid_b200 import synthetic
    coords, feats, bs = bench_batch()
    x = scn.InputLayer(3, list(synthetic.GRID_3D))((torch.as_tensor(coords).cuda(), torch.as_tensor(feats).cuda(), bs))
    md = x.metadata
    sp = tuple(synthetic.GRID_3D)
    rows = []
    for level in range(6):
        rows.append(md.levels[sp].n)
        if level < 5:
            sp = md.strided_rule(sp, (2, 2, 2), (2, 2, 2)).out_spatial
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("case", BN_CASES)
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp32"])
@pytest.mark.parametrize("level", range(6))
def test_bn_bench_levels(bench_rows, level, dtype, case):
    n, C = bench_rows[level], CHANNELS[level]
    x, d, gamma, beta, leak, arm = bn_inputs(n, C, dtype, case, 1000 + 10 * level)
    check_bn(x, d, gamma, beta, True, leak, arm, f"level {level} ({n} x {C}) {case} {dtype}")
    _done("bench")


# ==================================================================================== channel sweep, row edges

SWEEP_C = [1, 5, 8, 12, 16, 24, 40, 96, 256, 258, 264, 1028, 2048, 2056]


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["exact-0.5", "mu10"])
@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp32"])
@pytest.mark.parametrize("C", SWEEP_C)
def test_bn_channel_sweep(C, dtype, training, case):
    n = 3000
    x, d, gamma, beta, leak, arm = bn_inputs(n, C, dtype, case, 2000 + C)
    check_bn(x, d, gamma, beta, training, leak, arm, f"{n} x {C} {case} {dtype} {'train' if training else 'eval'}")
    check_col_sum(x, f"{n} x {C} {dtype}")
    _done("sweep")


def _edge_rows(C):
    ry = 256 // (C // 8)
    cap = 4 * ry * 148 * 4
    return [1, 2, ry - 1, ry, ry + 1, cap - 1, cap + 1]


EDGES = [(C, n) for C in (32, 192) for n in _edge_rows(C)]


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ["exact", "rounding"])
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp32"])
@pytest.mark.parametrize("C,n", EDGES)
def test_bn_row_edges(C, n, dtype, arm):
    """n = 1 (divisor max(n - 1, 1)), 2, RY - 1, RY, RY + 1 and the edges of the grid cap (4 RY rows a thread in 592
    blocks); the exact arm uses leak 1 below 3 rows, where no mean can be kept off the integers."""
    case = ("exact-0.5" if n >= 3 else "exact-1") if arm == "exact" else "mu10"
    x, d, gamma, beta, leak, arm = bn_inputs(n, C, dtype, case, 3000 + n + C)
    check_bn(x, d, gamma, beta, True, leak, arm, f"{n} x {C} {case} {dtype}")
    _done("edges")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp32"])
@pytest.mark.parametrize("C", [12, 32, 2056])
def test_bn_accumulate(C, dtype):
    """accumulate = 1: dgamma / dbeta and the column sums are added to what the buffers hold (integers: dbeta exact)."""
    n = 5000
    x, d, gamma, beta, leak, arm = bn_inputs(n, C, dtype, "exact-0.5", 4000 + C)
    rm, rv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    stats, _ = check_bn_forward(x, gamma, beta, rm, rv, True, leak, arm, f"{n} x {C}")
    g = torch.Generator(device="cuda").manual_seed(C)
    init = (torch.randint(-50, 50, (C,), device="cuda", generator=g).float(),
            torch.randint(-50, 50, (C,), device="cuda", generator=g).float())
    check_bn_backward(x, d, gamma, beta, stats, True, leak, arm, f"{n} x {C}", False, acc_init=init)
    rec = check_col_sum(x, f"{n} x {C} accumulate", accumulate=init[1])
    assert rec["path"] == (1 if C % 8 == 0 and C <= 2048 else 4)
    _done("accumulate")


@pytest.mark.gpu
@pytest.mark.parametrize("shift", ["1 element", "8 bytes"])
@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp32"])
@pytest.mark.parametrize("C", [12, 32, 264])
def test_bn_unaligned_views(C, dtype, training, shift):
    """Contiguous views t.view(-1)[k:] of a 16-byte-aligned buffer: the launchers must pick the vector width the
    pointer allows (VEC 4 needs 4-element alignment, VEC 8 and the two-launch kernels 16 bytes).  An 8-byte shift
    leaves bf16 rows aligned for VEC 4 only."""
    n = 4000
    k = 1 if shift == "1 element" else 8 // (2 if dtype == torch.bfloat16 else 4)
    x, d, gamma, beta, leak, arm = bn_inputs(n, C, dtype, "exact-0.5", 5000 + C + k)

    def shifted(t):
        buf = torch.empty(t.numel() + 16, dtype=t.dtype, device="cuda")
        v = buf.view(-1)[k:k + t.numel()].view(t.shape)
        v.copy_(t)
        assert v.is_contiguous() and v.data_ptr() % 16 != 0
        return v

    xs, ds = shifted(x), shifted(d)
    rm, rv = torch.full((C,), 0.375, device="cuda"), torch.ones(C, device="cuda")   # eval: no y = 0 on integer x
    what = f"{n} x {C} {dtype} view offset {k}"
    stats, rec = check_bn_forward(xs, gamma, beta, rm, rv, training, leak, arm, what)
    vec_ok = C % 4 == 0 and (xs.data_ptr() % (4 * xs.element_size())) == 0
    assert rec["path"] == 4, f"{what}: {rec}"
    assert rec["avec"] == (4 if vec_ok else 1), f"{what}: {rec}"
    for colsum in (True, False):
        brec = check_bn_backward(xs, ds, gamma, beta, stats, training, leak, arm, what, colsum)
        assert brec["path"] == 4 and brec["avec"] == (4 if vec_ok else 1), f"{what}: {brec}"
    crec = check_col_sum(xs, what)
    assert crec["path"] == 4 and crec["vec"] == (4 if vec_ok else 1), f"{what}: {crec}"
    _done("unaligned")


# ==================================================================================== shared scratch, interleaved


def _sequence(second_stream):
    """Two-launch BatchNorm with the channel count rising and falling, four-launch calls (C = 12, unaligned) between
    them, scn_col_sum and fused-colsum backwards on one stream; optionally one call on a second stream."""
    steps = [(3000, 160, "bn"), (5000, 32, "bn"), (777, 12, "bn4"), (900, 192, "bn"), (4000, 64, "col"),
             (7000, 32, "bn"), (2500, 128, "bn4"), (6000, 96, "bn"), (3333, 192, "col"), (64, 32, "bn")]
    side = torch.cuda.Stream() if second_stream else None
    for i, (n, C, kind) in enumerate(steps):
        x, d, gamma, beta, leak, arm = bn_inputs(n, C, torch.bfloat16 if i % 2 else torch.float32,
                                                 "exact-0.5" if i % 3 else "mu10", 6000 + i)
        if kind == "bn4":
            buf = torch.empty(x.numel() + 8, dtype=x.dtype, device="cuda")
            x = buf[1:1 + x.numel()].view(n, C).copy_(x)
        what = f"step {i} ({n} x {C} {kind}{', second stream' if side is not None and i == 5 else ''})"

        def run():
            if kind == "col":
                check_col_sum(x, what)
            else:
                check_bn(x, d, gamma, beta, True, leak, arm, what)
        if side is not None and i == 5:
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                run()
            torch.cuda.current_stream().wait_stream(side)
        else:
            run()


@pytest.mark.gpu
@pytest.mark.parametrize("second_stream", [False, True], ids=["one stream", "two streams"])
def test_interleaved_calls_share_the_scratch(second_stream):
    _sequence(second_stream)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [258, 2056])
def test_batchnorm_layer_trains_at_wide_odd_channel_counts(C):
    """BatchNormalization(C) forward and backward in training through the module, at channel counts whose column
    reductions need more than one channel slice."""
    import sparseconvnet as scn
    from helpers import blob_sites
    scn.set_precision("fp32")
    coords = torch.as_tensor(blob_sites(300, (16, 16, 16), 2, seed=C)).cuda()
    feats = torch.randn(coords.shape[0], C, device="cuda") * 2 + 1
    x = scn.InputLayer(3, [16, 16, 16])((coords, feats, 2))
    bn = scn.BatchNormalization(C).cuda().train()
    y = bn(x)
    y.features.square().sum().backward()
    f = x.features.double()
    want = (f - f.mean(0)) / torch.sqrt(f.var(0, unbiased=False) + EPS)
    assert float((y.features.double() - want).abs().max()) <= 1e-4
    assert bn.weight.grad is not None and bool(torch.isfinite(bn.weight.grad).all())


# ==================================================================================== data movement: bit-exact


def _vec_cases():
    # (count, pointer offset in elements) -> expected VEC: 8-wide, 4-wide by count, 1-wide by count and by pointer
    return [(4096 * 8, 0, 8), (4096 * 8 + 4, 0, 4), (4096 * 8 + 3, 0, 1), (4096 * 8, 1, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["leaky_fwd", "leaky_bwd", "add", "add_leaky"])
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp32"])
@pytest.mark.parametrize("count,offset,vec", _vec_cases())
def test_leaky_and_add(count, offset, vec, dtype, which):
    from sparseeventid_b200.scn import ops
    g = torch.Generator(device="cuda").manual_seed(count + offset)

    def view(t):
        buf = torch.empty(count + 8, dtype=dtype, device="cuda")
        return buf[offset:offset + count].copy_(t)
    a = view(torch.randn(count, device="cuda", generator=g).to(dtype))
    b = view(torch.randn(count, device="cuda", generator=g).to(dtype))
    a[:8] = torch.tensor([0.0, -0.0, 1.0, -1.0, 2 ** -130, -(2 ** -130), 3.0e38, -3.0e38], device="cuda").to(dtype)
    leak = LEAK_R
    af, bf = a.float(), b.float()

    def go():
        if which == "leaky_fwd":
            return ops.leaky_forward(a, leak)
        if which == "leaky_bwd":
            return ops.leaky_backward(a, b, leak)
        return ops.add_forward(a, b, leak if which == "add_leaky" else 1.0)
    out, again = go(), go()
    rec = last_launch("elem", (which, count, offset, dtype))
    assert rec["vec"] == vec, f"{which} {count} +{offset}: {rec}"
    if which == "leaky_fwd":
        want = torch.where(af > 0, af, af * leak)
    elif which == "leaky_bwd":
        want = torch.where(af > 0, bf, bf * leak)
    else:
        s = af + bf
        want = torch.where(s > 0, s, s * leak) if which == "add_leaky" else s
    want = want.to(dtype)
    assert torch.equal(out.view(torch.int16 if dtype == torch.bfloat16 else torch.int32),
                       want.view(torch.int16 if dtype == torch.bfloat16 else torch.int32)), \
        f"{which} {count} +{offset} {dtype}: {int((out != want).sum())} elements differ"
    assert torch.equal(out, again)
    _done("elem")


def _convert_specials():
    f = np.float32
    vals = [0.0, -0.0, 1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, -(1.0 + 2.0 ** -8), 1.0 + 2.0 ** -8 + 2.0 ** -20,
            2.0 ** -149, -(2.0 ** -149), 2.0 ** -133, 2.0 ** -126 * 0.75, 1.17e-38, float(np.finfo(f).max),
            -float(np.finfo(f).max), 3.3895314e38, 3.3961e38, float("inf"), float("-inf"), 65504.0, 1e-45]
    return torch.tensor(vals, dtype=torch.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("with_rows", [False, True], ids=["convert", "gather"])
def test_fp32_to_bf16_conversion(with_rows):
    """k_convert / k_rows_gather fp32 -> bf16 equal torch's .bfloat16() bit for bit: ties to even, +-0, subnormals,
    the largest finite value and overflow to inf, random bit patterns; NaN stays NaN."""
    from sparseeventid_b200.scn import ops
    g = torch.Generator(device="cuda").manual_seed(9)
    bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (1 << 16,), device="cuda", generator=g, dtype=torch.int64).to(torch.int32)
    ties = (torch.randint(0, 2 ** 16, (4096,), device="cuda", generator=g, dtype=torch.int64) << 16) | 0x8000
    ties = torch.where(ties >= 2 ** 31, ties - 2 ** 32, ties).to(torch.int32)       # halfway between two bf16 values
    src = torch.cat([_convert_specials().cuda(), bits.view(torch.float32), ties.view(torch.float32)])
    nan = torch.isnan(src)
    if with_rows:
        x = src.view(-1, 1).contiguous()
        rows = torch.randperm(x.shape[0], device="cuda", generator=g).to(torch.int32)
        out = ops.rows_gather(x, rows, torch.bfloat16)[:, 0]
        src, nan = src[rows.long()], nan[rows.long()]
    else:
        out = ops.convert(src, torch.bfloat16)
    want = src.bfloat16()
    assert bool(torch.isnan(out[nan]).all()), "NaN did not stay NaN"
    keep = ~nan
    ob, wb = out[keep].view(torch.int16), want[keep].view(torch.int16)
    bad = ob != wb
    assert not bool(bad.any()), f"{int(bad.sum())} conversions differ, e.g. {src[keep][bad][:4].tolist()}"
    _done("convert")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [3, 4])
@pytest.mark.parametrize("C", [1, 3])
def test_input_layer_and_scatter_add(C, mode):
    """InputLayer modes 3 (sum) and 4 (mean) and rows_scatter_add at bench scale with duplicates, integer features:
    sums are exact, the mean is the correctly rounded fp32 quotient."""
    from sparseeventid_b200.scn import ops
    g = torch.Generator(device="cuda").manual_seed(C * 10 + mode)
    n_in, n_active = 600_000, 400_000
    rows = torch.randint(0, n_active, (n_in,), device="cuda", generator=g, dtype=torch.int32)
    rows[:n_active] = torch.randperm(n_active, device="cuda", generator=g).to(torch.int32)   # every row hit
    feats = torch.randint(-8, 9, (n_in, C), device="cuda", generator=g).float()
    s = torch.zeros(n_active, C, dtype=torch.float64, device="cuda").index_add_(0, rows.long(), feats.double())
    cnt = torch.zeros(n_active, dtype=torch.float64, device="cuda").index_add_(
        0, rows.long(), torch.ones(n_in, dtype=torch.float64, device="cuda"))
    out, again = (ops.input_layer_forward(feats, rows, n_active, mode) for _ in range(2))
    want = s.float() if mode == 3 else s.float() / cnt.float()[:, None]
    assert torch.equal(out, want), f"InputLayer mode {mode}: {int((out != want).sum())} elements differ"
    assert torch.equal(out, again)
    for dtype in DTYPES:
        sc = ops.rows_scatter_add(feats.to(dtype), rows, n_active)
        assert torch.equal(sc, s.float()), f"rows_scatter_add {dtype}"
    _done("scatter")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp32"])
@pytest.mark.parametrize("col0,ncol,vec", [(0, 32, 4), (4, 24, 4), (1, 28, 1), (0, 5, 1), (3, 5, 1)])
@pytest.mark.parametrize("K,scale", [(8, 1 / 8), (4, 1 / 4)])
def test_pool_rows(K, scale, col0, ncol, vec, dtype):
    """AveragePooling rows: integer features, existing table entries only, exact sums times a power of two."""
    from sparseeventid_b200.scn import ops
    g = torch.Generator(device="cuda").manual_seed(K + col0 * 7 + ncol)
    n_src, n_rows, width = 20000, 7000, 36
    n_pad = ops.pad128(n_rows)
    nbr = torch.full((K, n_pad), -1, dtype=torch.int32, device="cuda")
    live = torch.rand(K, n_rows, device="cuda", generator=g) < 0.6
    idx = torch.randint(0, n_src, (K, n_rows), device="cuda", generator=g, dtype=torch.int32)
    nbr[:, :n_rows] = torch.where(live, idx, torch.full_like(idx, -1))
    nbr[K - 1, n_rows - 1] = n_src - 1
    x = torch.randint(-8, 9, (n_src, width), device="cuda", generator=g).to(dtype)
    out, again = (ops.pool_rows(x, nbr, n_rows, scale, col0=col0, ncol=ncol) for _ in range(2))
    rec = last_launch("pool", (K, col0, ncol, dtype))
    assert rec["vec"] == vec, f"pool col0 {col0} ncol {ncol}: {rec}"
    ref = torch.zeros(n_rows, ncol, dtype=torch.float64, device="cuda")
    x64 = x.double()[:, col0:col0 + ncol]
    for k in range(K):
        j = nbr[k, :n_rows].long()
        m = j >= 0
        ref[m] += x64[j[m]]
    assert_exact(out, ref * scale, f"pool K {K} col0 {col0} ncol {ncol} {dtype}")
    assert torch.equal(out, again)
    _done("pool")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp32"])
def test_sparse_to_dense(dtype):
    """Sites outside the dense volume (a coordinate >= the spatial size, a batch index >= the batch count) are dropped
    forward and get a zero gradient."""
    from oracle import scn_oracle as O
    from helpers import random_sites
    from sparseeventid_b200.scn import ops
    spatial, batch, C = (6, 5, 7), 3, 5
    inside = random_sites(300, spatial, batch, seed=4)
    outside = np.array([[6, 0, 0, 0], [0, 5, 0, 1], [0, 0, 7, 2], [1, 1, 1, 3], [5, 4, 6, 7], [6, 5, 7, 3]], dtype=np.int64)
    coords = np.concatenate([inside, outside])
    coords = coords[np.random.default_rng(1).permutation(coords.shape[0])]
    keys = torch.as_tensor(O.pack_keys(coords)).cuda()
    g = torch.Generator(device="cuda").manual_seed(5)
    n = coords.shape[0]
    x = torch.randn(n, C, device="cuda", generator=g).to(dtype)
    dense, again = (ops.sparse_to_dense_forward(x, keys, batch, spatial) for _ in range(2))
    want = torch.zeros((batch, C) + spatial, dtype=torch.float32, device="cuda")
    c = torch.as_tensor(coords).cuda()
    ok = (c[:, 0] < spatial[0]) & (c[:, 1] < spatial[1]) & (c[:, 2] < spatial[2]) & (c[:, 3] < batch)
    assert int((~ok).sum()) == outside.shape[0]
    ci = c[ok]
    want[ci[:, 3], :, ci[:, 0], ci[:, 1], ci[:, 2]] = x[ok].float()
    assert torch.equal(dense, want) and torch.equal(dense, again)
    dd = torch.randn((batch, C) + spatial, device="cuda", generator=g)
    dx = ops.sparse_to_dense_backward(dd, keys, n, C, batch, spatial, dtype)
    wx = torch.zeros(n, C, dtype=torch.float32, device="cuda")
    wx[ok] = dd[ci[:, 3], :, ci[:, 0], ci[:, 1], ci[:, 2]]
    assert torch.equal(dx, wx.to(dtype))
    assert torch.equal(dx, ops.sparse_to_dense_backward(dd, keys, n, C, batch, spatial, dtype))
    _done("s2d")


# ==================================================================================== coverage of the launchers


@pytest.mark.gpu
def test_launches_reached_every_launcher_branch():
    want = {"bench": 6 * 2 * len(BN_CASES), "sweep": len(SWEEP_C) * 2 * 2 * 2, "edges": 2 * 2 * len(EDGES),
            "accumulate": 6, "unaligned": 24, "elem": 32, "pool": 20}
    if any(_DONE.get(k, 0) < v for k, v in want.items()):
        pytest.skip(f"needs the whole file to have passed first: {_DONE} of {want}")
    fwd = [r for _, r in _LAUNCHES["bn_fwd"]]
    bwd = [r for _, r in _LAUNCHES["bn_bwd"]]
    cs = [r for _, r in _LAUNCHES["col_sum"]]
    for name, recs, cap in (("forward", fwd, 148 * 4), ("backward", bwd, 148 * 3)):
        two = [r for r in recs if r["path"] == 2]
        assert any(r["grid"] == cap for r in two), f"two-launch {name} at the grid cap"
        assert any(r["grid"] < cap for r in two), f"two-launch {name} below the grid cap"
        four = [r for r in recs if r["path"] == 4]
        assert {8, 4, 1} <= {r["vec"] for r in four}, f"four-launch {name} reductions VEC 8 / 4 / 1"
        assert {(1, 8), (2, 4), (2, 1)} <= {(r["apply"], r["avec"]) for r in four}, f"four-launch {name} apply forms"
        assert any(r["slices"] > 1 for r in four), f"four-launch {name} with several channel slices"
    assert any(r["path"] == 4 and r["vec"] == 0 for r in fwd), "eval-mode forward"
    assert {0, 1, 2} <= {r["colsum"] for r in bwd}, "backward without / with fused / with separate column sums"
    assert any(r["path"] == 2 and r["grid2"] == 148 * 3 and r["colsum"] == 1 for r in bwd), "fused colsum at the cap"
    assert any(r["path"] == 1 for r in cs) and {4, 1} <= {r["vec"] for r in cs if r["path"] == 4}, "column-sum paths"
    assert any(r["path"] == 4 and r["slices"] > 1 for r in cs), "column sums over several channel slices"
    two_c = {info[1] for info, r in _LAUNCHES["bn_fwd"] if r["path"] == 2}
    assert {8, 16, 256, 264, 2048} <= two_c, f"block_col_sums extremes: CV = 1, 2, 32, 33, 256 ({sorted(two_c)})"
    elem = {(r["path"], r["vec"]) for _, r in _LAUNCHES["elem"]}
    assert {(w, v) for w in (0, 1, 2) for v in (8, 4, 1)} <= elem, f"elementwise paths {sorted(elem)}"
    assert {4, 1} <= {r["vec"] for _, r in _LAUNCHES["pool"]}, "pool V = 4 and V = 1"
