"""The integer layer that builds every neighbour table -- key packing, the coordinate hash, InputLayer rules, the
submanifold / strided / pair-list rulebooks and the device larcv transform -- against the oracle, bit-exact, where
naturally spread inputs never reach:

  * a host model of the hash table (the murmur3 finaliser of csrc/common.cuh and a bucket-level linear-probing model,
    whose final bucket occupancy does not depend on insertion order) is pinned on the CPU against a literal slot-by-slot
    insertion loop, and on the GPU against the table the device builds (read back slot by slot);
  * keys chosen by hashing candidates on the host force what the benchmark batches never produce: chains of 3 and more
    full buckets, a chain that wraps from the last bucket through bucket 0, absent keys whose home buckets are full,
    all at the largest load the ABI allows (n = capacity / 2), and 2 M-row inputs whose duplicates race each other;
  * the 16-bit key fields at their edges (coordinates 0 and 65535, batch indices on both sides of the top bit);
  * the dune2d benchmark batch's six levels, the device larcv transform on both full benchmark arrays and its edges;
  * the entry points the modules do not call directly: the sort-based strided rulebook, scn_hash_build / lookup, the
    remap branch of Metadata.strided_rule and the pair list of a table.

Every device build runs twice, from different insertion orders, and must give the same tables; deeper levels are
compared in the coordinate-matched numbering of test_bench_scale_parity.py.
"""
import numpy as np
import pytest
import torch

from helpers import bench_batch, blob_sites, random_sites
from oracle import scn_oracle as O
from test_bench_scale_parity import check_level_rulebooks, rules_to_table, to_oracle

M1, M2, MASK64 = 0xFF51AFD7ED558CCD, 0xC4CEB9FE1A85EC53, (1 << 64) - 1
EMPTY = np.uint64(MASK64)
FULL = (65536, 65536, 65536)              # a grid on which every 16-bit coordinate is inside


# --------------------------------------------------------------------------------------- host model of the hash


def key_hash_py(k: int) -> int:
    """key_hash of csrc/common.cuh on Python integers."""
    k &= MASK64
    k ^= k >> 33
    k = (k * M1) & MASK64
    k ^= k >> 33
    k = (k * M2) & MASK64
    k ^= k >> 33
    return k & 0xFFFFFFFF


def key_hash(keys) -> np.ndarray:
    """The same on a uint64 array (numpy's uint64 products wrap modulo 2^64 like the device's)."""
    k = np.array(keys, dtype=np.uint64)
    k ^= k >> np.uint64(33)
    k *= np.uint64(M1)
    k ^= k >> np.uint64(33)
    k *= np.uint64(M2)
    k ^= k >> np.uint64(33)
    return (k & np.uint64(0xFFFFFFFF)).astype(np.int64)


def capacity(n: int) -> int:
    """scn_hash_capacity: the smallest power of two >= max(1024, 2n)."""
    c = 1024
    while c < 2 * n:
        c <<= 1
    return c


def home(keys, cap) -> np.ndarray:
    return key_hash(keys) & (cap // 8 - 1)


def bucket_model(keys, cap):
    """(final occupancy of every 8-slot bucket, number of keys that ran past the last bucket into bucket 0) after
    inserting the distinct `keys` with linear probing over buckets.  The occupancy does not depend on the order."""
    nb = cap // 8
    cnt = np.bincount(home(keys, cap), minlength=nb).tolist()
    occ = [0] * nb
    carry = wrapped = 0
    for rnd in range(2):                          # the second round only places what wrapped
        for b in range(nb):
            t = occ[b] + (cnt[b] if rnd == 0 else 0) + carry
            occ[b] = min(8, t)
            carry = t - occ[b]
            if rnd == 1 and carry == 0:
                break
        if rnd == 0:
            wrapped = carry
    return np.asarray(occ), wrapped


def insert_literal(keys, cap):
    """The insert of csrc/hash.cu one key at a time, slot by slot: probe the home bucket, take the first empty slot, else
    the next bucket (bucket + 1) & mask.  Returns the slots (None = empty)."""
    nb = cap // 8
    slots = [None] * cap
    for k in keys:
        b = key_hash_py(int(k)) & (nb - 1)
        while True:
            row = slots[8 * b:8 * b + 8]
            if k in row:
                break
            if None in row:
                slots[8 * b + row.index(None)] = k
                break
            b = (b + 1) & (nb - 1)
    return slots


def check_placement(table_keys, keys, cap):
    """A device table (int64 [cap] read back) holds exactly the distinct `keys`, once each, with the model's occupancy;
    a key sits in its home bucket when that bucket is not full, else inside the chain of full buckets that follows it.
    Returns the probe distance (buckets past home) of every stored key and its home bucket."""
    nb = cap // 8
    tk = np.asarray(table_keys).view(np.uint64).reshape(nb, 8)
    keys = np.unique(np.asarray(keys).view(np.uint64))
    occ, _ = bucket_model(keys, cap)
    assert np.array_equal((tk != EMPTY).sum(1), occ), "bucket occupancy differs from the model"
    b_of, s_of = np.nonzero(tk != EMPTY)
    stored = tk[b_of, s_of]
    assert np.array_equal(np.sort(stored), keys), "the table does not hold exactly the distinct keys"
    h = home(stored, cap)
    d = (b_of - h) % nb
    notfull = np.concatenate([[0], np.cumsum(np.concatenate([occ, occ]) < 8)])
    assert np.all(notfull[h + d] - notfull[h] == 0), "a key sits past a bucket that is not full"
    return d, h


def test_host_hash_model_matches_literal_insertion():
    """Pins the numpy key_hash against Python integers and the bucket model against slot-by-slot insertion in three
    orders, on a table with long chains and a wrap (the same construction as the forced GPU tables)."""
    rng = np.random.default_rng(0)
    cap = 1024
    coords = forced_sites(cap, {cap // 8 - 1: 30, 5: 26, 6: 9}, rng, batch=(0, 65535))
    keys = O.pack_keys(np.concatenate([coords, random_sites(300, (64, 64, 64), 4, seed=1)]))
    assert [key_hash_py(int(k)) for k in keys[:2000]] == key_hash(keys[:2000]).tolist()
    assert key_hash_py(0) == 0 and key_hash_py(MASK64) == int(key_hash(np.array([EMPTY]))[0])
    occ, wrapped = bucket_model(keys, cap)
    assert wrapped > 0 and occ[0] == 8 and occ[5] == occ[6] == occ[7] == 8
    for order in (np.arange(keys.shape[0]), rng.permutation(keys.shape[0]), np.arange(keys.shape[0])[::-1]):
        slots = insert_literal([int(k) for k in keys[order]], cap)
        tk = np.array([MASK64 if s is None else s for s in slots], dtype=np.uint64)
        d, h = check_placement(tk.view(np.int64), keys, cap)
        assert d.max() >= 3 and np.any(h + d >= cap // 8)
    # the check rejects a table in which one key moved from a full bucket to a bucket outside its chain
    tk = tk.copy().reshape(-1, 8)
    src, dst = int(np.nonzero(occ == 8)[0][0]), int(np.nonzero(occ == 0)[0][0])
    tk[dst, 0], tk[src, 7] = tk[src, 7], EMPTY
    with pytest.raises(AssertionError):
        check_placement(tk.reshape(-1).view(np.int64), keys, cap)


# --------------------------------------------------------------------------------------- forcing keys


def forced_sites(cap, want, rng, batch=(1, 4), coords_hi=65536, exclude=()):
    """Distinct sites (x0, x1, x2, b) whose keys have the given home buckets in a table of `cap` slots: `want` maps a
    bucket to a count.  Candidates are random sites with b in [batch[0], batch[1]); a hit costs about cap / 8 of them."""
    nb = cap // 8
    need = dict(want)
    got = {b: [] for b in need}
    seen = set(int(k) for k in np.asarray(exclude, dtype=np.uint64).tolist())
    while any(len(got[b]) < need[b] for b in need):
        m = int(min(1 << 22, max(1 << 14, 4 * nb * sum(need[b] - len(got[b]) for b in need))))
        c = np.concatenate([rng.integers(0, coords_hi, size=(m, 3)), rng.integers(batch[0], batch[1], size=(m, 1))], 1)
        k = O.pack_keys(c)
        hb = home(k, cap)
        for b in need:
            for i in np.nonzero(hb == b)[0].tolist():
                if len(got[b]) >= need[b]:
                    break
                ki = int(k[i])
                if ki not in seen:
                    seen.add(ki)
                    got[b].append(c[i])
    out = [np.asarray(got[b]).reshape(-1, 4) for b in need]
    return np.concatenate(out).astype(np.int64) if out else np.zeros((0, 4), np.int64)


SUBM_FILTERS = [(3, 3, 3), (5, 5, 5), (1, 5, 5), (3, 1, 5), (1, 1, 1)]


def forced_layout(n_total, seed=0):
    """n_total distinct sites for a table of capacity(n_total) slots, of which:
      * a clustered sample (batch 0) whose submanifold neighbourhoods are dense;
      * 24 filler sites homed in the home bucket of cluster site 0: a chain of >= 3 full buckets that cluster sites sit in;
      * 24 filler sites homed in the LAST bucket: a chain that wraps through bucket 0 and beyond;
      * 8 fillers in the home bucket of each of 6 more cluster sites (present keys behind full buckets);
      * 8 fillers in the home bucket of each of 8 ABSENT neighbours of the cluster (offsets (0, 0, +-1), inside every
        filter tested): probes for keys that are not there cross full buckets;
      * random fillers up to n_total.
    Fillers live in batches 1..3, so they never neighbour the cluster.  Returns (coords [n_total, 4] shuffled,
    cap, dict of the forced buckets, absent query keys)."""
    rng = np.random.default_rng(seed)
    cap = capacity(n_total)
    nb = cap // 8
    cl = blob_sites(60, (12, 12, 12), 1, seed=seed + 3)
    ck = O.pack_keys(cl)
    ch = home(ck, cap)
    q = cl.copy()
    absent = []
    for dz in (-1, 1):
        q = cl.copy()
        q[:, 2] += dz
        ok = (q[:, 2] >= 0)
        absent.append(O.pack_keys(q[ok]))
    absent = np.setdiff1d(np.concatenate(absent), ck)
    ah = home(absent, cap)
    absent_buckets = list(dict.fromkeys(ah.tolist()))[:8]
    want = {}
    chain_b, wrap_b = int(ch[0]), nb - 1
    for b in [int(x) for x in ch[1:7]] + absent_buckets:
        want[b] = want.get(b, 0) + 8
    want[chain_b] = want.get(chain_b, 0) + 24
    want[wrap_b] = want.get(wrap_b, 0) + 24
    fill = forced_sites(cap, want, rng, exclude=ck)
    n_rand = n_total - cl.shape[0] - fill.shape[0]
    assert n_rand >= 0
    taken = set(O.pack_keys(np.concatenate([cl, fill])).tolist())
    rnd = []
    while len(rnd) < n_rand:
        c = np.concatenate([rng.integers(0, 65536, size=3), rng.integers(1, 4, size=1)])
        k = int(O.pack_keys(c[None])[0])
        if k not in taken:
            taken.add(k)
            rnd.append(c)
    coords = np.concatenate([cl, fill, np.asarray(rnd, dtype=np.int64).reshape(-1, 4)])
    coords = coords[rng.permutation(coords.shape[0])]
    assert coords.shape[0] == n_total and np.unique(O.pack_keys(coords)).shape[0] == n_total
    absent = absent[np.isin(ah, absent_buckets)]
    return coords, cap, {"chain": chain_b, "wrap": wrap_b, "absent": absent_buckets}, absent


def assert_forced_preconditions(table_keys, coords, cap, forced, absent):
    """From the model AND the read-back table: a chain spans >= 3 full buckets, a chain wraps from the last bucket into
    bucket 0 and beyond, and the home bucket of every absent query is full."""
    keys = O.pack_keys(coords)
    occ, wrapped = bucket_model(keys, cap)
    nb = cap // 8
    c = forced["chain"]
    assert all(occ[(c + i) % nb] == 8 for i in range(3)), "model: the forced chain spans fewer than 3 full buckets"
    assert wrapped > 8 and occ[0] == 8, "model: the forced chain does not wrap through bucket 0"
    assert np.all(occ[home(absent, cap)] == 8), "model: an absent key's home bucket is not full"
    d, h = check_placement(table_keys, keys, cap)
    assert np.any((h == c) & (d >= 2)), "read-back: no key of the forced chain sits 2 buckets past its home"
    assert np.any((h == nb - 1) & (d >= 2)), "read-back: no key wrapped past bucket 0"
    tk = np.asarray(table_keys).view(np.uint64).reshape(nb, 8)
    assert np.all((tk[home(absent, cap)] != EMPTY).all(1)), "read-back: an absent key's home bucket is not full"


# --------------------------------------------------------------------------------------- GPU helpers


def _ops():
    from sparseeventid_b200.scn import ops
    return ops


def _lib():
    from sparseeventid_b200 import _lib as L
    return L


def metadata(coords, spatial=FULL, dimension=3, dtype=torch.int64):
    from sparseeventid_b200.scn.core import Metadata
    md = Metadata(dimension, "cuda")
    md.build_input(torch.as_tensor(coords).to(dtype).cuda(), spatial)
    return md


def table_of(md, spatial=FULL):
    lvl = md.levels[tuple(spatial)]
    return lvl.table_keys.cpu().numpy(), lvl.cap


def assert_input_rules(md, coords, spatial=FULL):
    rows_ref, active_ref = O.input_layer_rules(coords)
    assert np.array_equal(md.row_of_input.cpu().numpy().astype(np.int64), rows_ref)
    assert np.array_equal(md.coords(spatial).cpu().numpy(), active_ref)
    assert md.levels[tuple(spatial)].n == active_ref.shape[0]
    return rows_ref, active_ref


# --------------------------------------------------------------------------------------- A + B: forced tables


@pytest.mark.gpu
@pytest.mark.parametrize("n_total", [512, 3000])
def test_forced_table_readback_and_lookup(n_total):
    """scn_hash_build on the forced keys: the read-back table is the model's, every present key is found with its
    index, every absent neighbour query (full home bucket) returns -1.  n = 512 is the ABI's largest load on 1024 slots."""
    ops = _ops()
    coords, cap, forced, absent = forced_layout(n_total)
    assert ops.new_table(n_total, "cuda")[2] == cap
    keys = O.pack_keys(coords)
    rng = np.random.default_rng(1)
    for run in range(2):
        order = np.arange(n_total) if run == 0 else rng.permutation(n_total)
        kd = torch.as_tensor(keys[order].view(np.int64)).cuda()
        tk, tv, c = ops.hash_build(kd)
        assert c == cap
        assert_forced_preconditions(tk.cpu().numpy(), coords, cap, forced, absent)
        # the value of a slot is the key's index
        tkn, tvn = tk.cpu().numpy().view(np.uint64), tv.cpu().numpy()
        pos = {int(k): i for i, k in enumerate(keys[order])}
        live = tkn != EMPTY
        assert [pos[int(k)] for k in tkn[live]] == tvn[live].tolist()
        q_perm = rng.permutation(n_total)
        got = ops.hash_lookup(kd[torch.as_tensor(q_perm).cuda()], tk, tv, cap).cpu().numpy()
        assert np.array_equal(got, q_perm)
        got = ops.hash_lookup(torch.as_tensor(absent.view(np.int64)).cuda(), tk, tv, cap).cpu().numpy()
        assert np.all(got == -1)


@pytest.mark.gpu
@pytest.mark.parametrize("n_total", [512, 3000])
def test_forced_input_layer_rules(n_total):
    """InputLayer rules (first-appearance rows, keys_out, n_active) on the forced keys with duplicates, two orders."""
    coords, cap, forced, absent = forced_layout(n_total)
    rng = np.random.default_rng(2)
    for run in range(2):
        c = np.concatenate([coords, coords[rng.integers(0, n_total, n_total // 2)]])
        c = c[rng.permutation(c.shape[0])]
        md = metadata(c)
        assert_input_rules(md, c)
        tk, got_cap = table_of(md)
        assert got_cap == capacity(c.shape[0])
        check_placement(tk, O.pack_keys(coords), got_cap)


@pytest.mark.gpu
@pytest.mark.parametrize("filt", SUBM_FILTERS)
@pytest.mark.parametrize("n_total", [512, 3000])
def test_forced_submanifold_tables(n_total, filt):
    """Submanifold tables on the forced table: present neighbours behind full buckets, absent ones whose home buckets
    are full, and chains through the wrap.  Two builds of one order are identical; a second order matches its oracle."""
    coords, cap, forced, absent = forced_layout(n_total)
    n = n_total
    tables = []
    for run, c in enumerate([coords, coords, coords[np.random.default_rng(3).permutation(n)]]):
        md = metadata(c)
        tk, got_cap = table_of(md)
        assert got_cap == cap
        if run == 0:
            assert_forced_preconditions(tk, c, cap, forced, absent)
        nbr = md.subm_table(FULL, filt)
        assert nbr.shape == (int(np.prod(filt)), _ops().pad128(n))
        t = nbr.cpu().numpy().astype(np.int64)
        assert np.all(t[:, n:] == -1)
        assert np.array_equal(t[:, :n], rules_to_table(O.submanifold_rulebook(c, filt), n)), f"run {run}"
        tables.append(t)
    assert np.array_equal(tables[0], tables[1])


@pytest.mark.gpu
def test_forced_strided_hash_path():
    """The strided rulebook through the hash (the modules' path): coarse keys chosen first so that they collide -- a
    wrapping chain and a 4-bucket chain in the coarse table of capacity(n_fine) slots -- then 1..8 fine children each."""
    rng = np.random.default_rng(4)
    n_fine = 512
    cap = capacity(n_fine)
    nb = cap // 8
    coarse = forced_sites(cap, {nb - 1: 30, 17: 30}, rng, batch=(0, 3), coords_hi=32768)
    kids = []
    for c in coarse:
        offs = np.argwhere(np.ones((2, 2, 2), bool))
        pick = offs[rng.permutation(8)[:int(rng.integers(1, 9))]]
        kids.append(np.concatenate([2 * c[None, :3] + pick, np.full((pick.shape[0], 1), c[3])], 1))
    fine = np.concatenate(kids)
    while fine.shape[0] < n_fine:          # the rest: random fine sites elsewhere
        c = np.concatenate([rng.integers(0, 65536, size=(1, 3)), rng.integers(3, 5, size=(1, 1))], 1)
        if not np.isin(O.pack_keys(c), O.pack_keys(fine)).any():
            fine = np.concatenate([fine, c])
    fine = fine[:n_fine][rng.permutation(n_fine)]
    out_sp = (32768,) * 3
    for run in range(2):
        f = fine if run == 0 else fine[rng.permutation(n_fine)]
        md = metadata(f)
        rule = md.strided_rule(FULL, (2, 2, 2), (2, 2, 2))
        out_coords, rules, osp = O.strided_rulebook(f, (2, 2, 2), (2, 2, 2), FULL)
        assert osp == out_sp and rule.n_out == out_coords.shape[0]
        tk, got_cap = table_of(md, out_sp)
        assert got_cap == cap
        ckeys = O.pack_keys(out_coords)
        occ, wrapped = bucket_model(ckeys, cap)
        d, h = check_placement(tk, ckeys, cap)
        assert wrapped > 8 and np.any((h == nb - 1) & (d >= 2)) and np.any((h == 17) & (d >= 3))
        gmap = np.searchsorted(ckeys, O.pack_keys(md.coords(out_sp).cpu().numpy()))
        down = rule.down[:, :rule.n_out].cpu().numpy().astype(np.int64)
        assert np.array_equal(to_oracle(down, gmap, np.arange(n_fine)), rules_to_table(rules, rule.n_out))
        up = rule.up[:, :n_fine].cpu().numpy().astype(np.int64)
        assert np.array_equal(to_oracle(up, np.arange(n_fine), gmap), rules_to_table([r[:, ::-1] for r in rules], n_fine))
        assert np.all(rule.down[:, rule.n_out:].cpu().numpy() == -1) and np.all(rule.up[:, n_fine:].cpu().numpy() == -1)


# --------------------------------------------------------------------------------------- C: heavy duplication


@pytest.mark.gpu
@pytest.mark.parametrize("distinct", [1, 12, 1000])
def test_heavy_duplication(distinct):
    """2 M shuffled rows over 1, 12 or 1000 distinct sites: every duplicate races for its key's slot and the smallest
    row index must win.  The 12 keys share one home bucket of the 512 K-bucket table, so they also overflow it while
    racing.  Rows, sites and the mode-3 / mode-4 features (integer values: exact in fp32) against the oracle."""
    import sparseconvnet as scn
    rng = np.random.default_rng(5 + distinct)
    n = 2_000_000
    cap = capacity(n)
    if distinct == 12:
        sites = forced_sites(cap, {int(rng.integers(0, cap // 8)): 12}, rng, batch=(0, 3))
    else:
        sites = random_sites(distinct, (64, 64, 64), 2, seed=distinct)
    c = sites[np.concatenate([np.arange(distinct), rng.integers(0, distinct, n - distinct)])]
    c = c[rng.permutation(n)]
    feats = torch.as_tensor(rng.integers(0, 4, size=(n, 2)).astype(np.float32))
    rows_ref, active_ref = O.input_layer_rules(c)
    for mode in (3, 4):
        x = scn.InputLayer(3, list(FULL), mode=mode)((torch.as_tensor(c).cuda(), feats.cuda(), 0))
        md = x.metadata
        assert np.array_equal(md.row_of_input.cpu().numpy().astype(np.int64), rows_ref)
        assert np.array_equal(md.coords(FULL).cpu().numpy(), active_ref)
        want = O.input_layer_forward(feats.double(), rows_ref, active_ref.shape[0], mode).float()
        assert torch.equal(x.features.cpu(), want), f"mode {mode}"
        tk, got_cap = table_of(md)
        d, h = check_placement(tk, O.pack_keys(sites), got_cap)
        if distinct == 12:
            assert got_cap == cap and d.max() >= 1, "the 12 keys did not overflow their home bucket"


@pytest.mark.gpu
def test_strided_all_children_present():
    """Every coarse site has all 8 fine sites: each column of the down table is full."""
    rng = np.random.default_rng(6)
    coarse = random_sites(20000, (200, 100, 250), 2, seed=7)
    offs = np.argwhere(np.ones((2, 2, 2), bool))
    fine = (np.concatenate([2 * coarse[:, None, :3] + offs[None], np.broadcast_to(coarse[:, None, 3:], (coarse.shape[0], 8, 1))], 2)
            .reshape(-1, 4))
    fine = fine[rng.permutation(fine.shape[0])]
    grid = (400, 200, 500)
    md = metadata(fine, grid)
    rule = md.strided_rule(grid, (2, 2, 2), (2, 2, 2))
    out_coords, rules, osp = O.strided_rulebook(fine, (2, 2, 2), (2, 2, 2), grid)
    gmap = np.searchsorted(O.pack_keys(out_coords), O.pack_keys(md.coords(osp).cpu().numpy()))
    down = rule.down[:, :rule.n_out].cpu().numpy().astype(np.int64)
    assert np.all(down >= 0)
    assert np.array_equal(to_oracle(down, gmap, np.arange(fine.shape[0])), rules_to_table(rules, rule.n_out))


# --------------------------------------------------------------------------------------- D: key-field edges


EDGE_C = [0, 1, 65534, 65535]
EDGE_B = [0, 32767, 32768, 65534]


def edge_sites():
    g = np.array(np.meshgrid(EDGE_C, EDGE_C, EDGE_C, EDGE_B, indexing="ij")).reshape(4, -1).T
    return g[np.random.default_rng(8).permutation(g.shape[0])].astype(np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.int64, torch.int32, torch.float32, torch.float64])
def test_key_field_edges(dtype):
    """Coordinates 0, 1, 65534, 65535 on every axis and batch indices on both sides of the key's top bit: the ±2 steps
    of a 5^3 filter may not borrow into the next field, and the (2,2,2) map at 65535 keeps its batch."""
    ci = edge_sites()
    md = metadata(ci, FULL, dtype=dtype)
    assert md.max_batch_index == 65534
    check_level_rulebooks(md, ci, FULL, (5, 5, 5), (3, 3, 3), (2, 2, 2), levels=2)


@pytest.mark.gpu
@pytest.mark.parametrize("bad", [(0, 0, 0, 65535), (-1, 0, 0, 0), (0, 65536, 0, 0), (0, 0, 0, -1)])
def test_key_field_out_of_range_raises(bad):
    ok = edge_sites()[:10]
    for dtype in (torch.int64, torch.float32):
        with pytest.raises(ValueError):
            metadata(np.concatenate([ok, np.asarray([bad])]), FULL, dtype=dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_fractional_coordinates_truncate_like_long(dtype):
    rng = np.random.default_rng(9)
    c = np.concatenate([rng.uniform(-0.99, 65535.9, size=(400, 3)), rng.integers(0, 3, size=(400, 1))], 1)
    c[:4, :3] = [[-0.5, 0.5, 65535.5], [0.99, 1.01, 2.5], [-0.99, 65534.999, 7.0], [3.7, 3.2, 3.9]]
    t = torch.as_tensor(c).to(dtype)
    want = t.long().numpy()
    md = metadata(t, FULL, dtype=dtype)
    assert_input_rules(md, want)


@pytest.mark.gpu
@pytest.mark.parametrize("dimension", [1, 2, 3])
def test_low_dimensions_and_implicit_batch(dimension):
    """dimension 1 and 2 (the unused key fields are 0), and coords without a batch column (batch 0)."""
    rng = np.random.default_rng(10 + dimension)
    c = np.unique(np.concatenate([rng.integers(0, 40, size=(300, dimension)), rng.integers(0, 2, size=(300, 1))], 1), axis=0)
    c = np.concatenate([c, [[65535] * dimension + [65534], [0] * dimension + [32768]]])
    c = c[rng.permutation(c.shape[0])]
    full4 = np.zeros((c.shape[0], 4), np.int64)
    full4[:, :dimension], full4[:, 3] = c[:, :dimension], c[:, dimension]
    sp = (65536,) * dimension
    filt = (5,) * dimension
    md = metadata(c, sp, dimension)
    assert np.array_equal(md.coords(sp).cpu().numpy(), c)
    t = md.subm_table(sp, filt).cpu().numpy().astype(np.int64)[:, :c.shape[0]]
    assert np.array_equal(t, rules_to_table(O.submanifold_rulebook(full4, filt + (1,) * (3 - dimension)), c.shape[0]))
    md0 = metadata(c[:, :dimension], sp, dimension)                       # no batch column
    c0 = np.concatenate([c[:, :dimension], np.zeros((c.shape[0], 1), np.int64)], 1)
    assert_input_rules(md0, c0, sp)


@pytest.mark.gpu
def test_high_batch_indices_on_the_dense_head():
    """Samples 32767, 32768 and 65534 of a 65535-sample batch: the lazy full-extent pooled mean against avg_pool3d of
    the materialised dense tensor (forward and backward), SparseToDense against the float64 dense tensor, and
    SparseGroupNorm against a float64 per-sample group norm."""
    import torch.nn.functional as F
    import sparseconvnet as scn
    grid, C = (2, 3, 4), 4
    coords = random_sites(50, grid, 3, seed=11)
    coords[:, 3] = np.array([32767, 32768, 65534])[coords[:, 3]]
    feats = torch.randn(coords.shape[0], C).double()                  # fp32 values: the GPU's inputs exactly
    f_gpu = feats.float().cuda().requires_grad_(True)
    x = scn.InputLayer(3, list(grid))((torch.as_tensor(coords).cuda(), f_gpu, 0))
    assert x.batch_size() == 65535
    d = scn.SparseToDense(3, C)(x)
    y = F.avg_pool3d(torch.tanh(d), list(grid))
    assert d._dense is None, "the pooled head must run on the rows"
    f64 = feats.clone().requires_grad_(True)
    dense_ref = O.sparse_to_dense_forward(f64, coords, grid, 65535)
    y_ref = F.avg_pool3d(torch.tanh(dense_ref), list(grid))
    assert torch.allclose(y.double().cpu(), y_ref, rtol=1e-5, atol=1e-7)
    w = torch.randn(y.shape, dtype=torch.float64)
    (y * w.float().cuda()).sum().backward()
    (y_ref * w).sum().backward()
    assert torch.allclose(f_gpu.grad.double().cpu(), f64.grad, rtol=1e-5, atol=1e-7)
    assert torch.equal(d.dense().cpu(), dense_ref.detach().float())
    gn = scn.SparseGroupNorm(2, C).cuda()
    with torch.no_grad():
        gn.weight.copy_(torch.linspace(0.5, 1.5, C))
        gn.bias.copy_(torch.linspace(-0.2, 0.3, C))
    z = gn(x).features.double().cpu()
    ref = torch.empty_like(feats)
    for b in np.unique(coords[:, 3]):
        m = torch.as_tensor(coords[:, 3] == b)
        for g in range(2):
            v = feats[m][:, 2 * g:2 * g + 2]
            ref[m, 2 * g:2 * g + 2] = (v - v.mean()) / torch.sqrt(v.var(unbiased=False) + gn.eps)
    ref = ref * gn.weight.detach().double().cpu() + gn.bias.detach().double().cpu()
    assert torch.allclose(z, ref, rtol=1e-4, atol=1e-5)


# --------------------------------------------------------------------------------------- E: both benchmark batches


@pytest.mark.gpu
def test_dune2d_bench_batch_rulebooks_bit_exact():
    """bench.py --dataset dune2d's first batch (64 events x 3 planes, ~9e5 sites): the (1,5,5) stem and (1,3,3) tables at
    all six levels, the five (1,2,2) maps and their transposes, against the oracle."""
    from sparseeventid_b200 import synthetic
    from sparseeventid_b200.scn.core import Metadata
    coords, feats, bs = bench_batch(dataset="dune2d")
    ci = coords.astype(np.int64)
    assert ci.shape[0] > 800_000
    md = Metadata(3, "cuda")
    md.build_input(torch.as_tensor(coords).cuda(), tuple(synthetic.GRID_2D))
    cur = check_level_rulebooks(md, ci, tuple(synthetic.GRID_2D), (1, 5, 5), (1, 3, 3), (1, 2, 2))
    assert cur.shape[0] > 1000


def _larcv_pair(arr, layout):
    from sparseeventid_b200 import data_transforms as T
    host = T.larcvsparse_to_scnsparse_3d if layout == 0 else T.larcvsparse_to_scnsparse_2d
    dev = T.larcvsparse_to_scnsparse_3d_gpu if layout == 0 else T.larcvsparse_to_scnsparse_2d_gpu
    ch, fh, bh = host(arr)
    cg, fg, bg = dev(torch.from_numpy(np.ascontiguousarray(arr)).cuda())
    assert bh == bg == arr.shape[0]
    assert cg.dtype == torch.int32 and tuple(cg.shape) == (ch.shape[0], 4)
    assert np.array_equal(cg.cpu().numpy().astype(np.int64), np.asarray(ch).astype(np.int64)), "coordinates / row order"
    assert np.array_equal(fg.cpu().numpy(), np.asarray(fh, dtype=np.float32)), "features"
    return ch.shape[0]


@pytest.mark.gpu
@pytest.mark.parametrize("dataset", ["dune3d", "dune2d"])
def test_device_larcv_transform_on_full_bench_arrays(dataset):
    from sparseeventid_b200 import synthetic
    arr = synthetic.larcv_batch_3d(64, seed=1234) if dataset == "dune3d" else synthetic.larcv_batch_2d(64, seed=1234)
    assert arr.shape == ((64, 1, 50000, 4) if dataset == "dune3d" else (64, 3, 50000, 3))
    assert _larcv_pair(arr, 0 if dataset == "dune3d" else 1) > 400_000


@pytest.mark.gpu
@pytest.mark.parametrize("V", [1, 255, 256, 257, 1000])
@pytest.mark.parametrize("layout", [0, 1])
def test_device_larcv_transform_edges(V, layout):
    """Samples with no live row, with no padding, with padding between live rows (the last live row at V - 1), and
    V around the 256-row pass of the compaction."""
    rng = np.random.default_rng(V + 7 * layout)
    P, ncol = (1, 4) if layout == 0 else (3, 3)
    B = 5
    arr = np.concatenate([rng.integers(0, 1000, size=(B, P, V, ncol - 1)).astype(np.float32),
                          rng.normal(size=(B, P, V, 1)).astype(np.float32)], 3)
    value = arr[..., -1]                                            # a view
    value[0] = -999.0                                               # sample 0: all padding; sample 1: none
    live = rng.random((B, P, V)) < 0.5
    live[..., -1] = True                                            # the last row is live
    value[2:][~live[2:]] = -999.0                                   # padding between live rows
    value[4, :, : V // 2] = -999.0                                  # a padded prefix
    _larcv_pair(arr, layout)
    _larcv_pair(np.full_like(arr, -999.0), layout)                # no live row anywhere


# --------------------------------------------------------------------------------------- F: remaining entry points


def _strided_hash(keys_u64, stride):
    """scn_strided_rulebook_hash on device keys -> (keys_out uint64 [m], out_row_of_in, off_of_in)."""
    kout, orow, off, _ = _ops().strided_rulebook(torch.as_tensor(keys_u64.view(np.int64)).cuda(), stride)
    return kout.cpu().numpy().view(np.uint64), orow.cpu().numpy(), off.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("stride", [(2, 2, 2), (1, 2, 2), (4, 4, 4)])
def test_strided_rulebook_bit_exact(stride):
    """Output rows in FIRST-APPEARANCE order over the input rows (SparseConvNet's order), across batch indices 0, 1,
    32767, 32768 and 65534 and the 16-bit edge coordinates.  The oracle numbers rows by ascending key: its rows are
    renumbered by the first input row that reaches each."""
    c = blob_sites(800, (40, 30, 50), 5, seed=12)
    c[:, 3] = np.array([0, 1, 32767, 32768, 65534])[c[:, 3]]
    c = np.concatenate([c, edge_sites()])
    c = c[np.random.default_rng(13).permutation(c.shape[0])]
    out_coords, rules, _ = O.strided_rulebook(c, stride, stride, FULL)
    sorted_row, want_off = np.full(c.shape[0], -1), np.full(c.shape[0], -1)
    for k, r in enumerate(rules):
        sorted_row[r[:, 0]], want_off[r[:, 0]] = r[:, 1], k
    assert sorted_row.min() >= 0
    rows, first = np.unique(sorted_row, return_index=True)
    order = rows[np.argsort(first)]                      # oracle rows in first-appearance order
    renumber = np.empty_like(order)
    renumber[order] = np.arange(order.shape[0])
    for run in range(2):
        kout, orow, off = _strided_hash(O.pack_keys(c), stride)
        assert np.array_equal(kout, O.pack_keys(out_coords)[order])
        assert np.array_equal(orow, renumber[sorted_row]) and np.array_equal(off, want_off)


@pytest.mark.gpu
@pytest.mark.parametrize("order", ["2x2_then_4", "4_then_2x2"])
def test_strided_remap_branch(order):
    """A coarse level that already exists is re-indexed through scn_hash_lookup: S -> S/2 -> S/4 and then a
    Convolution(4, 4) from S, and the reverse.  Down and up tables against the oracle in the existing level's rows."""
    grid = (32, 24, 40)
    c = blob_sites(900, grid, 3, seed=14)
    c[:, 3] = np.array([0, 32768, 65534])[c[:, 3]]
    c = c[np.random.default_rng(15).permutation(c.shape[0])]
    md = metadata(c, grid)
    half = (16, 12, 20)
    steps = [(grid, 2), (half, 2), (grid, 4)] if order == "2x2_then_4" else [(grid, 4), (grid, 2), (half, 2)]
    sites = {grid: c}
    for sp, s in steps:
        rule = md.strided_rule(sp, (s,) * 3, (s,) * 3)
        out_coords, rules, osp = O.strided_rulebook(sites[sp], (s,) * 3, (s,) * 3, sp)
        sites.setdefault(osp, out_coords)
        # GPU rows of both levels -> oracle rows (oracle: ascending key; GPU: the level's own numbering)
        fmap = np.searchsorted(O.pack_keys(sites[sp]), O.pack_keys(md.coords(sp).cpu().numpy())) if sp != grid \
            else np.arange(c.shape[0])
        if sp != grid:
            fine_gpu = md.coords(sp).cpu().numpy()
            assert np.array_equal(np.sort(O.pack_keys(fine_gpu)), np.sort(O.pack_keys(sites[sp])))
        gloc = md.coords(osp).cpu().numpy()
        okeys = O.pack_keys(out_coords)
        assert rule.n_out == gloc.shape[0] == okeys.shape[0] and np.array_equal(np.sort(O.pack_keys(gloc)), okeys)
        omap = np.searchsorted(okeys, O.pack_keys(gloc))
        down = rule.down[:, :rule.n_out].cpu().numpy().astype(np.int64)
        assert np.array_equal(to_oracle(down, omap, fmap), rules_to_table(rules, rule.n_out)), f"{sp} / {s}: down"
        up = rule.up[:, :rule.n_in].cpu().numpy().astype(np.int64)
        assert np.array_equal(to_oracle(up, fmap, omap), rules_to_table([r[:, ::-1] for r in rules], rule.n_in)), f"{sp} / {s}: up"
    assert (8, 6, 10) in md.levels and len(md.strided) == 3


def _pairs_raw(nbr):
    """scn_rulebook_count + scn_rulebook_pairs -> (pair_in, pair_out, offsets [K + 1])."""
    L = _lib()
    K, n_pad = nbr.shape
    counts = torch.zeros(K, dtype=torch.int32, device="cuda")
    L.check(L.lib().scn_rulebook_count(nbr.data_ptr(), K, n_pad, n_pad, counts.data_ptr(), L.stream()), "count")
    total = int(counts.sum())
    pin = torch.full((max(total, 1),), -7, dtype=torch.int32, device="cuda")
    pout = torch.full((max(total, 1),), -7, dtype=torch.int32, device="cuda")
    offs = torch.full((K + 1,), -7, dtype=torch.int32, device="cuda")
    wsb = int(L.lib().scn_rulebook_workspace(K, n_pad))
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    L.check(L.lib().scn_rulebook_pairs(nbr.data_ptr(), K, n_pad, n_pad, pin.data_ptr(), pout.data_ptr(), offs.data_ptr(),
                                       ws.data_ptr(), wsb, L.stream()), "pairs")
    return pin.cpu().numpy()[:total], pout.cpu().numpy()[:total], offs.cpu().numpy(), counts.cpu().numpy()


def _assert_pairs_match_table(nbr):
    t = nbr.cpu().numpy()
    pin, pout, offs, counts = _pairs_raw(nbr)
    k_of, o_of = np.nonzero(t >= 0)                  # (k, out) order
    assert np.array_equal(pin, t[k_of, o_of]) and np.array_equal(pout, o_of)
    want_offs = np.concatenate([[0], np.cumsum((t >= 0).sum(1))])
    assert np.array_equal(offs, want_offs) and np.array_equal(counts, np.diff(want_offs))


@pytest.mark.gpu
def test_rulebook_pairs_of_the_bench_stem_table():
    from sparseeventid_b200 import synthetic
    coords, _, _ = bench_batch()
    md = metadata(coords.astype(np.int64), tuple(synthetic.GRID_3D))
    _assert_pairs_match_table(md.subm_table(tuple(synthetic.GRID_3D), (5, 5, 5)))


@pytest.mark.gpu
def test_rulebook_pairs_with_empty_first_and_last_offsets():
    rng = np.random.default_rng(16)
    K, n = 7, 300
    t = np.where(rng.random((K, 384)) < 0.3, rng.integers(0, n, (K, 384)), -1).astype(np.int32)
    t[0], t[-1], t[:, n:] = -1, -1, -1
    _assert_pairs_match_table(torch.as_tensor(t).cuda())


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 127, 128, 129])
def test_row_count_edges(n):
    """Tables of n rows are padded to a multiple of 128 columns, every padding column -1."""
    c = random_sites(n, (6, 6, 6), 2, seed=n)
    grid = (6, 6, 6)
    md = metadata(c, grid)
    pad = _ops().pad128(n)
    for filt in ((3, 3, 3), (1, 1, 1)):
        t = md.subm_table(grid, filt).cpu().numpy().astype(np.int64)
        assert t.shape == (int(np.prod(filt)), pad) and np.all(t[:, n:] == -1)
        assert np.array_equal(t[:, :n], rules_to_table(O.submanifold_rulebook(c, filt), n))
    rule = md.strided_rule(grid, (2, 2, 2), (2, 2, 2))
    assert rule.up.shape == (8, pad) and np.all(rule.up[:, n:].cpu().numpy() == -1)
    assert rule.down.shape == (8, _ops().pad128(rule.n_out)) and np.all(rule.down[:, rule.n_out:].cpu().numpy() == -1)
    out_coords, rules, osp = O.strided_rulebook(c, (2, 2, 2), (2, 2, 2), grid)
    omap = np.searchsorted(O.pack_keys(out_coords), O.pack_keys(md.coords(osp).cpu().numpy()))
    down = rule.down[:, :rule.n_out].cpu().numpy().astype(np.int64)
    assert np.array_equal(to_oracle(down, omap, np.arange(n)), rules_to_table(rules, rule.n_out))
