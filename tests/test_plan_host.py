"""The batch plan (csrc/lgmi_plan.h) built for the host: which kernel path each unit takes and the work tables
lgmi_batch_create uploads, and the groups lgmi_pipeline_create sets up, each checked against a computation of its
own here.  No device needed."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

UNIT_DESC = np.dtype([("plane_off", "<u8"), ("n_sites", "<u4"), ("n_reads", "<u4"),
                      ("row_words", "<u4"), ("site_off", "<u4")], align=True)
DEV_UNIT = np.dtype([("plane_off", "<u8"), ("dense_off", "<u8"), ("gram_off", "<u8"), ("S", "<u4"), ("R", "<u4"),
                     ("W", "<u4"), ("site_off", "<u4"), ("first_item", "<u4"), ("n_items", "<u4"), ("S_pad", "<u4"),
                     ("tiled", "<u4")], align=True)
ITEM = np.dtype([("unit", "<u4"), ("pair_begin", "<u4"), ("pair_cnt", "<u4"), ("flags", "<u4")])
FAST_ITEM = np.dtype([("plane_off", "<u8"), ("site_off", "<u4"), ("unit", "<u4"), ("item", "<u4"), ("S", "<u2"),
                      ("R", "<u2"), ("W", "<u4"), ("pad", "<u4")], align=True)
TILED_DESC = np.dtype([("item_idx", "<u4"), ("unit", "<u4"), ("pair_begin", "<u4"), ("pair_cnt", "<u4"),
                       ("flags", "<u4"), ("S", "<u4"), ("site_off", "<u4"), ("pad", "<u4"), ("dense_off", "<u8"),
                       ("pad2", "<u8")], align=True)
TILE_ITEM = np.dtype([("unit", "<u4"), ("I", "<u2"), ("J", "<u2")], align=True)
TG_TILE = np.dtype([("plane_off", "<u8"), ("dense_off", "<u8"), ("S", "<u4"), ("W", "<u4"), ("site_off", "<u4"),
                    ("I", "<u2"), ("J", "<u2")], align=True)
DENSE_TILE = np.dtype([("a", "u1"), ("b", "u1"), ("I", "<u2"), ("J", "<u2"), ("partial", "<u2"), ("kb0", "<u4"),
                       ("kb1", "<u4")], align=True)
MEAN_ITEM = np.dtype([("unit", "<u4"), ("site_begin", "<u4")])
TABLES = ["units", "items", "fast_items", "tiled_desc", "tile_items", "gram_tiles", "dense_tiles", "mean_items"]
DTYPES = [DEV_UNIT, ITEM, FAST_ITEM, TILED_DESC, TILE_ITEM, TG_TILE, DENSE_TILE, MEAN_ITEM]
SIZES = ["n_dense", "gram_words", "x_bytes", "xt_words", "oth_words", "oth_sites", "n_candidates", "max_reads",
         "n_tiled_work_items"]
PLAN_FIELDS = ["unit", "S", "W", "S_pad", "k_blocks", "rows", "oth_cap", "four", "plane_off", "gram_off",
               "off4", "n4", "n_whole4", "macs4", "off9", "n9", "n_whole9", "macs9"]

NO_SLOT = NO_GRAM = (1 << 64) - 1
ITEM_FIRST, ITEM_SINGLE, ITEM_FAST, ITEM_TILED, ITEM_TILED_GRAM, ITEM_GRAM = 1, 2, 4, 16, 32, 64
NO_PAIRS, SMALL, TILE_POPC, TILE_GRAM, DEEP = range(5)
PAIRS_MAX = 2048
DEFAULT = dict(num_sms=148, dense_path=4, tile_path=1, min_sites=48, min_reads=8192)
LGMI_ERR_ARG, LGMI_ERR_UNSUPPORTED = -2, -6
HET_SNP = 2


@pytest.fixture(scope="module")
def plan_host():
    """Host build of csrc/lgmi_plan.h through tests/csrc/plan_host.cpp."""
    out = os.path.join(ROOT, "tests", "csrc", "libplan_host.so")
    srcs = [os.path.join(ROOT, "tests", "csrc", "plan_host.cpp"),
            os.path.join(ROOT, "l-giremi_b200", "csrc", "lgmi_plan.h"),
            os.path.join(ROOT, "l-giremi_b200", "csrc", "lgmi_math.cuh"),
            os.path.join(ROOT, "include", "lgmi.h")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-o", out, srcs[0]], check=True)
    lib = ctypes.CDLL(out)
    vp, u32, u64 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64
    lib.p_plan.restype = vp
    lib.p_plan.argtypes = [vp, u32, vp, u64, u64, vp, vp, ctypes.c_char_p, u32]
    lib.p_free.restype = None
    lib.p_free.argtypes = [vp]
    lib.p_table.restype = u64
    lib.p_table.argtypes = [vp, ctypes.c_int, vp]
    lib.p_table_elem.restype = u32
    lib.p_table_elem.argtypes = [ctypes.c_int]
    lib.p_sizes.restype = None
    lib.p_sizes.argtypes = [vp, vp]
    lib.p_dense_plans.restype = u64
    lib.p_dense_plans.argtypes = [vp, vp]
    lib.p_route.restype = u32
    lib.p_route.argtypes = [vp, u32, vp]
    lib.p_het_candidates.restype = u64
    lib.p_het_candidates.argtypes = [vp, u32, vp, vp]
    lib.p_pipeline.restype = vp
    lib.p_pipeline.argtypes = [vp, u32, u32, vp, ctypes.c_char_p, u32]
    lib.p_pipeline_free.restype = None
    lib.p_pipeline_free.argtypes = [vp]
    lib.p_pipeline_sizes.restype = u64
    lib.p_pipeline_sizes.argtypes = [vp, vp]
    lib.p_group.restype = None
    lib.p_group.argtypes = [vp, u32, vp, vp, vp]
    for t, dt in enumerate(DTYPES):
        assert lib.p_table_elem(t) == dt.itemsize, TABLES[t]
    return lib


def row_words(R):
    return 4 * ((R + 127) // 128)


def descs(shapes):
    """Unit descriptors packed back to back; returns (units, plane_words, n_sites)."""
    u = np.zeros(len(shapes), UNIT_DESC)
    word = site = 0
    for k, (S, R) in enumerate(shapes):
        u[k] = (word, S, R, row_words(R), site)
        word += 3 * S * row_words(R)
        site += S
    return u, word, site


def cfg_array(**kw):
    c = dict(DEFAULT, **kw)
    return np.array([c["num_sms"], c["dense_path"], c["tile_path"], c["min_sites"], c["min_reads"]], np.uint32)


def pairs(S, limit=0):
    """Pairs (i, j), i < j < S, with i < limit for a piece: counted one row at a time."""
    return sum(S - 1 - i for i in range(limit if limit else S))


def plan(lib, units, plane_words, n_sites, row_limit=None, **cfg):
    """Every table and size of the plan, as numpy arrays / ints (raises on a planning error)."""
    rl = None if row_limit is None else np.ascontiguousarray(row_limit, np.uint32)
    rc, err = ctypes.c_int(0), ctypes.create_string_buffer(512)
    c = cfg_array(**cfg)
    h = lib.p_plan(units.ctypes.data, len(units), None if rl is None else rl.ctypes.data, plane_words, n_sites,
                   c.ctypes.data, ctypes.byref(rc), err, 512)
    if not h:
        raise ValueError(rc.value, err.value.decode())
    try:
        out = {}
        for t, (name, dt) in enumerate(zip(TABLES, DTYPES)):
            a = np.zeros(lib.p_table(h, t, None), dt)
            lib.p_table(h, t, a.ctypes.data)
            out[name] = a
        sizes = np.zeros(len(SIZES), np.uint64)
        lib.p_sizes(h, sizes.ctypes.data)
        out.update({k: int(v) for k, v in zip(SIZES, sizes)})
        dp = np.zeros((lib.p_dense_plans(h, None), len(PLAN_FIELDS)), np.uint64)
        lib.p_dense_plans(h, dp.ctypes.data)
        out["dense_plans"] = [{k: int(v) for k, v in zip(PLAN_FIELDS, row)} for row in dp]
        return out
    finally:
        lib.p_free(h)


def path_of(p, k):
    """A unit's path as the tables show it."""
    d = p["units"][k]
    if d["gram_off"] != NO_GRAM:
        return DEEP
    if d["tiled"]:
        return TILE_GRAM if d["tiled"] == 2 else TILE_POPC
    return SMALL if k in set(p["fast_items"]["unit"].tolist()) else NO_PAIRS


# (S, R, row limit, config, expected path): both sides of every routing boundary
ROUTES = [
    (64, 256, 0, {}, SMALL), (65, 256, 0, {}, TILE_GRAM), (64, 257, 0, {}, TILE_GRAM), (65, 257, 0, {}, TILE_GRAM),
    (48, 8192, 0, {}, DEEP), (47, 8192, 0, {}, TILE_GRAM), (48, 8191, 0, {}, TILE_GRAM), (47, 8191, 0, {}, TILE_GRAM),
    (47, 65535, 0, {}, TILE_GRAM), (47, 65536, 0, {}, TILE_POPC),
    (0, 10, 0, {}, NO_PAIRS), (1, 10, 0, {}, NO_PAIRS), (2, 10, 0, {}, SMALL), (2, 0, 0, {}, SMALL),
    (65, 256, 0, dict(tile_path=0), TILE_POPC), (47, 65535, 0, dict(tile_path=0), TILE_POPC),
    (48, 8192, 0, dict(dense_path=9), DEEP), (64, 256, 0, dict(dense_path=9), SMALL),
    (48, 8192, 0, dict(min_sites=100, min_reads=20000), TILE_GRAM),
    (100, 20000, 0, dict(min_sites=100, min_reads=20000), DEEP),
    (10, 10, 0, dict(min_sites=2, min_reads=1), DEEP), (1, 10, 0, dict(min_sites=2, min_reads=1), NO_PAIRS),
    (300, 200, 128, {}, TILE_GRAM), (300, 200, 256, {}, TILE_GRAM), (300, 200, 300, {}, TILE_GRAM),
    (300, 70000, 128, {}, DEEP), (300, 70000, 300, {}, DEEP),
    (40, 100, 40, {}, TILE_GRAM), (40, 100, 40, dict(tile_path=0), TILE_POPC), (1, 10, 1, {}, NO_PAIRS),
]


@pytest.mark.parametrize("S,R,limit,cfg,want", ROUTES)
def test_routing(plan_host, S, R, limit, cfg, want):
    """The path of a unit on each side of each boundary, and what the tables derive from it."""
    units, pw, ns = descs([(S, R)])
    c = cfg_array(**cfg)
    assert plan_host.p_route(units.ctypes.data, limit, c.ctypes.data) == want
    p = plan(plan_host, units, pw, ns, [limit] if limit else None, **cfg)
    d = p["units"][0]
    assert path_of(p, 0) == want
    assert d["tiled"] == {TILE_POPC: 1, TILE_GRAM: 2}.get(want, 0)
    assert (d["gram_off"] != NO_GRAM) == (want == DEEP)
    assert len(p["fast_items"]) == (want == SMALL)
    assert len(p["dense_plans"]) == (want == DEEP)
    tiled = want in (TILE_POPC, TILE_GRAM)
    assert len(p["tiled_desc"]) == (len(p["items"]) if tiled else 0)
    assert (len(p["gram_tiles"]) > 0) == (want == TILE_GRAM)
    assert (len(p["tile_items"]) > 0) == (want == TILE_POPC)
    for it in p["items"]:
        assert bool(it["flags"] & ITEM_FAST) == (want == SMALL)
        assert bool(it["flags"] & ITEM_TILED) == tiled
        assert bool(it["flags"] & ITEM_TILED_GRAM) == (want == TILE_GRAM)
        assert bool(it["flags"] & ITEM_GRAM) == (want == DEEP)
    assert p["n_tiled_work_items"] == (len(p["items"]) if tiled or want == DEEP else 0)


# a mixed batch: small, mid-depth (both forms), deep, pair-less and several-item units, pieces of each kind
MIXED = [(50, 200), (2, 6), (0, 0), (1, 9), (70, 300), (130, 17), (700, 120), (64, 256), (33, 1000), (300, 8192),
         (200, 9000), (47, 70000), (520, 400), (600, 8300), (129, 50), (1, 5), (129, 60), (100, 20000),
         (20, 1800)]
MIXED_LIMITS = [0, 0, 0, 0, 0, 0, 256, 0, 0, 128, 0, 0, 512, 0, 128, 1, 0, 0, 0]


def mixed(lib, **cfg):
    units, pw, ns = descs(MIXED)
    return units, plan(lib, units, pw, ns, MIXED_LIMITS, **cfg)


@pytest.mark.parametrize("cfg", [{}, dict(tile_path=0), dict(dense_path=9, num_sms=7)])
def test_items(plan_host, cfg):
    """Items cover each unit's pairs in order, 2 048 at a time; first / single flags; a piece's pair count."""
    units, p = mixed(plan_host, **cfg)
    items = p["items"]
    n = 0
    for k, (S, _R) in enumerate(MIXED):
        limit = MIXED_LIMITS[k]
        np_ = pairs(S, limit)
        d = p["units"][k]
        mine = items[d["first_item"]:d["first_item"] + d["n_items"]]
        assert d["first_item"] == n and (mine["unit"] == k).all()
        n += d["n_items"]
        want_begin = list(range(0, np_, PAIRS_MAX)) or [0]
        assert mine["pair_begin"].tolist() == want_begin
        assert mine["pair_cnt"].tolist() == [min(PAIRS_MAX, np_ - b) for b in want_begin]
        assert [bool(f & ITEM_FIRST) for f in mine["flags"]] == [True] + [False] * (len(mine) - 1)
        single = len(mine) == 1 and not limit
        assert all(bool(f & ITEM_SINGLE) == single for f in mine["flags"])
    assert n == len(items)
    assert p["n_candidates"] == sum(pairs(S, lim) for (S, _R), lim in zip(MIXED, MIXED_LIMITS))
    assert p["max_reads"] == max(R for _S, R in MIXED)
    # a piece's pairs are the first `limit` rows of the pair order (lg_row_off(limit, S))
    assert pairs(700, 256) == 256 * (2 * 700 - 256 - 1) // 2
    # every item of a mid-depth unit has its own record, in item order
    td = p["tiled_desc"]
    assert td["item_idx"].tolist() == [t for t, it in enumerate(items) if it["flags"] & ITEM_TILED]
    for r in td:
        it, d = items[r["item_idx"]], p["units"][r["unit"]]
        assert (r["unit"], r["pair_begin"], r["pair_cnt"], r["flags"]) == tuple(it)
        assert (r["S"], r["site_off"], r["dense_off"]) == (d["S"], d["site_off"], d["dense_off"])


def blocks_with_pair(S, rows, bi, bj):
    """(I, J) of the bi x bj site blocks holding a pair i < j with i < rows (brute force)."""
    out = []
    for I in range(-(-rows // bi)):
        for J in range(-(-S // bj)):
            i_lo = I * bi
            if any(i < j for i in range(i_lo, min(i_lo + bi, rows)) for j in range(J * bj, min(J * bj + bj, S))):
                out.append((I, J))
    return out


def test_mid_depth_tiles(plan_host):
    """k_tile_gram_ws's 128 x 48 tiles and k_tile_mi's 16 x 16 tiles: the blocks with a pair below the row limit,
    deepest unit first (stable), each gram tile carrying its unit's dense slot."""
    for cfg in ({}, dict(tile_path=0)):
        units, p = mixed(plan_host, **cfg)
        gram = p["gram_tiles"]
        tiles = p["tile_items"]
        want_gram, want_tiles = [], []
        for k, (S, R) in enumerate(MIXED):
            rows = MIXED_LIMITS[k] or S
            path = path_of(p, k)
            if path == TILE_GRAM:
                want_gram += [(k, I, J) for I, J in blocks_with_pair(S, rows, 128, 48)]
            if path == TILE_POPC:
                nb = -(-S // 16)
                want_tiles += [(k, I, J) for I in range(-(-rows // 16)) for J in range(I, nb)]
        order = lambda ts: sorted(ts, key=lambda t: -int(units[t[0]]["row_words"]))  # stable: unit, then I, J
        unit_of = {int(u["plane_off"]): k for k, u in enumerate(units) if u["n_sites"]}
        got_gram = [(unit_of[int(t["plane_off"])], int(t["I"]), int(t["J"])) for t in gram]
        assert got_gram == order(want_gram)
        assert [(int(t["unit"]), int(t["I"]), int(t["J"])) for t in tiles] == order(want_tiles)
        assert (len(want_gram) > 0) == (not cfg) and (len(want_tiles) > 0)
        for t in gram:
            k = unit_of[int(t["plane_off"])]
            d = p["units"][k]
            assert t["dense_off"] == d["dense_off"] != NO_SLOT
            assert (t["S"], t["W"], t["site_off"]) == (units[k]["n_sites"], units[k]["row_words"], units[k]["site_off"])


@pytest.mark.parametrize("num_sms", [148, 7, 3])
@pytest.mark.parametrize("dense_path", [4, 9])
@pytest.mark.parametrize("threshold", [(48, 8192), (2, 1)])
def test_dense_tiles(plan_host, num_sms, dense_path, threshold):
    """k_gram_i8's lists: the whole tiles are the needed (a, b, I, J); the last wave's tiles are cut along K into at
    most 8 contiguous parts of at least 8 k-blocks; macs is their sum."""
    units, p = mixed(plan_host, num_sms=num_sms, dense_path=dense_path, min_sites=threshold[0],
                     min_reads=threshold[1])
    dense = p["dense_tiles"]
    deep = [k for k in range(len(MIXED)) if path_of(p, k) == DEEP]
    assert [pl["unit"] for pl in p["dense_plans"]] == deep and deep
    gram_words = 0
    split_seen = False
    for pl in p["dense_plans"]:
        S, R = MIXED[pl["unit"]]
        rows = MIXED_LIMITS[pl["unit"]] or S
        assert pl["S_pad"] == -(-S // 256) * 256 and pl["k_blocks"] == row_words(R) * 32 // 128 and pl["rows"] == rows
        assert pl["gram_off"] == gram_words and p["units"][pl["unit"]]["gram_off"] == gram_words
        gram_words += 9 * pl["S_pad"] ** 2
        assert pl["four"] == (dense_path == 4)
        lists = [(0, pl["off9"], pl["n9"], pl["n_whole9"], pl["macs9"])]
        if pl["four"]:
            lists.append((1, pl["off4"], pl["n4"], pl["n_whole4"], pl["macs4"]))
        for g0, off, n, n_whole, macs in lists:
            L = dense[off:off + n]
            whole, tail = L[:n_whole], L[n_whole:]
            need = {(a, b, I, J) for a in range(g0, 3) for b in range(g0, 3)
                    for I, J in blocks_with_pair(S, rows, 128, 256)}
            assert (whole["partial"] == 0).all() and (whole["kb0"] == 0).all()
            assert (whole["kb1"] == pl["k_blocks"]).all()
            parts = {}
            for t in tail:
                parts.setdefault((int(t["a"]), int(t["b"]), int(t["I"]), int(t["J"])), []).append(
                    (int(t["kb0"]), int(t["kb1"])))
            assert (tail["partial"] == 1).all()
            got = [tuple(int(x) for x in (t["a"], t["b"], t["I"], t["J"])) for t in whole]
            assert len(set(got)) == len(got) and set(got) | set(parts) == need and not set(got) & set(parts)
            for rng in parts.values():
                split_seen = True
                rng.sort()
                assert 2 <= len(rng) <= 8
                assert rng[0][0] == 0 and rng[-1][1] == pl["k_blocks"]
                assert all(x[1] == y[0] for x, y in zip(rng, rng[1:]))
                assert all(e - b >= 8 for b, e in rng)
            assert macs == sum(128 * 256 * 128 * (int(t["kb1"]) - int(t["kb0"])) for t in L)
    assert p["gram_words"] == gram_words
    if num_sms == 7:
        assert split_seen


def test_dense_slots_and_means(plan_host):
    """Dense MI slots: mid-depth units, several-item units and pieces, back to back; pieces have no mean items; the
    mean items cover every other several-item unit in 32-site steps, larger units first."""
    for cfg in ({}, dict(tile_path=0), dict(min_sites=2, min_reads=1)):
        units, p = mixed(plan_host, **cfg)
        at = 0
        want_means = []
        for k, (S, _R) in enumerate(MIXED):
            d = p["units"][k]
            limit = MIXED_LIMITS[k]
            slot = path_of(p, k) in (TILE_POPC, TILE_GRAM) or d["n_items"] > 1 or limit
            if slot:
                assert d["dense_off"] == at
                at += pairs(S, limit)
            else:
                assert d["dense_off"] == NO_SLOT
            if d["n_items"] > 1 and not limit:
                want_means += [(k, s) for s in range(0, S, 32)]
        assert p["n_dense"] == at
        want_means.sort(key=lambda m: -MIXED[m[0]][0])
        assert [tuple(int(x) for x in m) for m in p["mean_items"]] == want_means
        assert not {int(m["unit"]) for m in p["mean_items"]} & {k for k, lim in enumerate(MIXED_LIMITS) if lim}


def het_brute(units, row_limit, flags):
    tot = 0
    for k, u in enumerate(units):
        S, off = int(u["n_sites"]), int(u["site_off"])
        het = (flags[off:off + S] & 3) == HET_SNP
        rows = int(row_limit[k]) if row_limit is not None and row_limit[k] else S
        tot += sum(1 for i in range(rows) for j in range(i + 1, S) if het[i] or het[j])
    return tot


def test_het_candidates(plan_host):
    """Candidate pairs next to a het_snp site, for whole units and pieces, against a count over the pairs."""
    rng = np.random.default_rng(7)
    shapes = [(0, 4), (1, 4), (2, 4), (17, 40), (130, 60), (300, 20), (260, 10)]
    units, _pw, ns = descs(shapes)
    for p_het in (0.0, 0.1, 0.5, 1.0):
        flags = np.where(rng.random(ns) < p_het, HET_SNP, rng.choice([0, 1, 4, 5], ns)).astype(np.uint8)
        for rl in (None, np.array([0, 1, 2, 17, 128, 256, 260], np.uint32)):
            got = plan_host.p_het_candidates(units.ctypes.data, len(units), None if rl is None else rl.ctypes.data,
                                             flags.ctypes.data)
            assert got == het_brute(units, rl, flags)


def test_errors(plan_host):
    """Malformed descriptors: the error code and message of lgmi_batch_create."""
    def err(shapes, row_limit=None, edit=None, extra_words=0):
        units, pw, ns = descs(shapes)
        if edit:
            edit(units)
        with pytest.raises(ValueError) as e:
            plan(plan_host, units, pw + extra_words, ns, row_limit)
        return e.value.args

    assert err([(65536, 4)]) == (LGMI_ERR_UNSUPPORTED, "unit 0: 65536 sites > 65535")

    def w(u):
        u[1]["row_words"] = 8
    assert err([(3, 4), (5, 100)], edit=w) == (
        LGMI_ERR_ARG, "unit 1: inconsistent descriptor (S=5 R=100 W=8 plane_off=36 site_off=3)")

    def unaligned(u):
        u[0]["plane_off"] = 2
    assert err([(5, 100)], edit=unaligned, extra_words=8) == (
        LGMI_ERR_ARG, "unit 0: inconsistent descriptor (S=5 R=100 W=4 plane_off=2 site_off=0)")

    def past_end(u):
        u[0]["plane_off"] = 4
    assert err([(5, 100)], edit=past_end) == (
        LGMI_ERR_ARG, "unit 0: inconsistent descriptor (S=5 R=100 W=4 plane_off=4 site_off=0)")

    def sites(u):
        u[0]["site_off"] = 1
    assert err([(5, 100)], edit=sites) == (
        LGMI_ERR_ARG, "unit 0: inconsistent descriptor (S=5 R=100 W=4 plane_off=0 site_off=1)")

    for limit in (100, 257, 301):
        assert err([(300, 100)], [limit]) == (
            LGMI_ERR_ARG, "unit 0: row limit %d is neither a multiple of 128 below S nor S = 300" % limit)


# --------------------------------------------------------------------------- the groups of a pipelined step
GROUP_FIELDS = ["unit0", "n_units", "plane0", "site0", "tight0", "tight_words", "plane_words", "n_sites"]


def pipeline_plan(lib, units, n_chunks):
    """(groups, n_candidates, max_sites) of plan_pipeline; each group a dict with its rebased descriptors and
    relative tight offsets (raises on a planning error)."""
    units = np.ascontiguousarray(units, UNIT_DESC)
    rc, err = ctypes.c_int(0), ctypes.create_string_buffer(512)
    h = lib.p_pipeline(units.ctypes.data, len(units), n_chunks, ctypes.byref(rc), err, 512)
    if not h:
        raise ValueError(rc.value, err.value.decode())
    try:
        sizes = np.zeros(2, np.uint64)
        groups = []
        for g in range(lib.p_pipeline_sizes(h, sizes.ctypes.data)):
            v = np.zeros(len(GROUP_FIELDS), np.uint64)
            lib.p_group(h, g, v.ctypes.data, None, None)
            grp = {k: int(x) for k, x in zip(GROUP_FIELDS, v)}
            grp["units"] = np.zeros(grp["n_units"], UNIT_DESC)
            grp["tight_off"] = np.zeros(grp["n_units"], np.uint64)
            lib.p_group(h, g, v.ctypes.data, grp["units"].ctypes.data, grp["tight_off"].ctypes.data)
            groups.append(grp)
        return groups, int(sizes[0]), int(sizes[1])
    finally:
        lib.p_pipeline_free(h)


def equal_cost_cut(units, n_chunks, clamp=True):
    """(unit0, n_units) of each group: group c ends at the first unit boundary where the running cost (candidate pairs
    + S * W / 4 + 1 per unit) reaches c + 1 shares of the total, the last group at the end; empty groups are dropped,
    except the one group of a batch without units.  clamp: at most one group per unit."""
    n = len(units)
    cost = [pairs(int(u["n_sites"])) + int(u["n_sites"]) * int(u["row_words"]) // 4 + 1 for u in units]
    prefix = np.concatenate(([0], np.cumsum(cost, dtype=np.int64)))
    total = int(prefix[-1])
    shares = min(n_chunks, max(1, n)) if clamp else n_chunks
    ends = [n if c + 1 == shares else int(np.searchsorted(prefix, total * (c + 1) // shares)) for c in range(shares)]
    bounds = [0] + ends
    return [(a, b - a) for a, b in zip(bounds, bounds[1:]) if b > a] or [(0, 0)]


def tight_layout(units):
    """First word of each unit in the tight two-plane input (rows of ceil(R/32) words, units back to back), and the
    end."""
    S, R = units["n_sites"].astype(np.int64), units["n_reads"].astype(np.int64)
    return np.concatenate(([0], np.cumsum(2 * S * ((R + 31) // 32))))


def check_pipeline(lib, units, n_chunks):
    """plan_pipeline against equal_cost_cut, the descriptors rebased by hand and tight_layout; returns the groups."""
    groups, n_candidates, max_sites = pipeline_plan(lib, units, n_chunks)
    assert [(g["unit0"], g["n_units"]) for g in groups] == equal_cost_cut(units, n_chunks)
    assert 1 <= len(groups) <= min(n_chunks, max(1, len(units)))
    # contiguous, in order, covering [0, n_units)
    assert groups[0]["unit0"] == 0 and groups[-1]["unit0"] + groups[-1]["n_units"] == len(units)
    assert all(a["unit0"] + a["n_units"] == b["unit0"] for a, b in zip(groups, groups[1:]))
    tight = tight_layout(units)
    for g in groups:
        mine = units[g["unit0"]:g["unit0"] + g["n_units"]]
        S, W = mine["n_sites"].astype(np.int64), mine["row_words"].astype(np.int64)
        assert g["plane0"] == (int(mine[0]["plane_off"]) if len(mine) else 0)
        assert g["site0"] == (int(mine[0]["site_off"]) if len(mine) else 0)
        want = mine.copy()
        want["plane_off"] -= g["plane0"]
        want["site_off"] -= g["site0"]
        assert g["units"].tobytes() == want.tobytes()
        assert g["plane_words"] == int((3 * S * W).sum()) and g["n_sites"] == int(S.sum())
        assert g["tight0"] == tight[g["unit0"]]
        assert g["tight_words"] == tight[g["unit0"] + g["n_units"]] - g["tight0"]
        assert g["tight_off"].tolist() == (tight[g["unit0"]:g["unit0"] + g["n_units"]] - g["tight0"]).tolist()
    assert n_candidates == sum(pairs(int(S)) for S in units["n_sites"])
    assert max_sites == max((int(S) for S in units["n_sites"]), default=0)
    return groups


@pytest.mark.parametrize("n_chunks", [1, 2, 5, 64])
def test_pipeline_groups_heavy_tail(plan_host, lg, n_chunks):
    """The 90-unit heavy tail of the GPU pipeline test: the equal-cost cut, and the relative tight offsets pick each
    unit's rows out of PlaneBatch.packed2(tight=True) (the padded two-plane rows without their padding)."""
    import importlib
    synth = importlib.import_module("l-giremi_b200.synth")
    pb, _ = synth.make_heavy_tail(20261024, 90, s_max=200, r_max=3000)
    groups = check_pipeline(plan_host, pb.units, n_chunks)
    assert len(groups) == n_chunks or n_chunks == 64
    padded, tight = pb.packed2(), pb.packed2(tight=True)
    assert groups[-1]["tight0"] + groups[-1]["tight_words"] == tight.size
    for g in groups:
        for q, u in enumerate(g["units"]):
            k = g["unit0"] + q
            S, W, wt = int(u["n_sites"]), int(u["row_words"]), (int(u["n_reads"]) + 31) // 32
            rows = tight[g["tight0"] + int(g["tight_off"][q]):][:2 * S * wt].reshape(S, 2, wt)
            want = padded[int(pb.units["plane_off"][k]) // 3 * 2:][:2 * S * W].reshape(S, 2, W)[:, :, :wt]
            assert np.array_equal(rows, want)


def test_pipeline_groups_uniform(plan_host):
    """A cfg2-like table (20 000 units of 50 sites x 200 reads) in 4 groups of 5 000 units."""
    units, pw, ns = descs([(50, 200)] * 20000)
    groups = check_pipeline(plan_host, units, 4)
    assert [g["n_units"] for g in groups] == [5000] * 4
    assert sum(g["plane_words"] for g in groups) == pw and sum(g["n_sites"] for g in groups) == ns


def test_pipeline_groups_edge_cases(plan_host):
    """More groups asked for than units, a unit that outweighs whole shares, no units at all, one unit."""
    # at most one group per unit: cut into 64 shares instead of 3, these units would make three groups, not two
    units, _, _ = descs([(2, 10), (4, 10), (2, 10)])
    assert equal_cost_cut(units, 64, clamp=False) == [(0, 1), (1, 1), (2, 1)]
    assert [(g["unit0"], g["n_units"]) for g in check_pipeline(plan_host, units, 64)] == [(0, 2), (2, 1)]
    # a dominant unit covers the shares of several groups: those groups are skipped, not left empty
    units, _, _ = descs([(10, 10)] * 3 + [(2000, 100)] + [(10, 10)] * 3)
    groups = check_pipeline(plan_host, units, 4)
    assert [(g["unit0"], g["n_units"]) for g in groups] == [(0, 4), (4, 3)]
    # no units: one empty group
    units, _, _ = descs([])
    for n_chunks in (1, 4):
        groups = check_pipeline(plan_host, units, n_chunks)
        assert len(groups) == 1 and groups[0]["n_units"] == 0 and groups[0]["plane_words"] == groups[0]["n_sites"] == 0
    # one unit, and units without pairs
    for shapes in ([(300, 5000)], [(0, 0), (1, 7), (0, 0)]):
        units, _, _ = descs(shapes)
        assert len(check_pipeline(plan_host, units, 8)) == len(shapes)


def test_pipeline_groups_random(plan_host):
    """Random tables, with units without pairs among them, at random group counts."""
    rng = np.random.default_rng(11)
    for _ in range(40):
        n = int(rng.integers(0, 60))
        shapes = [(int(rng.choice([0, 1, 2, int(rng.integers(2, 400))])), int(rng.integers(0, 5000))) for _ in range(n)]
        units, _, _ = descs(shapes)
        check_pipeline(plan_host, units, int(rng.integers(1, 80)))


def test_pipeline_errors(plan_host):
    """No groups, and units that are not back to back: the error code and message of lgmi_pipeline_create, naming
    the first unit out of place."""
    def err(units, n_chunks):
        with pytest.raises(ValueError) as e:
            pipeline_plan(plan_host, units, n_chunks)
        return e.value.args

    units, _, _ = descs([(5, 40)] * 4)
    assert err(units, 0) == (LGMI_ERR_ARG, "lgmi_pipeline_create: n_chunks must be >= 1")
    assert err(units[::-1], 2) == (LGMI_ERR_UNSUPPORTED, "lgmi_pipeline_create: unit 1 is not laid out right after unit 0")
    gap = units.copy()
    gap["plane_off"][2:] += 4
    assert err(gap, 2) == (LGMI_ERR_UNSUPPORTED, "lgmi_pipeline_create: unit 2 is not laid out right after unit 1")
    sites = units.copy()
    sites["site_off"][3] += 1
    gap["site_off"][3] += 1
    assert err(sites, 1) == (LGMI_ERR_UNSUPPORTED, "lgmi_pipeline_create: unit 3 is not laid out right after unit 2")
    assert err(gap, 1) == (LGMI_ERR_UNSUPPORTED, "lgmi_pipeline_create: unit 2 is not laid out right after unit 1")
    # the first unit may start anywhere
    start = units.copy()
    start["plane_off"] += 8
    start["site_off"] += 3
    groups = check_pipeline(plan_host, start, 2)
    assert groups[0]["plane0"] == 8 and groups[0]["site0"] == 3
