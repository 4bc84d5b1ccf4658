"""The het-anchored plan of a deep unit (plan_het_dense, take_het_form in csrc/lgmi_plan.h), built for the host
through tests/csrc/het_plan_host.cpp: the het site list, the tile lists against a brute-force search for tiles
that hold a needed pair, the K-split of the last wave, the multiply-accumulates and the decision.  No device needed."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

UNIT_DESC = np.dtype([("plane_off", "<u8"), ("n_sites", "<u4"), ("n_reads", "<u4"),
                      ("row_words", "<u4"), ("site_off", "<u4")], align=True)
DENSE_TILE = np.dtype([("a", "u1"), ("b", "u1"), ("I", "<u2"), ("J", "<u2"), ("partial", "<u2"), ("kb0", "<u4"),
                       ("kb1", "<u4")], align=True)
SCALARS = ["H", "H_pad", "fewer", "four", "k_blocks", "S_pad", "tri_macs4", "tri_macs9",
           "off4", "n4", "n_whole4", "macs4", "off9", "n9", "n_whole9", "macs9"]
HET_ONLY, EMIT_COUNTS, SKIP_NONHET = 0x1, 0x2, 0x4
HET_SNP, KNOWN_SNP = 2, 1
BM, BN, BK = 128, 256, 128


@pytest.fixture(scope="module")
def hp():
    out = os.path.join(ROOT, "tests", "csrc", "libhet_plan_host.so")
    srcs = [os.path.join(ROOT, "tests", "csrc", "het_plan_host.cpp"),
            os.path.join(ROOT, "l-giremi_b200", "csrc", "lgmi_plan.h"),
            os.path.join(ROOT, "l-giremi_b200", "csrc", "lgmi_math.cuh"),
            os.path.join(ROOT, "include", "lgmi.h")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-o", out, srcs[0]], check=True)
    lib = ctypes.CDLL(out)
    vp = ctypes.c_void_p
    lib.hp_plan.restype = vp
    lib.hp_plan.argtypes = [vp, ctypes.c_uint32, vp, vp, vp]
    lib.hp_free.argtypes = [vp]
    lib.hp_free.restype = None
    lib.hp_scalars.argtypes = [vp, vp]
    lib.hp_scalars.restype = None
    lib.hp_het.argtypes = [vp, vp]
    lib.hp_het.restype = ctypes.c_uint64
    lib.hp_tiles.argtypes = [vp, vp]
    lib.hp_tiles.restype = ctypes.c_uint64
    lib.hp_take.argtypes = [vp, ctypes.c_uint32, ctypes.c_int]
    lib.hp_take.restype = ctypes.c_int
    return lib


class HetPlan:
    def __init__(self, lib, S, R, het, row_limit=0, num_sms=148, dense_path=4):
        self.lib, self.S, self.R = lib, S, R
        u = np.zeros(1, UNIT_DESC)
        u["n_sites"], u["n_reads"], u["row_words"] = S, R, 4 * ((R + 127) // 128)
        flags = np.full(max(S, 1), KNOWN_SNP, np.uint8)
        flags[np.asarray(het, dtype=np.int64)] = HET_SNP
        cfg = np.array([num_sms, dense_path, 1, 2, 1], np.uint32)
        rc = ctypes.c_int(0)
        self.h = lib.hp_plan(u.ctypes.data, row_limit, cfg.ctypes.data, flags.ctypes.data, ctypes.byref(rc))
        assert self.h, "plan failed: %d" % rc.value
        sc = np.zeros(len(SCALARS), np.uint64)
        lib.hp_scalars(self.h, sc.ctypes.data)
        self.sc = {k: int(v) for k, v in zip(SCALARS, sc)}
        het_out = np.zeros(max(S, 1), np.uint32)
        self.het = het_out[:lib.hp_het(self.h, het_out.ctypes.data)].tolist()
        n = lib.hp_tiles(self.h, None)
        self.tiles = np.zeros(n, DENSE_TILE)
        lib.hp_tiles(self.h, self.tiles.ctypes.data)

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.hp_free(self.h)

    def take(self, mode, host_flags=True):
        return bool(self.lib.hp_take(self.h, mode, int(host_flags)))

    def lst(self, four):
        s = self.sc
        off, n = (s["off4"], s["n4"]) if four else (s["off9"], s["n9"])
        return self.tiles[off:off + n]


def needed_tiles(S, het, g0):
    """Brute force: (a, b, I, J) of every tile holding a pair (het[h], s), s != het[h]."""
    out = set()
    for h, site in enumerate(het):
        for s in range(S):
            if s != site:
                for a in range(g0, 3):
                    for b in range(g0, 3):
                        out.add((a, b, h // BM, s // BN))
    return out


def check_lists(p, S, het):
    k_blocks = p.sc["k_blocks"]
    for four in ([True, False] if p.sc["four"] else [False]):
        L = p.lst(four)
        n_whole = p.sc["n_whole4" if four else "n_whole9"]
        whole, parts = L[:n_whole], L[n_whole:]
        assert np.all(whole["partial"] == 0) and np.all(whole["kb0"] == 0) and np.all(whole["kb1"] == k_blocks)
        got = {}
        for t in L:
            key = (int(t["a"]), int(t["b"]), int(t["I"]), int(t["J"]))
            got.setdefault(key, []).append((int(t["kb0"]), int(t["kb1"])))
        assert set(got) == needed_tiles(S, het, 1 if four else 0)
        for key, ranges in got.items():  # each tile covers K once: whole, or cut into consecutive parts
            ranges.sort()
            assert ranges[0][0] == 0 and ranges[-1][1] == k_blocks
            assert all(x[1] == y[0] for x, y in zip(ranges, ranges[1:]))
        assert np.all(parts["partial"] == 1)
        macs = int(((L["kb1"].astype(np.int64) - L["kb0"]) * BM * BN * BK).sum())
        assert macs == p.sc["macs4" if four else "macs9"]


@pytest.mark.parametrize("S,R,het", [
    (300, 2048, [0, 5, 299]),
    (257, 1024, [256]),                       # one column in the last block: itself only
    (257, 1024, [0, 256]),
    (513, 4096, list(range(0, 513, 4))),      # H = 129
    (600, 8192, list(range(128))),            # H = 128
    (600, 8192, list(range(127))),            # H = 127
    (49, 300, [48]),
    (1000, 2048, list(range(1, 1000, 10))),
])
def test_het_lists_hold_exactly_the_needed_tiles(hp, S, R, het):
    p = HetPlan(hp, S, R, het)
    assert p.het == sorted(het)
    assert p.sc["H"] == len(het) and p.sc["H_pad"] == -(-len(het) // BM) * BM
    check_lists(p, S, sorted(het))


def test_last_wave_is_split_in_k(hp):
    # 3 het row blocks x 4 column blocks x 4 blocks = 48 tiles on 20 SMs: 2 whole waves, 8 tiles cut into 2 parts
    S, R = 1024, 64 * 128
    het = list(range(0, 3 * 128 - 10))
    p = HetPlan(hp, S, R, het, num_sms=20)
    assert p.sc["four"]
    n_whole, n = p.sc["n_whole4"], p.sc["n4"]
    assert n_whole == 40 and n == 40 + 2 * 8
    parts = p.lst(True)[n_whole:]
    assert sorted({(int(t["kb0"]), int(t["kb1"])) for t in parts}) == [(0, 32), (32, 64)]
    check_lists(p, S, het)
    # too few k-blocks to cut: whole tiles only
    q = HetPlan(hp, S, 8 * 128, het, num_sms=20)
    assert q.sc["n_whole4"] == q.sc["n4"] == 48


def test_decision(hp):
    S, R = 2000, 8192
    het = list(range(0, S, 10))
    p = HetPlan(hp, S, R, het)
    assert p.sc["fewer"] and 2 * p.sc["macs4"] <= p.sc["tri_macs4"] and 2 * p.sc["macs9"] <= p.sc["tri_macs9"]
    assert p.take(HET_ONLY | SKIP_NONHET) and p.take(HET_ONLY | SKIP_NONHET | EMIT_COUNTS)
    for mode in (0, HET_ONLY, EMIT_COUNTS, HET_ONLY | EMIT_COUNTS):
        assert not p.take(mode)
    assert not p.take(HET_ONLY | SKIP_NONHET, host_flags=False)
    # a piece of a split unit keeps the all-pairs form
    piece = HetPlan(hp, S, R, het, row_limit=512)
    assert not piece.sc["fewer"] and not piece.take(HET_ONLY | SKIP_NONHET)
    # half the sites het: fewer multiply-accumulates than the triangle, but more than half of them
    half = HetPlan(hp, S, R, list(range(0, S, 2)))
    assert half.sc["tri_macs4"] / 2 < half.sc["macs4"] < half.sc["tri_macs4"] and not half.take(HET_ONLY | SKIP_NONHET)
    # every site het: the rows of the whole square cost more than the triangle
    allhet = HetPlan(hp, S, R, list(range(S)))
    assert allhet.sc["macs9"] >= allhet.sc["tri_macs9"] and not allhet.take(HET_ONLY | SKIP_NONHET)
    # nine blocks only: the four-block lists are empty, the decision uses the nine-block ones
    nine = HetPlan(hp, S, R, het, dense_path=9)
    assert not nine.sc["four"] and nine.sc["n4"] == 0 and nine.take(HET_ONLY | SKIP_NONHET)


def test_no_het_sites(hp):
    p = HetPlan(hp, 700, 4096, [])
    assert p.het == [] and p.sc["H"] == 0 and p.sc["H_pad"] == 0
    assert p.sc["n4"] == p.sc["n9"] == 0 and p.sc["macs4"] == p.sc["macs9"] == 0
    assert p.take(HET_ONLY | SKIP_NONHET)


def test_cfg3_shape_tile_count(hp):
    # the bench's deep unit: 2000 sites x 100 000 reads, 10 % het: 2 row blocks x 8 column blocks x 4 blocks
    rng = np.random.default_rng(0)
    het = sorted(rng.choice(2000, 200, replace=False).tolist())
    p = HetPlan(hp, 2000, 100000, het)
    assert p.sc["four"]
    whole = int(np.sum(p.lst(True)["partial"] == 0))
    assert len({(int(t["a"]), int(t["b"]), int(t["I"]), int(t["J"])) for t in p.lst(True)}) == 64
    assert whole <= 64 and p.sc["macs4"] == 64 * BM * BN * p.sc["k_blocks"] * BK
    assert p.sc["tri_macs4"] / p.sc["macs4"] == pytest.approx(288 / 64)
