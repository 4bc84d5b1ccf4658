"""The block cache of a context (csrc/lgmi_pool.h) built for the host over a counting fake allocator: its size
buckets, reuse, cap, out-of-memory retry and release rules, and the owner of one block (PoolBuf).  No device
needed."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OOM = 2                      # what the fake allocator returns when its limit is reached
NO_LIMIT = (1 << 64) - 1
BIG_CAP = 1 << 40            # a cache that keeps every released block


@pytest.fixture(scope="module")
def lib():
    """Host build of csrc/lgmi_pool.h through tests/csrc/pool_host.cpp."""
    out = os.path.join(ROOT, "tests", "csrc", "libpool_host.so")
    srcs = [os.path.join(ROOT, "tests", "csrc", "pool_host.cpp"),
            os.path.join(ROOT, "l-giremi_b200", "csrc", "lgmi_pool.h")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-o", out, srcs[0]], check=True)
    lib = ctypes.CDLL(out)
    vp, u64 = ctypes.c_void_p, ctypes.c_uint64
    for name, res, args in [("fake_reset", None, [u64]), ("fake_counts", None, [vp]), ("fake_raw", vp, [u64]),
                            ("pool_new", vp, [u64]), ("pool_delete", None, [vp]), ("pool_bucket", u64, [u64]),
                            ("pool_alloc", ctypes.c_int, [vp, u64, vp]), ("pool_release", None, [vp, vp]),
                            ("pool_destroy", None, [vp]), ("pool_stats", None, [vp, vp]),
                            ("buf_new", vp, []), ("buf_moved", vp, [vp]), ("buf_assign", None, [vp, vp]),
                            ("buf_delete", None, [vp]), ("buf_alloc", ctypes.c_int, [vp, vp, u64, u64]),
                            ("buf_ptr", vp, [vp]), ("buf_size", u64, [vp])]:
        getattr(lib, name).restype = res
        getattr(lib, name).argtypes = args
    return lib


class Fake:
    """The fake allocator's counters: raw allocs (failed ones included), frees, out-of-memory returns, frees of
    unknown pointers, outstanding bytes and blocks."""

    def __init__(self, lib):
        self.lib = lib

    def __call__(self):
        v = np.zeros(6, np.uint64)
        self.lib.fake_counts(v.ctypes.data)
        return dict(zip(["allocs", "frees", "ooms", "bad", "bytes", "blocks"], map(int, v)))


@pytest.fixture
def fake(lib):
    lib.fake_reset(NO_LIMIT)
    f = Fake(lib)
    yield f
    assert f()["bad"] == 0, "a raw free of a pointer that was not outstanding"


@pytest.fixture
def make_pool(lib, fake):
    made = []

    def make(cap):
        made.append(lib.pool_new(cap))
        return made[-1]
    yield make
    for p in made:
        lib.pool_delete(p)
    assert fake()["blocks"] == 0, "a pool left raw blocks behind"


def alloc(lib, pool, n):
    out = ctypes.c_void_p()
    assert lib.pool_alloc(pool, n, ctypes.byref(out)) == 0
    return out.value


def stats(lib, pool):
    v = np.zeros(5, np.uint64)
    lib.pool_stats(pool, v.ctypes.data)
    return dict(zip(["cached", "hits", "misses", "cached_blocks", "live"], map(int, v)))


def test_bucket(lib):
    rng = np.random.default_rng(5)
    ns = [0, 1, 4095, 4096, 4097, 5000, 8191, 8192, 8193, 1 << 20, (1 << 20) + 1, (3 << 30) + 7]
    ns += [int(x) for x in rng.integers(1, 1 << 36, 2000)]
    for n in ns:
        b = lib.pool_bucket(n)
        if n <= 4096:
            assert b == 4096, n
            continue
        step = (1 << (n - 1).bit_length()) // 16   # a sixteenth of the octave n lies in
        assert b % step == 0 and n <= b < n + step, n
        assert b - n <= n // 8, n


def test_reuse_within_slack(lib, fake, make_pool):
    pool = make_pool(BIG_CAP)
    p = alloc(lib, pool, 100_000)
    size = lib.pool_bucket(100_000)
    lib.pool_release(pool, p)
    assert stats(lib, pool)["cached"] == size and fake()["frees"] == 0
    # the smallest request whose bucket the cached block covers within 1/4 slack takes it, with no raw call
    n = min(m for m in range(4097, 100_001, 16) if lib.pool_bucket(m) * 5 // 4 >= size)
    assert alloc(lib, pool, n) == p
    assert fake()["allocs"] == 1 and stats(lib, pool)["hits"] == 1
    lib.pool_release(pool, p)
    # ... and the next smaller bucket does not (nor does a larger request)
    below = max(m for m in range(4097, n) if lib.pool_bucket(m) < lib.pool_bucket(n))
    assert lib.pool_bucket(below) + lib.pool_bucket(below) // 4 < size
    q, r = alloc(lib, pool, below), alloc(lib, pool, 100_001 + size)
    assert p not in (q, r) and fake()["allocs"] == 3 and stats(lib, pool)["cached_blocks"] == 1


def test_repeated_shape_allocates_nothing(lib, fake, make_pool):
    """A batch of a shape seen before: every block comes from the cache."""
    pool = make_pool(BIG_CAP)
    sizes = [int(x) for x in np.random.default_rng(7).integers(1, 1 << 22, 40)] + [1, 8, 8, 4096, 0]
    first = [alloc(lib, pool, n) for n in sizes]
    for p in first:
        lib.pool_release(pool, p)
    raw = fake()["allocs"]
    assert raw == len(sizes)
    for _ in range(3):
        again = [alloc(lib, pool, n) for n in sizes]
        assert sorted(again) == sorted(first) and fake()["allocs"] == raw
        for p in again:
            lib.pool_release(pool, p)
    assert stats(lib, pool)["hits"] == 3 * len(sizes) and fake()["frees"] == 0


def test_cap(lib, fake, make_pool):
    size = lib.pool_bucket(10_000)
    pool = make_pool(2 * size)
    blocks = [alloc(lib, pool, 10_000) for _ in range(3)]
    for p in blocks:
        lib.pool_release(pool, p)
    assert stats(lib, pool)["cached"] == 2 * size and fake()["frees"] == 1  # the third would pass the cap
    pool0 = make_pool(0)
    for n in (1, 5000, 10_000):
        lib.pool_release(pool0, alloc(lib, pool0, n))
    assert stats(lib, pool0)["cached"] == 0 and fake()["frees"] == 1 + 3


def test_out_of_memory_trims_and_retries_once(lib, fake, make_pool):
    pool = make_pool(BIG_CAP)
    a = lib.pool_bucket(1 << 20)
    lib.pool_release(pool, alloc(lib, pool, 1 << 20))
    b = lib.pool_bucket(3 << 20)
    lib.fake_reset(b + a // 2)  # room for the new block only once the cached one is given back
    alloc(lib, pool, 3 << 20)
    assert fake() == dict(allocs=2, frees=1, ooms=1, bad=0, bytes=b, blocks=1)
    assert stats(lib, pool)["cached"] == 0
    # a request that does not fit even then: two attempts, the error comes back, nothing changes
    out = ctypes.c_void_p()
    assert lib.pool_alloc(pool, 8 << 20, ctypes.byref(out)) == OOM
    assert fake() == dict(allocs=4, frees=1, ooms=3, bad=0, bytes=b, blocks=1)
    assert stats(lib, pool)["live"] == 1


def test_foreign_pointer_is_freed_raw(lib, fake, make_pool):
    pool = make_pool(BIG_CAP)
    p = lib.fake_raw(1000)
    lib.pool_release(pool, p)
    assert fake()["frees"] == 1 and fake()["blocks"] == 0 and stats(lib, pool)["cached"] == 0
    lib.pool_release(pool, None)
    assert fake()["frees"] == 1


def test_destroy_frees_cached_and_live_blocks(lib, fake, make_pool):
    pool = make_pool(BIG_CAP)
    blocks = [alloc(lib, pool, n) for n in (100, 50_000, 1 << 20)]
    lib.pool_release(pool, blocks[1])
    lib.pool_destroy(pool)
    assert fake()["frees"] == 3 and fake()["blocks"] == 0
    assert stats(lib, pool) == dict(cached=0, hits=0, misses=3, cached_blocks=0, live=0)
    # the destructor (make_pool's teardown) releases whatever a pool still holds
    alloc(lib, make_pool(BIG_CAP), 7)


def test_owner(lib, fake, make_pool):
    pool = make_pool(0)  # every release is a raw free: counted exactly
    b = lib.buf_new()
    assert lib.buf_size(b) == 0 and lib.buf_ptr(b) is None
    assert lib.buf_alloc(b, pool, 1000, 0) == 0
    p = lib.buf_ptr(b)
    assert lib.buf_size(b) == 1000 and fake()["bytes"] == lib.pool_bucket(4000)
    # move: the block goes along, the source holds nothing and releases nothing
    c = lib.buf_moved(b)
    assert lib.buf_ptr(c) == p and lib.buf_size(c) == 1000 and lib.buf_ptr(b) is None and lib.buf_size(b) == 0
    lib.buf_delete(b)
    assert fake()["frees"] == 0
    # move-assignment releases the block assigned over
    d = lib.buf_new()
    lib.buf_alloc(d, pool, 10, 0)
    lib.buf_assign(d, c)
    assert lib.buf_ptr(d) == p and fake()["frees"] == 1
    lib.buf_delete(c)
    assert fake()["frees"] == 1
    # destruction releases once
    lib.buf_delete(d)
    assert fake()["frees"] == 2 and fake()["blocks"] == 0


def test_owner_reallocation(lib, fake, make_pool):
    pool = make_pool(BIG_CAP)
    b = lib.buf_new()
    lib.buf_alloc(b, pool, 5000, 0)
    p = lib.buf_ptr(b)
    # the block held goes back first: an allocation of the same size gets it again from the cache
    assert lib.buf_alloc(b, pool, 5000, 0) == 0
    assert lib.buf_ptr(b) == p and fake()["allocs"] == 1 and stats(lib, pool)["hits"] == 1
    # with a prefix kept: a new block, the prefix copied, the old block back in the cache
    vals = np.arange(5000, dtype=np.uint32) * 7 + 3
    ctypes.memmove(p, vals.ctypes.data, vals.nbytes)
    assert lib.buf_alloc(b, pool, 20_000, 1234) == 0
    q = lib.buf_ptr(b)
    assert q != p and lib.buf_size(b) == 20_000
    assert np.array_equal(np.ctypeslib.as_array((ctypes.c_uint32 * 1234).from_address(q)), vals[:1234])
    assert stats(lib, pool)["live"] == 1 and stats(lib, pool)["cached"] == lib.pool_bucket(5000 * 4)
    # a failed allocation with a prefix kept leaves the block in place; without, the block is gone
    lib.fake_reset(fake()["bytes"])
    assert lib.buf_alloc(b, pool, 1 << 20, 10) == OOM
    assert lib.buf_ptr(b) == q and lib.buf_size(b) == 20_000 and stats(lib, pool)["live"] == 1
    assert lib.buf_alloc(b, pool, 1 << 20, 0) == OOM
    assert lib.buf_ptr(b) is None and lib.buf_size(b) == 0 and stats(lib, pool)["live"] == 0
    lib.buf_delete(b)
    assert stats(lib, pool)["live"] == 0
