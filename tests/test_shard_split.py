"""Deep units split over the processes of a one-process-per-GPU launch (l-giremi_b200/shard.py: local_run,
gather_run_to_rank0; lgmi_piece_export, lgmi_batch_copy_planes_ipc, lgmi_split_means_ipc).

On the CPU: every rank derives the same piece plan, the layout of lgmi_piece_ipc matches its ctypes mirror, and a
two-rank gloo gather of hand-made shard and piece results is what merge_shards builds in one process.  On the GPU:
two ranks (one device each, or both on device 0, which exercises CUDA IPC between two processes on one device) split
a deep unit among ordinary units, and rank 0's merged result is one process's step over the whole batch, bit for bit."""
import ctypes
import importlib
import os
import socket
import subprocess
from concurrent.futures import ProcessPoolExecutor
import multiprocessing

import numpy as np
import pytest
from numpy.random import PCG64, Generator

from conftest import ROOT

lg_mod = importlib.import_module("l-giremi_b200")
L = importlib.import_module("l-giremi_b200._lib")
mg = importlib.import_module("l-giremi_b200.multigpu")
enc = importlib.import_module("l-giremi_b200.encode")
synth = importlib.import_module("l-giremi_b200.synth")


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _descs(shapes):
    u = np.zeros(len(shapes), dtype=L.UNIT_DESC)
    u['n_sites'] = [s for s, _r in shapes]
    u['n_reads'] = [r for _s, r in shapes]
    u['row_words'] = 4 * ((u['n_reads'] + 127) // 128)
    u['site_off'] = np.concatenate(([0], np.cumsum(u['n_sites'])[:-1]))
    return u


def _cfg4_plus_cfg3():
    S, R = synth.heavy_tail_shapes(Generator(PCG64(20261022)), 20000)    # make_heavy_tail(20261022, 20000)'s shapes
    return _descs(list(zip(S.tolist(), R.tolist())) + [(2000, 100000)])


def _plan_in_process(world):
    """What one rank of a fresh process derives (no state shared with the caller)."""
    shards, pieces, splits = mg.plan_pieces(_cfg4_plus_cfg3(), world)
    return [s.tolist() for s in shards], pieces, {u: list(map(int, b)) for u, b in splits.items()}


# --------------------------------------------------------------------------- no device
@pytest.mark.timeout(600)
def test_every_rank_derives_the_same_piece_plan():
    """local_run exchanges no plan: each rank's own plan_pieces must agree, at world sizes 2, 4 and 8."""
    units = _cfg4_plus_cfg3()
    deep = len(units) - 1
    with ProcessPoolExecutor(max_workers=4, mp_context=multiprocessing.get_context("spawn")) as pool:
        for world in (2, 4, 8):
            plans = list(pool.map(_plan_in_process, [world] * world))
            assert all(p == plans[0] for p in plans[1:])
            shards, pieces, splits = plans[0]
            assert list(splits) == [deep] and len(splits[deep]) >= 3
            got = sorted((a, e) for p in pieces for u, a, e in p if u == deep)
            assert got == list(zip(splits[deep][:-1], splits[deep][1:]))
            assert sorted(u for s in shards for u in s) == list(range(deep))
            assert _plan_in_process(world) == plans[0]


def test_piece_ipc_layout_matches_the_header():
    out = os.path.join(ROOT, "tests", "csrc", "libipc_host.so")
    srcs = [os.path.join(ROOT, "tests", "csrc", "ipc_host.cpp"), os.path.join(ROOT, "include", "lgmi.h")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-o", out, srcs[0]], check=True)
    lib = ctypes.CDLL(out)
    lib.piece_ipc_size.restype = ctypes.c_uint64
    lib.piece_ipc_offset.restype = ctypes.c_int64
    lib.piece_ipc_offset.argtypes = [ctypes.c_char_p]
    assert ctypes.sizeof(L.PieceIpc) == lib.piece_ipc_size() == 288
    for name, _t in L.PieceIpc._fields_:
        assert getattr(L.PieceIpc, name).offset == lib.piece_ipc_offset(name.encode()), name


# hand-made results of a world of ordinary units and one unit that plan_pieces splits between two ranks
def _world():
    shapes = [(40, 150)] * 12 + [(300, 2000)] + [(25, 90)] * 9
    units = _descs(shapes)
    n_sites = int(units['n_sites'].sum())
    pb = enc.PlaneBatch(units, np.zeros(0, np.uint32), np.zeros(n_sites, np.uint8))
    rng = np.random.default_rng(5150)
    rows = []              # per unit: its records (unit field 0), tables, per-site means and counts
    for S in units['n_sites'].tolist():
        i, j = np.triu_indices(S, 1)
        keep = rng.random(len(i)) < 0.3
        rec = np.zeros(int(keep.sum()), dtype=L.PAIR_REC)
        rec['i'], rec['j'], rec['mi'] = i[keep], j[keep], rng.random(int(keep.sum()))
        tab = rng.integers(0, 1000, size=(len(rec), 9)).astype(np.uint32)
        mean = np.where(rng.random(S) < 0.2, np.nan, rng.random(S))
        rows.append((rec, tab, mean, rng.integers(0, 50, size=S).astype(np.uint32)))
    return pb, rows


def _shard_result(rows, index):
    r = type("Shard", (), {})()
    recs = []
    for k, g in enumerate(index):
        rec = rows[g][0].copy()
        rec['unit'] = k
        recs.append(rec)
    r.records = np.concatenate(recs) if recs else np.zeros(0, L.PAIR_REC)
    r.counts = np.concatenate([rows[g][1] for g in index]) if len(index) else np.zeros((0, 9), np.uint32)
    r.site_mean = np.concatenate([rows[g][2] for g in index]) if len(index) else np.zeros(0)
    r.site_cnt = np.concatenate([rows[g][3] for g in index]) if len(index) else np.zeros(0, np.uint32)
    r.unit_rec_off = np.concatenate(([0], np.cumsum([len(rows[g][0]) for g in index]))).astype(np.uint64)
    return r


def _local(shard_mod, pb, rows, rank, world):
    """What local_run would leave on `rank`, from the hand-made rows."""
    shards, pieces, splits = mg.plan_pieces(pb.units, world)
    index = shards[rank]
    mine = []
    for u, a, e in pieces[rank]:
        rec, tab = rows[u][0], rows[u][1]
        sel = (rec['i'] >= a) & (rec['i'] < e)
        r = rec[sel].copy()
        r['unit'] = 7                                  # a piece's unit field is its index in the piece batch
        r['i'] -= a
        r['j'] -= a
        mine.append((u, a, e, r, tab[sel]))
    means = {u: rows[u][2:] for u, a, _e in pieces[rank] if a == 0}
    return shard_mod.LocalRun(_shard_result(rows, index) if len(index) else None, index, mine, means), shards, pieces


def _gather_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    shard = importlib.import_module("l-giremi_b200.shard")
    pb, rows = _world()
    run, _s, _p = _local(shard, pb, rows, rank, world)
    merged = shard.gather_run_to_rank0(pb, run, device="cpu")
    if rank == 0:
        np.savez(os.path.join(out_dir, "merged.npz"), records=merged.records, counts=merged.counts,
                 site_mean=merged.site_mean, site_cnt=merged.site_cnt, unit_rec_off=merged.unit_rec_off,
                 split=np.array([(u, k, a, e) for u, v in merged.split_units.items() for k, a, e in v]))
    else:
        assert merged is None
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_rank_gather_of_pieces_equals_merge_in_one_process(tmp_path):
    import torch.multiprocessing as mp
    world = 2
    pb, rows = _world()
    shards, pieces, splits = mg.plan_pieces(pb.units, world)
    deep = 12
    assert list(splits) == [deep] and all(any(u == deep for u, _a, _e in p) for p in pieces)   # one piece per rank
    ctx = mp.spawn(_gather_worker, args=(world, free_port(), str(tmp_path)), nprocs=world, join=False)
    while not ctx.join():
        pass
    assert all(not p.is_alive() for p in ctx.processes)          # joined: no rank left behind
    got = np.load(tmp_path / "merged.npz")
    # merge_shards in one process over the same hand-made parts
    shard = importlib.import_module("l-giremi_b200.shard")
    parts, split = [], []
    locs = [_local(shard, pb, rows, k, world)[0] for k in range(world)]
    for run in locs:
        r = run.result
        if r is not None:
            parts.append((run.index, r.records, r.site_mean, r.site_cnt, r.unit_rec_off, r.counts))
    ps = sorted((a, rec, tab) for run in locs for _u, a, _e, rec, tab in run.pieces)
    owner = [run for run in locs if deep in run.means][0]
    split.append((deep, ps) + tuple(owner.means[deep]))
    want = mg.merge_shards(pb.units, pb.n_sites, parts, split)
    assert np.array_equal(got["records"], want.records) and np.array_equal(got["counts"], want.counts)
    assert np.array_equal(got["site_mean"].view(np.uint64), want.site_mean.view(np.uint64))
    assert np.array_equal(got["site_cnt"], want.site_cnt) and np.array_equal(got["unit_rec_off"], want.unit_rec_off)
    # ... which is the hand-made whole, in global order
    whole = np.concatenate([r[0] for r in rows])
    assert np.array_equal(got["records"][['i', 'j', 'mi']], whole[['i', 'j', 'mi']])
    assert np.array_equal(got["records"]['unit'], np.repeat(np.arange(pb.n_units), [len(r[0]) for r in rows]))
    assert np.array_equal(got["counts"], np.concatenate([r[1] for r in rows]))
    where = sorted(tuple(x) for x in got["split"].tolist())
    assert where == sorted((deep, k, a, e) for k in range(world) for u, a, e in pieces[k] if u == deep)


# --------------------------------------------------------------------------- on the device
def _unit(rng, S, R, cov, third=0.0):
    a, k = synth.draw_alleles(rng, 1, S, R, cov)
    al = a[0]
    if third:
        al[(rng.random(al.shape) < third) & (al != synth.NOCOV)] = synth.THIRD
    return enc.EncodedUnit(list(range(S)), [("mismatch", "snp", "het_snp")[int(x)] for x in k[0]],
                           synth.labels_from_alleles(al))


# deep unit (sites, reads, coverage) and the context settings that send it down each path
FORMS = {
    "four_blocks": ((550, 9000, 0.6), dict(dense_path=4, tile_path=1)),
    "nine_blocks": ((550, 9000, 0.6), dict(dense_path=9, tile_path=1)),
    "mid_depth_tiles": ((540, 2000, 0.5), dict(dense_path=4, tile_path=1)),
}
MODES = [L.MODE_ALL_PAIRS | L.MODE_EMIT_COUNTS, L.MODE_HET_ONLY | L.MODE_EMIT_COUNTS,
         L.MODE_HET_ONLY | L.MODE_SKIP_NONHET]


def _gpu_world(form):
    (S, R, cov), _cfg = FORMS[form]
    rng = np.random.default_rng(4711)
    eus = [_unit(rng, 40, 150, 0.5) for _ in range(6)] + [_unit(rng, S, R, cov)] + \
          [_unit(rng, 70, 1200, 0.5) for _ in range(3)] + [_unit(rng, 25, 90, 0.5) for _ in range(6)]
    return lg_mod.pack_units(eus)


def _configure(ctx, form):
    cfg = FORMS[form][1]
    if form == "mid_depth_tiles":
        ctx.set_dense_threshold(48, 1 << 30)   # nothing deep: the 540 x 2 000 unit takes the mid-depth tiles
    else:
        ctx.set_dense_threshold(48, 4096)      # lowered: the 9 000-read unit is deep, the 1 200-read ones are not
    ctx.set_dense_path(cfg["dense_path"])
    ctx.set_tile_path(cfg["tile_path"])


def _gpu_worker(rank, world, port, form):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lg = importlib.import_module("l-giremi_b200")
    shard = importlib.import_module("l-giremi_b200.shard")
    ctx = lg.Context(rank if lg.device_count() >= world else 0)
    _configure(ctx, form)
    pb = _gpu_world(form)
    deep = 6
    got = {}
    try:
        for mode in MODES:
            run = shard.local_run(pb, rank, world, 6, mode, ctx)
            assert len(run.pieces) == 1 and run.pieces[0][0] == deep    # one piece per rank
            got[mode] = shard.gather_run_to_rank0(pb, run, device="cpu")
        dist.barrier()
    finally:
        dist.destroy_process_group()
    if rank == 0:
        for mode in MODES:
            want = lg.mi_step_batched(pb, 6, mode, ctx=ctx, n_chunks=1)
            m = got[mode]
            assert list(m.split_units) == [deep] and sorted(k for k, _a, _e in m.split_units[deep]) == [0, 1]
            assert np.array_equal(m.records.view(np.uint8), want.records.view(np.uint8)), mode   # MI bits included
            assert np.array_equal(m.unit_rec_off, want.unit_rec_off)
            if mode & L.MODE_EMIT_COUNTS:
                assert np.array_equal(m.counts, want.counts), mode
            assert np.array_equal(m.site_mean.view(np.uint64), want.site_mean.view(np.uint64)), mode
            assert np.array_equal(m.site_cnt, want.site_cnt), mode
        if form != "mid_depth_tiles":
            assert want.n_dense_units == 1 and want.n_dense_four == (1 if form == "four_blocks" else 0)
        else:
            assert want.n_dense_units == 0
    ctx.close()


@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("form", list(FORMS))
def test_two_ranks_split_a_deep_unit_bit_for_bit(form):
    import torch.multiprocessing as mp
    pb = _gpu_world(form)
    _shards, pieces, splits = mg.plan_pieces(pb.units, 2)
    assert list(splits) == [6] and all(len(p) == 1 for p in pieces)
    mp.spawn(_gpu_worker, args=(2, free_port(), form), nprocs=2, join=True)


@pytest.mark.gpu
def test_ipc_errors(lg, gpu_ctx):
    """A piece imported into the process that exported it is LGMI_ERR_ARG; one exported before its run is
    LGMI_ERR_STATE from split_means_ipc."""
    rng = np.random.default_rng(406)
    pb = lg.pack_units([_unit(rng, 300, 500, 0.6)])
    pieces = [(0, 0, 128), (0, 128, 300)]
    b = mg.piece_batch(gpu_ctx, pb, pieces)
    other = mg.piece_batch(gpu_ctx, pb, pieces)
    try:
        mg.upload_piece_rows(b, pb, pieces)
        mg.upload_piece_rows(other, pb, pieces)
        early = [b.export_piece(0), b.export_piece(1)]
        with pytest.raises(lg.LgmiError) as e:
            other.copy_planes_from_ipc(0, early[1], L.PieceIpc.from_buffer_copy(early[1]).plane_word, 4)
        assert e.value.code == -2 and "lgmi_batch_copy_planes" in str(e.value)
        other.copy_planes_from(0, b, 0, 4)         # (what the message points to works)
        with pytest.raises(lg.LgmiError) as e:
            lg.split_means_ipc(gpu_ctx, pb.site_flags, early)
        assert e.value.code == -4
        # after the run, the same pieces of this process give split_means' bits
        W = int(pb.units['row_words'][0])
        b.copy_planes_from(int(b.pb.units['plane_off'][0]) + 3 * 128 * W, b, int(b.pb.units['plane_off'][1]),
                           3 * 172 * W)
        b.run(6, lg.MODE_HET_ONLY)
        b.sync()
        late = [b.export_piece(0), b.export_piece(1)]
        with pytest.raises(lg.LgmiError) as e:    # a piece missing
            lg.split_means_ipc(gpu_ctx, pb.site_flags, late[:1])
        assert e.value.code == -2
        mean, cnt = lg.split_means_ipc(gpu_ctx, pb.site_flags, late)
        want_mean, want_cnt = lg.split_means(gpu_ctx, pb.site_flags, [(b, 0), (b, 1)])
        assert np.array_equal(mean.view(np.uint64), want_mean.view(np.uint64)) and np.array_equal(cnt, want_cnt)
        whole = lg.mi_step_batched(pb, 6, lg.MODE_HET_ONLY, ctx=gpu_ctx, n_chunks=1)
        assert np.array_equal(mean.view(np.uint64), whole.site_mean.view(np.uint64))
    finally:
        b.close()
        other.close()
