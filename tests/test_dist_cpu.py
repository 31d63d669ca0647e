"""CPU tier (gloo, world_size 2): the multi-GPU host logic of the path -- slide-aligned sharding and the
all-gather of per-slide aggregates and names that `threshold.ShardedTable` runs -- reproduces the single-process
group table exactly.  The per-shard aggregates are produced here by the oracle's pandas-order Kahan mean (the
CUDA reduction is checked against the same oracle in the GPU tier)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from biscuit_b200 import dist as bdist
from oracle import synth, threshold_oracle as O


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _local_groups(df):
    codes, uniques = df["slide"].factorize()
    L = len(uniques)
    gp, cnt = O.kahan_group_mean(df["y_pred"].to_numpy(), codes, L)
    gu, _ = O.kahan_group_mean(df["uncertainty"].to_numpy(), codes, L)
    gt, _ = O.kahan_group_mean(df["y_true"].to_numpy().astype(np.float64), codes, L)
    first = np.array([np.flatnonzero(codes == g)[0] for g in range(L)], dtype=np.int64)
    return list(uniques), gp, gu, gt, cnt, first


def _worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        df = synth.tile_table(n_slides=11, tiles_per_slide=40, seed=21, ragged=True)
        counts = df.groupby("slide", sort=False).size().to_numpy()
        lo, hi = bdist.shard_bounds(counts, world)[rank]
        local = df.iloc[int(counts[:lo].sum()):int(counts[:hi].sum())].reset_index(drop=True)
        # "split": slide-aligned shards; "empty": rank 0 holds the whole table and the last rank an EMPTY shard
        for case, shard in (("split", local), ("empty", df if rank == 0 else df.iloc[0:0])):
            names, gp, gu, gt, cnt, first = _local_groups(shard)
            g, all_names, n_keys = bdist.all_gather_groups(names, (gp, gu, gt, cnt, first), len(shard), len(names),
                                                           np.float32)
            np.savez(os.path.join(out_dir, f"{case}{rank}.npz"), **g, names=np.array(all_names), n_keys=n_keys)
    finally:
        dist.destroy_process_group()


def test_shard_bounds_properties():
    rng = np.random.default_rng(0)
    for world in (1, 2, 4, 8):
        for _ in range(20):
            counts = rng.integers(1, 3000, rng.integers(world, 60))
            b = bdist.shard_bounds(counts, world)
            assert len(b) == world and b[0][0] == 0 and b[-1][1] == len(counts)
            assert all(b[i][1] == b[i + 1][0] for i in range(world - 1))       # contiguous, slide aligned
            assert all(lo <= hi for lo, hi in b)
            loads = [counts[lo:hi].sum() for lo, hi in b]
            assert max(loads) - counts.sum() / world <= counts.max()               # balanced within one slide
    # the TCGA-scale config: 1000 slides x 2000 tiles over 8 GPUs -> 125 slides each
    assert bdist.shard_bounds([2000] * 1000, 8) == [(125 * r, 125 * (r + 1)) for r in range(8)]


def test_all_gather_groups_exchange_world2(tmp_path):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    df = synth.tile_table(n_slides=11, tiles_per_slide=40, seed=21, ragged=True)
    names, gp, gu, gt, cnt, first = _local_groups(df)
    for case in ("split", "empty"):
        for r in range(world):
            g = np.load(tmp_path / f"{case}{r}.npz")
            assert np.array_equal(g["code"], np.arange(len(names)))
            assert np.array_equal(g["count"], cnt)
            assert g["y_pred"].tobytes() == gp.tobytes()            # bit-exact: slides never straddle ranks
            assert g["uncertainty"].tobytes() == gu.tobytes()
            assert np.array_equal(g["y_true"], gt.astype(np.uint8))
            assert list(g["names"]) == names and int(g["n_keys"]) == len(names)


def test_all_gather_groups_single_process():
    g, names, n_keys = bdist.all_gather_groups(
        ["a", "b", "c"], (np.float32([.1, np.nan, .3]), np.float32([.01, np.nan, .03]), [0.0, np.nan, 1.0], [3, 0, 2],
                          [0, -1, 5]), 6, 3, np.float32)
    assert list(g["code"]) == [0, 2] and list(g["y_true"]) == [0, 1]
    assert names == ["a", "b", "c"] and n_keys == 3


# ----------------------------------------------------------------------------------------------------------------
# byte-level collectives behind apply_sharded / detect_sharded (tensor all-gathers, no pickled objects)
# ----------------------------------------------------------------------------------------------------------------
def _bytes_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        df = synth.tile_table(n_slides=7, tiles_per_slide=30, seed=5, ragged=True)
        counts = df.groupby("slide", sort=False).size().to_numpy()
        lo, hi = bdist.shard_bounds(counts, world)[rank]
        r0, r1 = int(counts[:lo].sum()), int(counts[:hi].sum())
        local = df.iloc[r0:r1]
        if rank == world - 1:                               # the last rank contributes an EMPTY shard of names
            names = []
        else:
            names = list(local["slide"].unique()) + ["slide with spaces \u00e9"]
        nbuf, nlen = bdist.pack_names(names)
        meta = bdist.all_gather_meta([len(local), len(names), nbuf.shape[0]])
        assert meta.shape == (world, 3)
        tiles = bdist.pack_tiles(local["y_pred"].to_numpy(), local["uncertainty"].to_numpy(), local["y_true"].to_numpy().astype(np.uint8))
        parts = bdist.all_gather_bytes(tiles, [int(m[0]) * 9 for m in meta])
        cols = [bdist.unpack_tiles(part, int(m[0]), np.float32) for m, part in zip(meta, parts)]
        payload = np.concatenate([nlen.view(np.uint8), nbuf])
        nparts = bdist.all_gather_bytes(payload, [int(m[1]) * 4 + int(m[2]) for m in meta])
        all_names = []
        for m, part in zip(meta, nparts):
            L = int(m[1])
            all_names += bdist.unpack_names(part[L * 4:], part[:L * 4].copy().view(np.int32))
        np.savez(os.path.join(out_dir, f"b{rank}.npz"), y_pred=np.concatenate([c[0] for c in cols]),
                 unc=np.concatenate([c[1] for c in cols]), y_true=np.concatenate([c[2] for c in cols]),
                 names=np.array(all_names, dtype=object), meta=meta)
    finally:
        dist.destroy_process_group()


def test_byte_collectives_world2(tmp_path):
    world = 2
    mp.spawn(_bytes_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    df = synth.tile_table(n_slides=7, tiles_per_slide=30, seed=5, ragged=True)
    for r in range(world):
        g = np.load(tmp_path / f"b{r}.npz", allow_pickle=True)
        assert g["y_pred"].tobytes() == df["y_pred"].to_numpy().tobytes()          # rank order == table order
        assert g["unc"].tobytes() == df["uncertainty"].to_numpy().tobytes()
        assert np.array_equal(g["y_true"], df["y_true"].to_numpy().astype(np.uint8))
        assert int(g["meta"][:, 0].sum()) == len(df)
        assert g["names"][-1] == "slide with spaces \u00e9" and len(g["names"]) == int(g["meta"][:, 1].sum())


def test_byte_collectives_single_process():
    nbuf, nlen = bdist.pack_names(["a", "bc", ""])
    assert bdist.unpack_names(nbuf, nlen) == ["a", "bc", ""]
    assert bdist.all_gather_meta([3, 4]).tolist() == [[3, 4]]
    t = bdist.pack_tiles(np.float64([.5, .25]), np.float64([.1, .2]), np.uint8([1, 0]))
    assert t.shape[0] == 2 * 17
    yp, un, yt = bdist.unpack_tiles(bdist.all_gather_bytes(t, [t.shape[0]])[0], 2, np.float64)
    assert yp.tolist() == [.5, .25] and un.tolist() == [.1, .2] and yt.tolist() == [1, 0]


# ---- property tests of the host-side exchange helpers (hypothesis): the N > 1 path must be lossless byte for byte ----
from hypothesis import given, settings, strategies as st  # noqa: E402


@settings(max_examples=150, deadline=None)
@given(st.lists(st.integers(min_value=0, max_value=5000), min_size=0, max_size=80), st.integers(min_value=1, max_value=16))
def test_shard_bounds_partition_any_cohort(counts, world):
    """Any cohort (empty, fewer slides than ranks, empty slides) is split into `world` contiguous, slide-aligned,
    ordered ranges that cover it exactly; with more ranks than slides the surplus ranks get empty shards."""
    b = bdist.shard_bounds(counts, world)
    assert len(b) == world
    assert b[0][0] == 0 and b[-1][1] == len(counts)
    assert all(lo <= hi for lo, hi in b)
    assert all(b[i][1] == b[i + 1][0] for i in range(world - 1))
    if counts and sum(counts) > 0 and len(counts) >= world:
        loads = [sum(counts[lo:hi]) for lo, hi in b]
        assert max(loads) - sum(counts) / world <= max(counts)


@settings(max_examples=100, deadline=None)
@given(st.lists(st.text(min_size=0, max_size=12), min_size=0, max_size=40))
def test_names_round_trip(names):
    buf, lens = bdist.pack_names(names)
    assert buf.dtype == np.uint8 and lens.dtype == np.int32 and int(lens.sum()) == buf.size
    assert bdist.unpack_names(buf, lens) == [str(n) for n in names]


@settings(max_examples=100, deadline=None)
@given(st.integers(min_value=0, max_value=300), st.sampled_from([np.float32, np.float64]), st.integers(0, 2 ** 31 - 1))
def test_tile_triples_round_trip_bit_exact(n, dtype, seed):
    """(pred, unc, label) triples cross ranks as raw bytes: NaN payloads, denormals and -0.0 must survive."""
    rng = np.random.default_rng(seed)
    bits = rng.integers(0, 2 ** (8 * np.dtype(dtype).itemsize - 1), n, dtype=np.uint64)
    yp = bits.astype({4: np.uint32, 8: np.uint64}[np.dtype(dtype).itemsize]).view(dtype)
    un = rng.standard_normal(n).astype(dtype)
    yt = rng.integers(0, 2, n).astype(np.uint8)
    buf = bdist.pack_tiles(yp, un, yt)
    assert buf.size == n * (2 * np.dtype(dtype).itemsize + 1)
    a, b, c = bdist.unpack_tiles(buf, n, dtype)
    assert a.tobytes() == yp.tobytes() and b.tobytes() == un.tobytes() and c.tobytes() == yt.tobytes()


@settings(max_examples=100, deadline=None)
@given(st.integers(min_value=1, max_value=40), st.integers(0, 2 ** 31 - 1))
def test_group_messages_keep_first_appearance_order(L, seed):
    """pack_groups / unpack_groups: float32 means are exact in the float64 message, groups with no surviving tile drop
    out, and the survivors come back ordered by their first surviving ROW (the reference's first-appearance order)."""
    rng = np.random.default_rng(seed)
    counts = rng.integers(0, 5, L)
    first = np.where(counts > 0, rng.permutation(L * 3)[:L], -1)
    yp, un = rng.random(L).astype(np.float32), rng.random(L).astype(np.float32)
    yt = rng.integers(0, 2, L).astype(np.float64)
    msg = bdist.pack_groups(7, counts, first, 100, yp, un, yt)
    g = bdist.unpack_groups(msg, np.float32)
    alive = np.nonzero(counts > 0)[0]
    order = alive[np.argsort(first[alive], kind="stable")]
    assert list(g["code"]) == list(order + 7)
    assert g["y_pred"].tobytes() == yp[order].tobytes() and g["uncertainty"].tobytes() == un[order].tobytes()
    assert list(g["count"]) == list(counts[order]) and list(g["y_true"]) == list(yt[order].astype(np.uint8))
