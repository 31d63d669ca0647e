"""Multi-GPU sharding of the hot path: one process per GPU, tiles sharded by WHOLE slides, and all-gathers
of small per-rank messages (SURVEY.md 8e).

Why slide-aligned: the reference's slide means are row-order Kahan sums in the column dtype
(pandas `group_mean`, reference threshold.py:191-192); summing per-GPU partials would change the
rounding and can flip a threshold decision, so a slide is never split across ranks and every slide's
reduction stays local and bit-exact.  What crosses ranks (`threshold.ShardedTable`): the validation counts
and row counts (`all_gather_meta`), the per-slide aggregates and slide names (`all_gather_groups`: 52 B per
slide plus its name) and, only where a tile-level ROC is detected over the whole cohort, the per-tile
`(pred, unc, label)` triples (`pack_tiles`) -- over NCCL/NVLink (gloo in the CPU tests), latency-, not
bandwidth-bound for the group level.

`torch.distributed` is plumbing only; the arithmetic stays in libbiscuit_b200.so.
"""
from __future__ import annotations

import numpy as np

GROUP_FIELDS = ("code", "count", "first_row", "y_pred", "uncertainty", "y_true_mean")


def shard_bounds(tiles_per_slide, world_size: int):
    """Contiguous, slide-aligned partition of a cohort balanced by tile count.

    tiles_per_slide: tile counts in table order.  Returns [(slide_lo, slide_hi)] * world_size;
    rank r owns slides [lo, hi) -- greedy prefix split at the slide boundary closest to r/world of
    the tiles."""
    counts = np.asarray(tiles_per_slide, dtype=np.int64)
    n_slides = int(counts.shape[0])
    cum = np.concatenate([[0], np.cumsum(counts)])
    total = int(cum[-1])
    cuts = [0]
    for r in range(1, world_size):
        target = total * r / world_size
        j = int(np.searchsorted(cum, target, side="left"))
        if j > 0 and abs(cum[j - 1] - target) <= abs(cum[min(j, n_slides)] - target):
            j -= 1
        j = min(max(j, cuts[-1]), n_slides)
        cuts.append(j)
    cuts.append(n_slides)
    return [(cuts[r], cuts[r + 1]) for r in range(world_size)]


def pack_groups(code_offset, counts, first_rows, row_offset, y_pred, uncertainty, y_true_mean):
    """Local per-slide aggregates -> float64 [L, 6] message (float32 means are exact in float64)."""
    L = len(counts)
    msg = np.empty((L, len(GROUP_FIELDS)), dtype=np.float64)
    msg[:, 0] = np.arange(L) + code_offset
    msg[:, 1] = counts
    msg[:, 2] = np.where(np.asarray(first_rows) >= 0, np.asarray(first_rows) + row_offset, -1)
    msg[:, 3] = y_pred
    msg[:, 4] = uncertainty
    msg[:, 5] = y_true_mean
    return msg


# ----------------------------------------------------------------------------------------------------------------
# byte-level collectives (tensor all-gathers only: no pickled objects, so the exchange stays on NCCL / NVLink)
# ----------------------------------------------------------------------------------------------------------------
class NativeComm:
    """NCCL communicator owned by the C library (`bq_comm_init`, include/biscuit_b200.h): pass it as `group=` to
    `threshold.apply_sharded / detect_sharded` and the exchange step runs through the C ABI (`bq_allgather_bytes`) on
    the context's stream instead of torch.distributed -- the path a non-Python host drives.

    Rank 0 obtains `NativeComm.unique_id()` and ships the 128 bytes to the other ranks by any host-side channel."""

    def __init__(self, ctx, rank: int, world: int, unique_id: bytes):
        from . import _ffi
        if len(unique_id) != 128:
            raise ValueError("unique_id must be the 128 bytes of bq_comm_unique_id")
        self.ctx, self.rank, self.world = ctx, int(rank), int(world)
        buf = np.frombuffer(bytes(unique_id), dtype=np.uint8).copy()
        _ffi.check(ctx.handle, ctx.lib.bq_comm_init(ctx.handle, self.rank, self.world, _ffi.ptr(buf)), "bq_comm_init")

    @staticmethod
    def unique_id() -> bytes:
        from . import _ffi
        lib = _ffi.load_library()
        buf = np.zeros(128, np.uint8)
        rc = lib.bq_comm_unique_id(_ffi.ptr(buf))
        if rc != 0:
            raise _ffi.NativeLibraryError(f"bq_comm_unique_id failed (rc={rc}): NCCL unavailable")
        return buf.tobytes()

    def all_gather_fixed(self, buf: np.ndarray) -> np.ndarray:
        """uint8 [n] from every rank -> uint8 [world, n] in rank order"""
        from . import _ffi
        buf = np.ascontiguousarray(buf, dtype=np.uint8).reshape(-1)
        out = np.empty((self.world, buf.shape[0]), np.uint8)
        _ffi.check(self.ctx.handle, self.ctx.lib.bq_allgather_bytes(self.ctx.handle, _ffi.ptr(buf), buf.shape[0],
                                                                    _ffi.ptr(out)), "bq_allgather_bytes")
        return out

    def close(self):
        if getattr(self, "ctx", None) is not None:
            self.ctx.lib.bq_comm_destroy(self.ctx.handle)
            self.ctx = None


def _dist_state(group=None):
    if isinstance(group, NativeComm):
        return group, group.world, group.rank
    import torch.distributed as dist
    if not dist.is_available() or not dist.is_initialized():
        return None, 1, 0
    return dist, dist.get_world_size(group), dist.get_rank(group)


def _collective_device(dist, group, device):
    import torch
    return torch.device("cpu") if dist.get_backend(group) == "gloo" else torch.device(device if device is not None else "cuda")


def all_gather_meta(values, group=None, device=None):
    """int64 [k] per rank -> int64 [world, k] (one small all-gather: row counts, group counts, error codes ...)."""
    import torch
    dist, world, _ = _dist_state(group)
    v = np.asarray(values, dtype=np.int64).reshape(1, -1)
    if world == 1:
        return v
    if isinstance(group, NativeComm):
        return group.all_gather_fixed(v.view(np.uint8).reshape(-1)).copy().view(np.int64).reshape(world, v.shape[1])
    dev = _collective_device(dist, group, device)
    t = torch.from_numpy(v[0].copy()).to(dev)
    out = torch.empty(world * v.shape[1], dtype=torch.int64, device=dev)     # flat: gloo requires world * numel
    dist.all_gather_into_tensor(out, t, group=group)
    return out.cpu().numpy().reshape(world, v.shape[1])


def all_gather_bytes(buf, sizes, group=None, device=None):
    """Variable-length all-gather of raw bytes when every rank already knows all `sizes` (from `all_gather_meta`).
    -> list of uint8 arrays, one per rank, in rank order."""
    import torch
    dist, world, _ = _dist_state(group)
    buf = np.ascontiguousarray(buf).view(np.uint8).reshape(-1)
    if world == 1:
        return [buf]
    sizes = [int(x) for x in sizes]
    pad = max(max(sizes), 1)
    if isinstance(group, NativeComm):
        send = np.zeros(pad, np.uint8)
        send[: buf.shape[0]] = buf
        host = group.all_gather_fixed(send)
        return [host[r, : sizes[r]] for r in range(world)]
    dev = _collective_device(dist, group, device)
    t = torch.zeros(pad, dtype=torch.uint8, device=dev)
    if buf.shape[0]:
        t[: buf.shape[0]] = torch.from_numpy(buf).to(dev)
    out = torch.empty(world * pad, dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(out, t, group=group)
    host = out.cpu().numpy().reshape(world, pad)
    return [host[r, : sizes[r]] for r in range(world)]


def pack_names(names):
    """slide / patient names -> (uint8 buffer of the utf-8 bytes, int32 lengths): strings cross ranks as tensors"""
    enc = [str(x).encode("utf-8") for x in names]
    lens = np.asarray([len(e) for e in enc], dtype=np.int32)
    return np.frombuffer(b"".join(enc), dtype=np.uint8).copy(), lens


def unpack_names(buf, lens):
    out, o = [], 0
    raw = np.asarray(buf, dtype=np.uint8).tobytes()
    for n in np.asarray(lens, dtype=np.int64):
        out.append(raw[o:o + n].decode("utf-8"))
        o += int(n)
    return out


def pack_tiles(y_pred, uncertainty, y_true):
    """per-tile (pred, unc, label) triples -> bytes (2 * itemsize + 1 B per tile: 9 B for float32 tables)"""
    yp, un = np.ascontiguousarray(y_pred), np.ascontiguousarray(uncertainty)
    yt = np.ascontiguousarray(y_true, dtype=np.uint8)
    return np.concatenate([yp.view(np.uint8).reshape(-1), un.view(np.uint8).reshape(-1), yt])


def unpack_tiles(buf, n, dtype):
    isz = np.dtype(dtype).itemsize
    b = np.asarray(buf, dtype=np.uint8)
    yp = b[: n * isz].copy().view(dtype)
    un = b[n * isz: 2 * n * isz].copy().view(dtype)
    yt = b[2 * n * isz: 2 * n * isz + n].copy()
    return yp, un, yt


def unpack_groups(msg: np.ndarray, dtype):
    """-> dict of arrays for the surviving groups, ordered by first surviving row (first appearance)."""
    alive = msg[:, 1] > 0
    m = msg[alive]
    order = np.argsort(m[:, 2], kind="stable")
    m = m[order]
    return {"code": m[:, 0].astype(np.int64), "count": m[:, 1].astype(np.int64),
            "y_pred": m[:, 3].astype(dtype), "uncertainty": m[:, 4].astype(dtype),
            "y_true": m[:, 5].astype(np.uint8)}


def all_gather_groups(names, groups, n_rows, n_keys, dtype, group=None, device=None):
    """The exchange of the group level: every rank's per-group aggregates and group names -> the cohort's.

    names: this rank's group names in code order; groups: its `(y_pred, uncertainty, y_true_mean, count, first_row)`
    arrays, one entry per name (`first_row` counts from the start of the shard, -1 where no tile survived the filter);
    n_rows: the shard's row count; n_keys: its key count before the filter.  One meta all-gather (the sizes) and ONE
    payload all-gather (the aggregate records and the names, as bytes).
    -> (the surviving groups as `unpack_groups` returns them in `dtype`, every rank's names in rank order, the cohort's
    key count).  Every rank must call it, with an empty shard too (no names, empty arrays, n_rows 0)."""
    y_pred, uncertainty, y_true_mean, counts, first_rows = groups
    name_buf, name_len = pack_names(names)
    meta = all_gather_meta([n_rows, len(names), n_keys, name_buf.shape[0]], group=group, device=device)
    _, _, rank = _dist_state(group)
    msg = pack_groups(int(meta[:rank, 1].sum()), counts, first_rows, int(meta[:rank, 0].sum()),
                      y_pred, uncertainty, y_true_mean)
    payload = np.concatenate([msg.view(np.uint8).reshape(-1), name_len.view(np.uint8), name_buf])
    rec = msg.itemsize * len(GROUP_FIELDS)                  # bytes of one group's aggregates
    nrec = rec + name_len.itemsize                          # ... and its name length
    parts = all_gather_bytes(payload, [int(L) * nrec + int(nb) for _, L, _, nb in meta], group=group, device=device)
    msgs, all_names = [], []
    for (_, L, _, nb), part in zip(meta, parts):
        L, nb = int(L), int(nb)
        msgs.append(part[:L * rec].copy().view(np.float64).reshape(L, len(GROUP_FIELDS)))
        all_names += unpack_names(part[L * nrec:L * nrec + nb], part[L * rec:L * nrec].copy().view(np.int32))
    return unpack_groups(np.concatenate(msgs, axis=0), dtype), all_names, int(meta[:, 2].sum())
