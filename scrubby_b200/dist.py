"""Multi-GPU driver for the depletion path: one process per GPU, torch.distributed for the plumbing.

SURVEY 8e: every FASTQ file is cut into `world` contiguous byte ranges (mate files independently -- the
reference filters each file on its own ids against the same set, cleaner.rs:236-254).  The only exchanges
are tiny or one-off:
    all_gather  per-shard '\\n' counts        -> each shard's starting line number (line phase mod 4)
    broadcast   file-level CRLF decision      (needletail decides on the FIRST record, i.e. on shard 0)
    broadcast   id-set table + key arena      (set built once on rank 0, replicated over NVLink by NCCL)
    all_reduce  report counters               (reads_in, reads_out)
    all_gather  output sizes                  -> each rank's write offset in the concatenated output
Outputs concatenated in rank order are byte-identical to the single-GPU output.

The compute calls go through `ops` (default: the C ABI via scrubby_b200.api, i.e. the GPU; there is no CPU
path in the product).  tests/test_dist_gloo.py passes a CPU stand-in built on the oracle to exercise this
file's host logic with the gloo backend at world_size 2.
"""
from __future__ import annotations

import os
import sys
from dataclasses import dataclass


@dataclass
class Shard:
    rank: int
    start: int      # first owned byte of the file
    own_len: int    # owned bytes [start, start + own_len)
    buf_len: int    # bytes uploaded: owned bytes + halo, clipped to the file
    is_first: bool
    is_last: bool


def plan_shards(n_bytes: int, world: int, halo: int = 1 << 20, align: int = 16) -> list[Shard]:
    """`world` contiguous ranges covering [0, n_bytes); cuts are multiples of `align` so that every shard
    buffer keeps the 16-byte alignment the kernels want when it is a view of one device buffer.
    A shard may be empty (tiny files); the last shard always ends at EOF and carries no halo.
    A shard whose halo would reach EOF owns the rest of the file and IS the last shard (the C ABI's contract: only the
    shard that holds EOF may apply the end-of-file rules -- a last record without a newline, a tail of blank lines --
    and a buffer that ends at EOF without being that shard would have to call a short tail a halo problem)."""
    assert world >= 1 and n_bytes >= 0
    assert halo > 0 or world == 1, "a record that starts exactly at a cut is owned by the shard before it: halo >= 1"
    per = -(-n_bytes // world)
    per = max(align, -(-per // align) * align)
    out, eof_seen = [], False
    for r in range(world):
        a = min(n_bytes, r * per)
        b = n_bytes if r == world - 1 else min(n_bytes, (r + 1) * per)
        if eof_seen:  # ranks after the one that reaches EOF own nothing
            out.append(Shard(r, n_bytes, 0, 0, False, False))
            continue
        if b + halo >= n_bytes:
            b = n_bytes
        is_last = b == n_bytes
        eof_seen = is_last
        end = n_bytes if is_last else min(n_bytes, b + halo)
        out.append(Shard(r, a, b - a, end - a, r == 0, is_last))
    return out


class GpuOps:
    """the product's compute: libscrubby_gpu.so on this rank's device"""

    def __init__(self, ctx):
        import torch

        from . import api

        self.torch, self.api, self.ctx = torch, api, ctx
        self.device = torch.device("cuda", ctx.device)

    def upload(self, host_bytes):
        t = self.torch.frombuffer(bytearray(host_bytes), dtype=self.torch.uint8) if len(host_bytes) else \
            self.torch.empty(0, dtype=self.torch.uint8)
        d = self.torch.zeros(len(host_bytes) + 16, dtype=self.torch.uint8, device=self.device)
        d[: len(host_bytes)].copy_(t)
        return d

    def count_newlines(self, d_buf, n):
        return self.api.count_newlines_dev(self.ctx, d_buf, n) if n else 0

    def first_line_crlf(self, d_buf, n):
        head = bytes(d_buf[: min(n, 1 << 16)].cpu().numpy())
        p = head.find(b"\n")
        if p < 0 and n > len(head):
            head = bytes(d_buf[:n].cpu().numpy())
            p = head.find(b"\n")
        return p > 0 and head[p - 1 : p] == b"\r"

    def clean_shard(self, ids, d_buf, sh: Shard, newlines_before, crlf, reverse, want_other):
        cap = 2 * sh.buf_len + 64
        d_out = self.torch.empty(cap, dtype=self.torch.uint8, device=self.device)
        d_oth = self.torch.empty(cap, dtype=self.torch.uint8, device=self.device) if want_other else None
        r = self.api.clean_fastq_shard_dev(self.ctx, ids, d_buf, sh.buf_len, sh.own_len, newlines_before,
                                           sh.is_first, sh.is_last, crlf, d_out, d_oth, reverse)
        written = bytes(d_out[: r.n_written].cpu().numpy())
        other = bytes(d_oth[: r.n_other].cpu().numpy()) if want_other else b""
        return written, other, r.reads_in, r.reads_out

    def new_set(self):
        return self.api.IdSet.empty(self.ctx)

    def ids_shard(self, probe, d_buf, sh: Shard, newlines_before, into):
        """ids of the shard's own records that are absent from `probe` (None: all) -> `into`; (records, picked)"""
        return self.api.fastq_ids_shard_dev(self.ctx, probe, d_buf, sh.buf_len, sh.own_len, newlines_before,
                                            sh.is_first, sh.is_last, into)

    def fasta_ids_shard(self, probe, d_buf, sh: Shard, into):
        """the same for a FASTA file (no line phase: a record starts at any '>' after a newline)"""
        return self.api.fasta_ids_shard_dev(self.ctx, probe, d_buf, sh.buf_len, sh.own_len, sh.is_first, sh.is_last, into)

    def set_ids(self, ids):
        return ids.sorted_ids()

    def set_from_ids(self, id_list):
        return self.api.IdSet.from_ids(self.ctx, id_list)

    def unite_sets(self, sets, dist):
        """the union of `sets` over ALL ranks, replicated on every rank, without leaving the device: every set's
        keys as an "id\\n" list (sgpu_idset_keys_dev), all-gathered (NCCL over NVLink), one set build from the
        concatenation (sgpu_idset_from_txt_dev).  Exact for FASTQ ids (no whitespace, valid UTF-8)."""
        torch = self.torch
        parts = [s.keys_dev() for s in sets]
        txt = torch.cat(parts) if parts else torch.empty(0, dtype=torch.uint8, device=self.device)
        world = dist.get_world_size() if dist is not None else 1
        if world > 1:
            sizes = [r[0] for r in _all_gather_ints(dist, [txt.numel()], world)]
            pad = torch.zeros(max(max(sizes), 16), dtype=torch.uint8, device=self.device)
            pad[: txt.numel()] = txt
            gathered = [torch.empty_like(pad) for _ in range(world)]
            dist.all_gather(gathered, pad)
            txt = torch.cat([g[:n] for g, n in zip(gathered, sizes)])
        return self.api.IdSet.from_txt(self.ctx, txt) if txt.numel() else self.api.IdSet.empty(self.ctx)

    def replicate_set(self, ids, dist, src: int = 0):
        """broadcast the table and the key arena of rank `src`'s set (NCCL over NVLink) and import them"""
        torch, api = self.torch, self.api
        rank = dist.get_rank()
        meta = torch.zeros(5, dtype=torch.int64, device=self.device)
        if rank == src:
            img = ids.image()
            meta = torch.tensor([img.table_bytes, img.arena_bytes, img.capacity, img.count, img.has_empty],
                                dtype=torch.int64, device=self.device)
        dist.broadcast(meta, src)
        tb, ab, cap, cnt, he = (int(x) for x in meta.tolist())
        table = torch.empty(max(tb, 16), dtype=torch.uint8, device=self.device)
        arena = torch.empty(max(ab, 16), dtype=torch.uint8, device=self.device)
        if rank == src:
            if tb:
                table[:tb].copy_(_as_tensor(torch, img.d_table, tb, self.device))
            if ab:
                arena[:ab].copy_(_as_tensor(torch, img.d_arena, ab, self.device))
        if tb:
            dist.broadcast(table, src)
        if ab:
            dist.broadcast(arena, src)
        if rank == src:
            return ids
        from . import _lib

        img = _lib.IdSetImage()
        img.d_table, img.table_bytes = table.data_ptr() if tb else None, tb
        img.d_arena, img.arena_bytes = arena.data_ptr() if ab else None, ab
        img.capacity, img.count, img.has_empty = cap, cnt, he
        torch.cuda.current_stream(self.device).synchronize()
        return api.IdSet.from_image(self.ctx, img)  # copies: `table` / `arena` may be dropped afterwards


class _DevMem:
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


def _as_tensor(torch, ptr, n, device):
    return torch.as_tensor(_DevMem(ptr, n), device=device)


@dataclass
class ShardedResult:
    written: bytes          # this rank's part of the output file
    other: bytes
    offset_written: int     # where this rank's part starts in the concatenated output
    offset_other: int
    total_written: int
    total_other: int
    reads_in: int           # allreduced: whole file
    reads_out: int
    crlf: bool


def clean_fastq_sharded(ops, ids, file_bytes, dist=None, reverse: bool = False, want_other: bool = False,
                        halo: int = 1 << 20, max_halo: int = 1 << 30) -> ShardedResult:
    """FastqCleaner::clean_reads (cleaner.rs:731-760) for ONE file across all ranks.  `file_bytes` is any
    sliceable view of the decompressed file (bytes, memoryview, numpy memmap ...); every rank touches only
    its own range + halo.  A record longer than the halo makes the owning shard report SGPU_ERR_HALO; all
    ranks then retry with a larger halo (collective decision, so nobody deadlocks)."""
    world = dist.get_world_size() if dist is not None else 1
    rank = dist.get_rank() if dist is not None else 0
    n = len(file_bytes)
    while True:
        sh = plan_shards(n, world, halo)[rank]
        d_buf = ops.upload(file_bytes[sh.start : sh.start + sh.buf_len])
        own_nl = ops.count_newlines(d_buf, sh.own_len)
        crlf = ops.first_line_crlf(d_buf, sh.buf_len) if rank == 0 else False
        counts = _all_gather_ints(dist, [own_nl, int(crlf)], world)
        newlines_before = sum(c[0] for c in counts[:rank])
        crlf = bool(counts[0][1])
        halo_short, failed = 0, None
        try:
            if sh.own_len == 0:
                w, o, rin, rout = b"", b"", 0, 0
            else:
                w, o, rin, rout = ops.clean_shard(ids, d_buf, sh, newlines_before, crlf, reverse, want_other)
        except Exception as e:  # SGPU_ERR_HALO == 21
            w, o, rin, rout = b"", b"", 0, 0
            if getattr(e, "status", None) == 21:
                halo_short = 1
            else:
                failed = e
        res = _all_gather_ints(dist, [halo_short, len(w), len(o), rin, rout, _status_of(failed)], world)
        _raise_collectively(res, 5, failed, rank)  # an error in one shard ends the run on EVERY rank (nobody is left waiting)
        if any(r[0] for r in res):
            if halo >= max_halo:
                raise RuntimeError("a record is longer than the maximum shard halo")
            halo = min(max_halo, halo * 8)
            continue
        return ShardedResult(w, o, sum(r[1] for r in res[:rank]), sum(r[2] for r in res[:rank]),
                             sum(r[1] for r in res), sum(r[2] for r in res), sum(r[3] for r in res),
                             sum(r[4] for r in res), crlf)


@dataclass
class ShardedDiff:
    reads_in: int       # allreduced over ranks and file pairs (utils.rs:250-285)
    reads_out: int
    difference: int
    diff_ids: list      # sorted unique ids of the input records missing from their output file (every rank)


def _ids_of_file_sharded(ops, file_bytes, dist, probe, collect, halo, max_halo, fasta=False):
    """one loop of ReadDifference::get_difference over one file, every rank on its own byte range; the set of the
    rank's ids goes to `collect`; returns the (records, picked) totals of this rank.  A record longer than the halo
    makes all ranks retry with a larger one.  FASTA shards need no newline counts."""
    world = dist.get_world_size() if dist is not None else 1
    rank = dist.get_rank() if dist is not None else 0
    n = len(file_bytes)
    while True:
        sh = plan_shards(n, world, halo)[rank]
        d_buf = ops.upload(file_bytes[sh.start : sh.start + sh.buf_len])
        if not fasta:
            own_nl = ops.count_newlines(d_buf, sh.own_len)
            counts = _all_gather_ints(dist, [own_nl], world)
            newlines_before = sum(c[0] for c in counts[:rank])
        halo_short, rec, picked, failed = 0, 0, 0, None
        scratch = ops.new_set()  # a retry must not leave ids of the failed attempt behind
        try:
            if sh.own_len and fasta:
                rec, picked = ops.fasta_ids_shard(probe, d_buf, sh, scratch)
            elif sh.own_len:
                rec, picked = ops.ids_shard(probe, d_buf, sh, newlines_before, scratch)
        except Exception as e:  # SGPU_ERR_HALO == 21
            if getattr(e, "status", None) == 21:
                halo_short = 1
            else:
                failed = e
        res = _all_gather_ints(dist, [halo_short, _status_of(failed)], world)
        _raise_collectively(res, 1, failed, rank)
        if any(r[0] for r in res):
            if halo >= max_halo:
                raise RuntimeError("a record is longer than the maximum shard halo")
            halo = min(max_halo, halo * 8)
            continue
        collect(scratch)
        return rec, picked


def diff_sharded(ops, pairs, dist=None, halo: int = 1 << 20, max_halo: int = 1 << 30, fasta: bool = False) -> ShardedDiff:
    """ReadDifference::get_difference (utils.rs:250-285) across all ranks (SURVEY 8e, config 5).  For every
    (input, output) file pair: each rank lists the ids of its byte range of the OUTPUT file, the lists are
    all-gathered into the replicated set O_i, each rank probes its byte range of the INPUT file against it;
    counters are summed over ranks, the absent ids are united (the reference keeps one global diff set, so mates
    with the same id appear once but count twice).  fasta=True: the files are FASTA (the caller knows it from byte 0)."""
    world = dist.get_world_size() if dist is not None else 1
    reads_in = reads_out = difference = 0
    on_device = hasattr(ops, "unite_sets")  # the product: id lists never leave the GPUs until the final TSV
    diff_local: list = []                   # ids (host stand-in) or per-file sets (device) of this rank
    for fin, fout in pairs:
        out_local: list = []
        keep = out_local.append if on_device else (lambda s: out_local.extend(ops.set_ids(s)))
        rec_out, _ = _ids_of_file_sharded(ops, fout, dist, None, keep, halo, max_halo, fasta)
        if on_device:
            o_set = ops.unite_sets(out_local, dist)
        else:
            gathered = [out_local]
            if world > 1:
                gathered = [None] * world
                dist.all_gather_object(gathered, out_local)
            o_set = ops.set_from_ids(sorted(set(x for part in gathered for x in part)))
        keep = diff_local.append if on_device else (lambda s: diff_local.extend(ops.set_ids(s)))
        rec_in, picked = _ids_of_file_sharded(ops, fin, dist, o_set, keep, halo, max_halo, fasta)
        reads_out += rec_out
        reads_in += rec_in
        difference += picked
    tot = _all_gather_ints(dist, [reads_in, reads_out, difference], world)
    if on_device:
        ids = ops.set_ids(ops.unite_sets(diff_local, dist))
    else:
        gathered = [diff_local]
        if world > 1:
            gathered = [None] * world
            dist.all_gather_object(gathered, diff_local)
        ids = sorted(set(x for part in gathered for x in part))
    return ShardedDiff(sum(t[0] for t in tot), sum(t[1] for t in tot), sum(t[2] for t in tot), ids)


class ShardError(RuntimeError):
    """another rank's shard failed: every rank leaves the collective together (the lowest failing rank holds the
    earliest record of the file, i.e. the error the reference would have stopped at)"""

    def __init__(self, rank: int, status: int):
        super().__init__(f"shard {rank} failed with status {status}")
        self.rank, self.status = rank, status


def _status_of(exc) -> int:
    if exc is None:
        return 0
    st = getattr(exc, "status", None)
    return int(st) if isinstance(st, int) and st > 0 else 1 << 20  # not a library status: still an error


def _raise_collectively(res, col: int, mine, rank: int):
    """res: the all-gathered rows; column `col` holds every rank's error status (0 = fine).  Raises on EVERY rank when
    any shard failed: the first failing rank re-raises its own exception (it carries the record index), the others a
    ShardError that names it."""
    bad = [(r, row[col]) for r, row in enumerate(res) if row[col]]
    if not bad:
        return
    first_rank, status = bad[0]
    if mine is not None and rank == first_rank:
        raise mine
    raise ShardError(first_rank, status)


def _all_gather_ints(dist, vals, world):
    """all_gather of a short list of non-negative ints (works on gloo and nccl)"""
    if dist is None or world == 1:
        return [list(vals)]
    import torch

    dev = "cpu"
    if dist.get_backend() == "nccl":
        dev = torch.device("cuda", torch.cuda.current_device())
    t = torch.tensor(vals, dtype=torch.int64, device=dev)
    out = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return [[int(x) for x in o.tolist()] for o in out]


# ----------------------------------------------------------------------------------------------------------------
# Device-resident data plane (round 2): nothing below goes through host `bytes`.  Inputs are device tensors holding this
# rank's byte range (+ halo) of every file, outputs stay in caller-owned device tensors; the exchanges are NCCL
# collectives on device tensors (bench.py times exactly these calls).
# ----------------------------------------------------------------------------------------------------------------
@dataclass
class DevShardResult:
    n_written: int          # bytes this rank produced (in its d_out / d_other)
    n_other: int
    offset_written: int     # where they start in the concatenated output (shards are concatenated in rank order)
    offset_other: int
    total_written: int
    total_other: int
    reads_in: int           # whole file (summed over ranks)
    reads_out: int
    crlf: bool
    one_pass: bool          # the speculative single pass was accepted on every rank (no newline count before it)
    path: int


def evidence_shard_len(total: int, world: int, align: int = 16) -> int:
    """bytes per rank when an evidence file is cut into `world` EQUAL byte ranges (the last one padded): equal sizes
    make the all-gather's output buffer a contiguous image of the file"""
    per = -(-total // world)
    return max(align, -(-per // align) * align)


def replicate_file_dev(d_shard, per: int, total: int, dist=None, out=None):
    """all-gather of the `world` equal byte ranges of a file (NCCL over NVLink): every rank ends up with the whole file
    in HBM, contiguous.  For a one-column id list this IS the replication of the depletion set in its most compact
    form (alignment.rs:60-82 then runs on every rank over the same bytes -- one global set, cleaner.rs:236-254)."""
    import torch

    world = dist.get_world_size() if dist is not None else 1
    if world == 1:
        return d_shard[:total]
    assert d_shard.numel() >= per
    if out is None:
        out = torch.empty(world * per + 16, dtype=torch.uint8, device=d_shard.device)
    dist.all_gather_into_tensor(out[: world * per], d_shard[:per])
    return out[:total]


class PeerFile:
    """The byte ranges of a file in SYMMETRIC memory (torch.distributed._symmetric_memory): every rank's range is mapped
    into every other rank's address space over NVLink / NVSwitch, so a rank PULLS the ranges it needs with plain
    device-to-device copies -- no rendezvous per use.  An NCCL all-gather makes every rank wait until the slowest one
    has arrived (measured at 8 GPUs: 3.2 ms per step for a 0.8 ms transfer); ranges that are resident and immutable
    (the evidence shards, uploaded once) need no such hand-shake."""

    def __init__(self, per: int, dist, device):
        import torch
        import torch.distributed._symmetric_memory as symm

        self.per, self.world, self.rank = per, dist.get_world_size(), dist.get_rank()
        self.local = symm.empty(per + 16, dtype=torch.uint8, device=device)
        self.local.zero_()
        self.handle = symm.rendezvous(self.local, dist.group.WORLD)
        self.peers = [self.handle.get_buffer(r, (per,), torch.uint8) for r in range(self.world)]
        self.streams = [torch.cuda.Stream(device=device) for _ in range(min(4, self.world - 1))]
        self.ready = torch.cuda.Event()

    def publish(self, dist):
        """after the local range has been (re)written: every rank's range is final before anyone pulls"""
        import torch

        torch.cuda.current_stream().synchronize()
        dist.barrier()

    def pull(self, total: int, out):
        """the whole file, contiguous, in `out`: the other ranks' ranges are copied over NVLink (up to four peers at a
        time on side streams), the own range locally; the current stream continues when all of it has landed"""
        import torch

        cur = torch.cuda.current_stream()
        self.ready.record(cur)
        per = self.per
        for k in range(1, self.world):
            r = (self.rank + k) % self.world
            st = self.streams[(k - 1) % len(self.streams)]
            st.wait_event(self.ready)
            with torch.cuda.stream(st):
                out[r * per: (r + 1) * per].copy_(self.peers[r], non_blocking=True)
        out[self.rank * per: (self.rank + 1) * per].copy_(self.local[:per], non_blocking=True)
        for st in self.streams:
            cur.wait_stream(st)
        return out[:total]


def evidence_shard_with_halo(full, rank: int, world: int, per: int, halo: int = 1 << 16):
    """this rank's byte range of a line-oriented evidence file plus a halo (the start of the next range: a line of this
    range may end there), as (device tensor padded by 16 readable bytes, n, own_len, starts_line, is_last).  `full` is
    any 1-D uint8 tensor holding the file (each rank only touches its range, the halo and the byte before its range)."""
    import torch

    total = int(full.numel())
    a, b = min(total, rank * per), min(total, (rank + 1) * per)
    e = min(total, b + halo)
    buf = torch.zeros(e - a + 16, dtype=torch.uint8, device=full.device)
    buf[: e - a] = full[a:e]
    starts_line = a == 0 or int(full[a - 1]) == 10
    return buf, e - a, b - a, starts_line, b == total and e == total


class ShardedTxtSet:
    """Sharded build of the id set of a one-column id list (ReadAlignment::from_txt, alignment.rs:60-82) across the ranks.
    Replicating the evidence makes every rank parse, hash and partition ALL keys; here every rank does that for ITS byte
    range only (sgpu_idset_partition_txt_dev: slot images grouped by virtual page, in symmetric memory), one barrier says
    "lists final", and every rank assembles the whole table from all ranks' lists (sgpu_idset_assemble_dev) -- read
    straight out of the peers' memory over NVLink (`direct`), or pulled into local buffers first.  Only 16-byte images
    travel; the result is the same exact set on every rank (cleaner.rs:236-254: one global set).  The symmetric
    buffers are double-buffered: a rank may start its next partition while a peer still reads the previous lists."""

    def __init__(self, api, ctx, dist, ev_total: int, per: int, device, direct: bool | None = None):
        import math

        import torch
        import torch.distributed._symmetric_memory as symm

        self.api, self.ctx, self.dist = api, ctx, dist
        self.world, self.rank = dist.get_world_size(), dist.get_rank()
        # measured on C4 (DESIGN.md 5): reading the peers' lists in place wins on two GPUs (3.5 vs 3.9 ms); from four on
        # a page's list on one peer is a few hundred bytes and the bulk pull is faster (4.4 vs 5.1 ms at N = 4, 5.9 vs
        # 8.5 ms at N = 8).  `direct` may be flipped between builds (bench.py times both).
        self.direct = (self.world <= 2) if direct is None else direct
        # virtual pages: the same on every rank; sized for lines of >= 8 bytes at ~410 keys (load 0.2) per page
        self.log2_v = max(8, int(math.ceil(math.log2(max(1.0, ev_total / 8 / 410)))))
        V = 1 << self.log2_v
        self.cap = per // 6 + 65536  # records per rank (lines of >= 6 bytes on average; else the replicated build)
        self.step = 0
        self.recs, self.vs, self.p_recs, self.p_vs = [], [], [], []
        for _ in range(2):
            r = symm.empty(self.cap * 16, dtype=torch.uint8, device=device)
            v = symm.empty(V + 2, dtype=torch.int64, device=device)
            hr, hv = symm.rendezvous(r, dist.group.WORLD), symm.rendezvous(v, dist.group.WORLD)
            self.recs.append(r)
            self.vs.append(v)
            self.p_recs.append([hr.get_buffer(q, (self.cap * 16,), torch.uint8) for q in range(self.world)])
            self.p_vs.append([hv.get_buffer(q, (V + 2,), torch.int64) for q in range(self.world)])
        self.l_vs = [torch.empty(V + 2, dtype=torch.int64, device=device) for _ in range(self.world)]
        self.device = device
        self.l_recs = None  # local copies of the peers' lists: allocated by the first pulled build
        self.streams = [torch.cuda.Stream(device=device) for _ in range(min(4, self.world - 1))]
        self.ready = torch.cuda.Event()

    def build(self, d_buf, n: int, own_len: int, starts_line: bool, is_last: bool, mark=None):
        """-> IdSet, or None on every rank when the evidence cannot take this path (decided collectively).
        `mark` (optional) is called between the exchange and the assembly (bench.py's phase boundary)."""
        import torch

        k = self.step & 1
        self.step += 1
        V = 1 << self.log2_v
        got = self.api.idset_partition_txt_dev(self.ctx, d_buf, n, own_len, starts_line, is_last, self.log2_v, self.recs[k],
                                               self.vs[k])
        if got is None:  # flag it for the others: they read it with the counts
            self.vs[k][V + 1] = 1
            self.vs[k][V] = 0
            torch.cuda.current_stream().synchronize()
        self.dist.barrier()  # every rank's lists are final
        cur = torch.cuda.current_stream()
        # the offset tables are small: always pulled (the page kernel looks two of them up per page and rank)
        for q in range(self.world):
            self.l_vs[q].copy_(self.p_vs[k][q], non_blocking=True)
        if self.direct:
            recs = self.p_recs[k]
        else:
            if self.l_recs is None:
                self.l_recs = [None if q == self.rank else torch.empty(self.cap * 16, dtype=torch.uint8, device=self.device)
                               for q in range(self.world)]
            tail = torch.stack([v[V] for v in self.l_vs]).tolist()
            self.ready.record(cur)
            for j in range(1, self.world):
                q = (self.rank + j) % self.world
                st = self.streams[(j - 1) % len(self.streams)]
                st.wait_event(self.ready)
                with torch.cuda.stream(st):
                    self.l_recs[q][: tail[q] * 16].copy_(self.p_recs[k][q][: tail[q] * 16], non_blocking=True)
            for st in self.streams:
                cur.wait_stream(st)
            recs = [self.recs[k] if q == self.rank else self.l_recs[q] for q in range(self.world)]
        if mark is not None:
            mark()
        return self.api.idset_assemble_dev(self.ctx, recs, self.l_vs, self.log2_v)


def _gather_rows(dist, vals, world, device):
    """all_gather of a short int64 row per rank, on the device the ranks compute on"""
    import torch

    if dist is None or world == 1:
        return [list(vals)]
    t = torch.tensor(vals, dtype=torch.int64, device=device)
    out = torch.empty(world * len(vals), dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(out, t)
    flat = out.tolist()
    return [flat[r * len(vals): (r + 1) * len(vals)] for r in range(world)]


def _clean_files_sharded(call, count_own_newlines, first_line_crlf, shards, dist, device, ShardFailure):
    """the one-pass protocol over several files; `call(f, newlines_before, crlf)` runs file f's shard of this rank
    (None, None = speculate), `count_own_newlines(f)` / `first_line_crlf(f)` serve the exact protocol"""
    from . import _lib

    world = dist.get_world_size() if dist is not None else 1
    rank = dist.get_rank() if dist is not None else 0
    W = 10  # integers per file in the exchange
    row, failures = [], {}
    for f, sh in enumerate(shards):
        st, r = 0, None
        if sh.own_len:
            try:
                r = call(f, 0 if sh.is_first else None, None)
                st = r.status
            except ShardFailure as e:
                st, r = e.status, None
                failures[f] = e
        if r is None or st:
            row += [st, 0, 0, 0, 0, 0, 0, 0, 0, int(bool(sh.own_len))]
        else:
            row += [0, r.path, r.own_newlines, r.lead_newlines, int(r.crlf), r.n_written, r.n_other, r.reads_in,
                    r.reads_out, 1]
    rows = _gather_rows(dist, row, world, device)
    results = []
    for f, sh in enumerate(shards):
        col = [rw[f * W: (f + 1) * W] for rw in rows]
        hard = [(q, c[0]) for q, c in enumerate(col) if c[0] not in (0, _lib.SGPU_ERR_PHASE_UNKNOWN)]
        if hard:  # a parse error / halo / capacity problem in one shard ends the run on EVERY rank
            if f in failures and hard[0][0] == rank:
                raise failures[f]
            raise ShardError(hard[0][0], hard[0][1])
        ok = col[0][4] == 0
        before = 0
        for q, c in enumerate(col):
            if not c[9]:
                continue  # owns nothing
            ok = ok and c[0] == 0 and c[1] == 1 and (q == 0 or (before + c[3]) % 4 == 0)
            before += c[2]
        if not ok and os.environ.get("SGPU_DIST_DEBUG") and rank == 0:
            sys.stderr.write(f"[dist] file {f}: one pass not accepted; rows (status, path, own_nl, lead_nl, crlf, n_w, n_o, "
                             f"reads_in, reads_out, owns) = {col}\n")
        if ok:
            results.append(DevShardResult(col[rank][5], col[rank][6], sum(c[5] for c in col[:rank]),
                                          sum(c[6] for c in col[:rank]), sum(c[5] for c in col), sum(c[6] for c in col),
                                          sum(c[7] for c in col), sum(c[8] for c in col), False, True, 1))
            continue
        # ---- exact protocol for this file: newline counts and shard 0's line ending first
        own_nl = count_own_newlines(f) if sh.own_len else 0
        crlf = int(first_line_crlf(f)) if (rank == 0 and sh.buf_len) else 0
        cnt = _gather_rows(dist, [own_nl, crlf], world, device)
        nb, crlf = sum(c[0] for c in cnt[:rank]), bool(cnt[0][1])
        st, r, exc = 0, None, None
        if sh.own_len:
            try:
                r = call(f, nb, crlf)
            except ShardFailure as e:
                st, exc = e.status, e
        fin = _gather_rows(dist, [st, r.n_written if r else 0, r.n_other if r else 0, r.reads_in if r else 0,
                                  r.reads_out if r else 0, r.path if r else 0], world, device)
        _raise_collectively(fin, 0, exc, rank)
        results.append(DevShardResult(fin[rank][1], fin[rank][2], sum(c[1] for c in fin[:rank]),
                                      sum(c[2] for c in fin[:rank]), sum(c[1] for c in fin), sum(c[2] for c in fin),
                                      sum(c[3] for c in fin), sum(c[4] for c in fin), crlf, False,
                                      max(c[5] for c in fin)))
    return results


def _crlf_of_head(head: bytes, fetch_all):
    p = head.find(b"\n")
    if p < 0:
        head = fetch_all()
        p = head.find(b"\n")
    return p > 0 and head[p - 1: p] == b"\r"


def clean_files_sharded_dev(api, ctx, ids, jobs, dist=None, reverse: bool = False):
    """FastqCleaner::clean_reads (cleaner.rs:731-760) for several files at once (the mate files of cleaner.rs:238-248),
    each cut into one byte range per rank.  jobs: [(d_buf, Shard, d_out, d_other_or_None), ...], all DEVICE tensors.

    ONE pass per file: every rank runs the single-pass kernel on its range with a speculated line phase
    (SGPU_NEWLINES_UNKNOWN), then ONE all-gather of a few integers per file carries the own-range newline counts that
    prove (or refute) every speculation, the file-level CRLF decision of shard 0, the output sizes (-> write offsets
    of the concatenation) and the read counters.  A refuted speculation, a non-canonical shard or a CRLF file takes the
    exact protocol: newline counts first, then the shard call with the exact phase (two passes over the range)."""
    import torch

    device = torch.device("cuda", ctx.device)

    def call(f, nb, crlf):
        d_buf, sh, d_out, d_oth = jobs[f]
        return api.clean_fastq_shard_dev(ctx, ids, d_buf, sh.buf_len, sh.own_len, nb, sh.is_first, sh.is_last, crlf,
                                         d_out, d_oth, reverse)

    def count(f):
        return api.count_newlines_dev(ctx, jobs[f][0], jobs[f][1].own_len)

    def crlf(f):
        d_buf, sh = jobs[f][0], jobs[f][1]
        return _crlf_of_head(bytes(d_buf[: min(sh.buf_len, 1 << 16)].cpu().numpy()),
                             lambda: bytes(d_buf[: sh.buf_len].cpu().numpy()))

    return _clean_files_sharded(call, count, crlf, [j[1] for j in jobs], dist, device, api.ScrubbyGpuError)


def clean_files_sharded_host(api, ctx, ids, jobs, dist=None, reverse: bool = False):
    """the same protocol on HOST buffers (pinned for full PCIe rate): jobs = [(h_buf, Shard, h_out, h_other_or_None)],
    torch CPU uint8 tensors; every shard goes through sgpu_clean_fastq_shard (chunked H2D / kernels / D2H overlapped
    inside the call).  The exchanges are the same few integers, on the device the rank computes on."""
    import torch

    device = torch.device("cuda", ctx.device)

    def call(f, nb, crlf):
        h_buf, sh, h_out, h_oth = jobs[f]
        return api.clean_fastq_shard_host(ctx, ids, h_buf, sh.buf_len, sh.own_len, nb, sh.is_first, sh.is_last, crlf,
                                          h_out, h_oth, reverse)

    def count(f):
        h_buf, sh = jobs[f][0], jobs[f][1]
        step = 1 << 28  # (bounded temporaries: the comparison makes a byte per byte)
        return sum(int((h_buf[a: min(sh.own_len, a + step)] == 10).sum()) for a in range(0, sh.own_len, step))

    def crlf(f):
        h_buf, sh = jobs[f][0], jobs[f][1]
        return _crlf_of_head(bytes(h_buf[: min(sh.buf_len, 1 << 16)].numpy()), lambda: bytes(h_buf[: sh.buf_len].numpy()))

    return _clean_files_sharded(call, count, crlf, [j[1] for j in jobs], dist, device, api.ScrubbyGpuError)


def _clean_fasta_files_sharded(call, shards, dist, device, ShardFailure):
    """the one-pass protocol of FASTA shards over several files.  `call(f, le_before)` runs file f's shard of this rank
    and returns a result with n_written, n_other, reads_in, reads_out and le_own (api.FastaShardResult).

    Every rank runs once, rank 0 with le_before = -1 and every other rank with 0 (LF); ONE all-gather carries status,
    le_own, output sizes and counters.  Let d be the first le_own != -1 in rank order.  No d, or d == 0 (LF): every
    shard is right.  d == 1 (CRLF) at rank q: the ranks before q wrote only records before the decision (LF, right);
    rank q runs again with -1 (unless q == 0, which already did), every rank after q with 1."""
    world = dist.get_world_size() if dist is not None else 1
    rank = dist.get_rank() if dist is not None else 0
    W = 7  # integers per file in the exchange
    row, mine, failures = [], {}, {}
    for f, sh in enumerate(shards):
        st, r = 0, None
        if sh.own_len:
            try:
                r = call(f, -1 if rank == 0 else 0)
            except ShardFailure as e:
                st, failures[f] = e.status, e
        mine[f] = r
        row += [st, r.le_own if r else -1, r.n_written if r else 0, r.n_other if r else 0, r.reads_in if r else 0,
                r.reads_out if r else 0, int(r is not None)]
    rows = _gather_rows(dist, row, world, device)
    results = []
    for f, sh in enumerate(shards):
        col = [rw[f * W: (f + 1) * W] for rw in rows]
        bad = [q for q, c in enumerate(col) if c[0]]
        if bad:  # a parse error / halo / capacity problem in one shard ends the run on EVERY rank
            q = bad[0]
            if f in failures and q == rank:
                e = failures[f]
                if 3 <= e.status <= 9:  # a parse error (FASTQ_INVALID_START .. FASTQ_HEADER): the index in the whole file
                    raise type(e)(e.status, e.index + sum(c[4] for c in col[:rank])) from e
                raise e
            raise ShardError(q, col[q][0])
        d = next((q for q, c in enumerate(col) if c[6] and c[1] != -1), None)
        crlf = d is not None and col[d][1] == 1
        if not crlf:
            results.append(DevShardResult(col[rank][2], col[rank][3], sum(c[2] for c in col[:rank]),
                                          sum(c[3] for c in col[:rank]), sum(c[2] for c in col), sum(c[3] for c in col),
                                          sum(c[4] for c in col), sum(c[5] for c in col), False, True, 3))
            continue
        # CRLF decided at rank d: rank d (unless it is rank 0) and every rank after it run again
        st, r, exc = 0, mine[f], None
        if col[rank][6] and rank >= d and rank > 0:
            try:
                r = call(f, -1 if rank == d else 1)
            except ShardFailure as e:
                st, r, exc = e.status, None, e
        fin = _gather_rows(dist, [st, r.n_written if r else 0, r.n_other if r else 0, r.reads_in if r else 0,
                                  r.reads_out if r else 0], world, device)
        _raise_collectively(fin, 0, exc, rank)
        results.append(DevShardResult(fin[rank][1], fin[rank][2], sum(c[1] for c in fin[:rank]),
                                      sum(c[2] for c in fin[:rank]), sum(c[1] for c in fin), sum(c[2] for c in fin),
                                      sum(c[3] for c in fin), sum(c[4] for c in fin), True,
                                      not any(c[6] for c in col[max(d, 1):]), 3))
    return results


def clean_fasta_files_sharded_dev(api, ctx, ids, jobs, dist=None, reverse: bool = False):
    """FastqCleaner::clean_reads over FASTA files (the caller knows the format from byte 0), each cut into one byte range
    per rank: jobs = [(d_buf, Shard, d_out, d_other_or_None), ...], all DEVICE tensors.  The one-pass protocol of
    _clean_fasta_files_sharded: one shard call and one all-gather per file, a second call on the ranks from the one
    that decides CRLF on."""
    import torch

    def call(f, le_before):
        d_buf, sh, d_out, d_oth = jobs[f]
        return api.clean_fasta_shard_dev(ctx, ids, d_buf, sh.buf_len, sh.own_len, sh.is_first, sh.is_last, le_before,
                                         d_out, d_oth, reverse)

    return _clean_fasta_files_sharded(call, [j[1] for j in jobs], dist, torch.device("cuda", ctx.device),
                                      api.ScrubbyGpuError)


def clean_fasta_files_sharded_host(api, ctx, ids, jobs, dist=None, reverse: bool = False):
    """the same on HOST buffers (pinned for full PCIe rate): jobs = [(h_buf, Shard, h_out, h_other_or_None)], torch CPU
    uint8 tensors; every shard goes through sgpu_clean_fasta_shard (chunked H2D / kernels / D2H inside the call)"""
    import torch

    def call(f, le_before):
        h_buf, sh, h_out, h_oth = jobs[f]
        return api.clean_fasta_shard_host(ctx, ids, h_buf, sh.buf_len, sh.own_len, sh.is_first, sh.is_last, le_before,
                                          h_out, h_oth, reverse)

    return _clean_fasta_files_sharded(call, [j[1] for j in jobs], dist, torch.device("cuda", ctx.device),
                                      api.ScrubbyGpuError)
