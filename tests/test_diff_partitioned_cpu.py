"""The hash-partitioned diff (scrubby_b200/dist.py diff_partitioned) on the CPU under gloo, world 1, 2 and 3.

The compute calls are served by CPU stand-ins built on the oracle (the FASTQ and FASTA stand-ins of test_dist_gloo.py and
test_fasta_shards_cpu.py, plus route / probe-lines with a fixed owner function of their own); what is under test is the
driver: the collective halo retry and error agreement it shares with diff_sharded, the real _all_to_all_bytes exchange
(gloo all_to_all_single on CPU tensors), the owner sets, the counters and the merge of the partitions' sorted dumps.
Every result must equal the oracle's ReadDifference::get_difference and dist.diff_sharded on the same pairs."""
import hashlib
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from oracle import oracle as orc  # noqa: E402
from scrubby_b200 import synth  # noqa: E402
from scrubby_b200.dist import _all_to_all_bytes  # noqa: E402
from test_dist_gloo import OracleOps  # noqa: E402
from test_fasta_shards_cpu import FastaIdsOps  # noqa: E402


def owner(rid: bytes, n_parts: int) -> int:
    """a fixed owner function for the stand-in (the library's is route_owner in csrc/idset.cuh)"""
    return (int.from_bytes(hashlib.blake2b(rid, digest_size=8).digest(), "little") * n_parts) >> 64


class _InOrder(list):
    """collects the ids an ids pass picks, in file order"""

    add = list.append


def _route(ids, n_parts):
    parts = [b"".join(k + b"\n" for k in ids if owner(k, n_parts) == p) for p in range(n_parts)]
    flat = b"".join(parts)
    t = torch.frombuffer(bytearray(flat), dtype=torch.uint8) if flat else torch.empty(0, dtype=torch.uint8)
    return t, [len(p) for p in parts]


def _lines(t):
    return bytes(t.numpy()).split(b"\n")[:-1] if t.numel() else []


class _PartitionedMixin:
    """route / owner set / probe-lines of GpuOps on the CPU (TEST ONLY)"""

    def route_shard(self, buf, sh, newlines_before, n_parts):
        got = _InOrder()
        rec, _ = self.ids_shard(None, buf, sh, newlines_before, got)
        return (*_route(got, n_parts), rec)

    def fasta_route_shard(self, buf, sh, n_parts):
        got = _InOrder()
        rec, _ = self.fasta_ids_shard(None, buf, sh, got)
        return (*_route(got, n_parts), rec)

    def set_from_lines(self, t):
        return set(_lines(t))

    def probe_lines(self, probe, t, into):
        ids = _lines(t)
        absent = [k for k in ids if probe is None or k not in probe]
        into.update(absent)
        return len(ids), len(absent)

    def free_set(self, s):
        s.clear()


class FastqPartOps(_PartitionedMixin, OracleOps):
    pass


class FastaPartOps(_PartitionedMixin, FastaIdsOps):
    pass


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q, pairs, fasta, halo):
    from scrubby_b200.dist import ShardError, diff_partitioned, diff_sharded

    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        out = []
        for fn in (diff_partitioned, diff_sharded):
            ops = FastaPartOps() if fasta else FastqPartOps()
            try:
                r = fn(ops, pairs, dist, halo=halo, fasta=fasta)
                out.append(("ok", r.reads_in, r.reads_out, r.difference, r.diff_ids))
            except ShardError as e:
                out.append(("shard", e.rank, e.status))
            except Exception as e:  # the failing rank's own error
                out.append(("own", type(e).__name__, getattr(e, "code", getattr(e, "status", None)),
                            getattr(e, "index", None)))
        q.put((rank, out))
    finally:
        dist.destroy_process_group()


def _run(world, pairs, fasta=False, halo=4096):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_worker, args=(r, world, port, q, pairs, fasta, halo)) for r in range(world)]
    for p in ps:
        p.start()
    res = sorted(q.get(timeout=180) for _ in range(world))
    for p in ps:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


def _check(res, pairs):
    want = orc.diff(pairs)
    for rank, (part, shard) in res:
        assert part[0] == "ok" and shard[0] == "ok", (rank, part, shard)
        assert part[1:4] == tuple(want[:3]) == shard[1:4]
        assert part[4] == want[3].sorted_ids() == shard[4]


def _fastq_pairs(n, dup=0):
    """both mates (they share ids) against their clean outputs; `dup`: the output files repeat their first records"""
    ids = orc.set_from_txt(synth.gen_txt_ids(n).numpy().tobytes())
    pairs = []
    for mate in (1, 2):
        fq = synth.gen_fastq(n, mate, read_len=60).numpy().tobytes()
        w = orc.clean_fastq(fq, ids).written
        if dup:
            w = b"\n".join(w.split(b"\n")[: 4 * dup]) + b"\n" + w
        pairs.append((fq, w))
    return pairs


@pytest.mark.parametrize("world", [1, 2, 3])
def test_partitioned_diff_fastq(world):
    pairs = _fastq_pairs(1200, dup=40)
    want = orc.diff(pairs)
    assert 0 < want[2] < want[0] and want[1] > 2 * 40
    _check(_run(world, pairs), pairs)


@pytest.mark.parametrize("world", [1, 2, 3])
def test_partitioned_diff_fasta(world):
    fa1 = synth.gen_fasta(500, 1, wrap=60).numpy().tobytes()
    fa2 = synth.gen_fasta(500, 2, crlf=True).numpy().tobytes()
    ids = orc.OSet.from_ids([b"syn.%d" % i for i in range(0, 500, 3)])
    pairs = [(fa1, orc.clean_fastq(fa1, ids).written), (fa2, orc.clean_fastq(fa2, ids).written)]
    _check(_run(world, pairs, fasta=True, halo=128), pairs)


def test_partitioned_diff_empty_partitions():
    """more ranks than distinct ids: most owner sets and diff partitions are empty; duplicate ids count per record"""
    fin = b"".join(b"@r%d x\nACGT\n+\nIIII\n" % (i % 2) for i in range(8))
    fout = b"@r0\nACGT\n+\nIIII\n@r0\nACGT\n+\nIIII\n"
    pairs = [(fin, fout), (fin, b"")]
    want = orc.diff(pairs)
    assert want[:3] == (16, 2, 12)
    for world in (3,):
        _check(_run(world, pairs, halo=16), pairs)


def test_partitioned_diff_halo_retry():
    """records longer than the first halo: every rank retries with a larger one, the result is unchanged"""
    recs = [b"@long.%d x\n" % i + b"A" * (3000 + 37 * i) + b"\n+\n" + b"I" * (3000 + 37 * i) + b"\n" for i in range(40)]
    fin = b"".join(recs)
    fout = b"".join(recs[::3])
    pairs = [(fin, fout)]
    _check(_run(2, pairs, halo=64), pairs)


def test_partitioned_diff_error_ends_every_rank():
    """a header without an id in the last third of the input file: diff_partitioned ends every rank exactly as
    diff_sharded does -- the owning rank with its own error, the others with a ShardError naming it"""
    pairs = _fastq_pairs(1500)
    fin = bytearray(pairs[1][0])
    pos = fin.rfind(b"\n@syn.", 0, len(fin) - 2000)
    end = fin.index(b"\n", pos + 1)
    fin[pos + 2: end] = b" " * (end - pos - 2)  # "@    ": FASTQ_HEADER
    pairs[1] = (bytes(fin), pairs[1][1])
    res = _run(3, pairs)
    for rank, (part, shard) in res:
        assert part == shard, (rank, part, shard)
    assert [r[1][0][0] for r in res] == ["shard", "shard", "own"]
    assert res[0][1][0][1] == 2


def _a2a_worker(rank, world, port, q):
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        # rank r sends (r, d) repeated d + 1 times to rank d, nothing to rank r itself when r == 1
        parts = [bytes([rank, d]) * (d + 1) if not (rank == 1 and d == 1) else b"" for d in range(world)]
        flat = b"".join(parts)
        t = torch.frombuffer(bytearray(flat), dtype=torch.uint8)
        got = _all_to_all_bytes(dist, t, [len(p) for p in parts])
        q.put((rank, bytes(got.numpy())))
    finally:
        dist.destroy_process_group()


def test_all_to_all_bytes():
    world = 3
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_a2a_worker, args=(r, world, port, q)) for r in range(world)]
    for p in ps:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(world))
    for p in ps:
        p.join(timeout=60)
        assert p.exitcode == 0
    for d, got in res:
        assert got == b"".join(bytes([r, d]) * (d + 1) if not (r == 1 and d == 1) else b"" for r in range(world))
    t = torch.arange(10, dtype=torch.uint8)
    assert bytes(_all_to_all_bytes(None, t, [7]).numpy()) == bytes(range(7))  # no process group: a local copy
