"""The FASTA shard contract (include/scrubby_gpu.h, sgpu_clean_fasta_shard_dev) on the CPU: a stand-in built on the
oracle produces each shard's records, and the shards chained the way the drivers chain them (le_before of shard k+1 =
le_before(k) when decided, else le_own(k)) must give the oracle's whole-file bytes, counters and error.  The same
stand-in serves the multi-GPU driver's FASTA protocol (scrubby_b200/dist.py) under gloo.  CPU only.

The stand-in runs the oracle on the shard's owned records with a sentinel record on each side: the next record start
stays in the slice (its newline is not the input's last byte, where the end-of-file rule would discard it), and a
first record emulates le_before (undecided: a header-only record, which decides nothing; LF / CRLF: a record that
decides).  The sentinels' bytes and counts are removed again."""
import os
import random
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import oracle as orc  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from scrubby_b200 import synth  # noqa: E402
from scrubby_b200.dist import Shard, ShardError, plan_shards  # noqa: E402
from test_oracle_differential import FASTA_CASES, rand_fasta  # noqa: E402

SGPU_ERR_HALO = 21
FRONT = {-1: (b">~front~\n", b">~front~\n\n"), 0: (b">~front~\nA\n", b">~front~\nA\n"),
         1: (b">~front~\r\nA\r\n", b">~front~\r\nA\r\n")}
END = b">~end~\nA\n"


class ShardFailure(Exception):
    def __init__(self, status, index=0):
        super().__init__(f"status {status} at record {index}")
        self.status, self.index = status, index


def record_starts(b: bytes, own_len: int, is_first: bool):
    """(owned starts, the first start after them or None)"""
    starts = [p + 1 for p in range(len(b) - 1) if b[p] == 10 and b[p + 1] == 62]
    owned = ([0] if is_first else []) + [p for p in starts if p <= own_len]
    nxt = next((p for p in starts if p > own_len), None)
    return owned, nxt


def le_own_of(seg: bytes, is_last: bool) -> int:
    """needletail's line-ending decision over the owned records `seg` (+ the next record's '>' when not last)"""
    chunks = seg.split(b"\n>")
    n = len(chunks) if is_last else len(chunks) - 1
    for idx in range(n):
        body = chunks[idx][1:] if idx == 0 else chunks[idx]
        pos = [i for i, c in enumerate(body) if c == 10]
        if is_last and idx == len(chunks) - 1:
            if pos and pos[-1] == len(body) - 1:
                pos = pos if len(pos) > 1 else []
            elif pos:
                pos.append(len(body))
        else:
            pos.append(len(body))
        if not pos:
            return -1
        if 10 in body[: pos[-1]]:
            f = body.find(b"\n")
            return int(f > 0 and body[f - 1] == 13)
    return -1


def shard_clean(b: bytes, own_len: int, is_first: bool, is_last: bool, le_before: int, ids, reverse: bool):
    """the FASTA shard contract on the CPU -> (status, error_record, written, other, reads_in, reads_out, le_own)"""
    if is_first and is_last and len(b) < 5:
        return 0, 0, b"", b"", 0, 0, -1
    owned, nxt = record_starts(b, own_len, is_first)
    if not owned:
        return 0, 0, b"", b"", 0, 0, -1
    if not is_last and nxt is None:
        raise ShardFailure(SGPU_ERR_HALO)
    seg = b[owned[0]:] if is_last else b[owned[0]: nxt]
    front_in, front_out = (b"", b"") if is_first else FRONT[le_before]
    end = b"" if is_last else END
    r = orc.clean_fastq(front_in + seg + end, ids, reverse, raise_on_error=False)
    side = [r.written, r.other]
    k = 1 if reverse else 0  # the sentinel ids are not in the set
    n_sent = 0
    if front_in:
        assert side[k].startswith(front_out)
        side[k] = side[k][len(front_out):]
        n_sent += 1
    if end and not r.error:
        side[k] = side[k][: side[k].rfind(b">~end~")]
        n_sent += 1
    le_own = le_own_of(seg + (b"" if is_last else b">"), is_last) if not r.error else -2
    return (r.error, r.error_record - (1 if front_in else 0) if r.error else 0, side[0], side[1], r.reads_in - n_sent,
            r.reads_out - (0 if reverse else n_sent), le_own)


def shards_from_cuts(n: int, cuts, halo: int):
    """shards for cut offsets (sorted, inside (0, n)); a shard whose buffer would reach EOF owns the rest (plan_shards)"""
    out, a = [], 0
    for i, c in enumerate(list(cuts) + [n]):
        if c <= a:
            continue
        last = c == n or c + halo >= n
        b = n if last else c
        out.append((a, b - a, n - a if last else b + halo - a, a == 0, last))
        a = b
        if last:
            break
    if not out:
        out.append((0, n, n, True, True))
    return out


def run_chain(run, n: int, cuts, halo: int):
    """the shards in order, le_before chained -> (status, global error index, written, other, reads_in, reads_out).
    `run(start, own_len, buf_len, is_first, is_last, le_before)` serves one shard; SGPU_ERR_HALO doubles the halo."""
    while True:
        try:
            w = o = b""
            rin = rout = 0
            le = -1
            for a, own, blen, first, last in shards_from_cuts(n, cuts, halo):
                st, err, sw, so, ri, ro, lo = run(a, own, blen, first, last, -1 if first else le)
                w, o = w + sw, o + so
                if st:
                    return st, rin + err, w, o, rin + ri, rout + ro
                rin, rout = rin + ri, rout + ro
                if le < 0:
                    le = lo
            return 0, 0, w, o, rin, rout
        except ShardFailure as e:
            assert e.status == SGPU_ERR_HALO
            halo *= 2


def whole(buf: bytes, ids, reverse: bool):
    r = orc.clean_fastq(buf, ids, reverse, raise_on_error=False)
    return r.error, r.error_record if r.error else 0, r.written, r.other, r.reads_in, r.reads_out


def standin(buf, ids, reverse):
    return lambda a, own, blen, first, last, le: shard_clean(buf[a: a + blen], own, first, last, le, ids, reverse)


HAND = [
    b">a\n>b\r\nAC\r\n>c\nGG\n",                 # header-only first record: the line ending is decided by the second
    b">a\nAC\n>b\n>c\n>d\nTT\r\n>e\r\nA\r\n",     # header-only records around a cut
    b">a\nAC>\nGT\n>b\nT>T\n",                    # '>' inside sequence lines: not record starts
    b">a\r\nAC\r\n>b\r\nTT\r\n>c\r\nG\r\n",       # CRLF
    b">a\nAC\n>b\r\nTT\r\n>c\nG\n>d\r\nC",         # mixed, no final newline
    b">a\nAC\n>b\nTT\n\n\n\n",                    # a trailing blank tail
    b">a\nAC\n>b\n",                              # UnexpectedEnd at the last record
    b">a\nAC\n>b\nTT\n>\nGG\n>c\nA\n",            # an empty id (get_id error) in the middle
    b">a\nAC\n>b\nTT\n>\xff\nGG\n>c\nA\n",        # invalid UTF-8 id
    b">a\n>b\n>c\n>d\n>e\n>f\n>g\nA",             # no record decides until the last
]


def _sweep(buf, ids_list, halos=(1, 3, 8, 64)):
    ids = orc.OSet.from_ids(ids_list)
    for rev in (False, True):
        want = whole(buf, ids, rev)
        run = standin(buf, ids, rev)
        if len(buf) < 5:
            assert run_chain(run, len(buf), [], 1) == want
            continue
        for halo in halos:
            for c in range(1, len(buf)):
                assert run_chain(run, len(buf), [c], halo) == want, (buf, c, halo, rev)


def test_standin_two_shards_every_cut():
    for buf, ids, _, _, _ in FASTA_CASES:
        _sweep(buf, ids)
    for buf in HAND:
        _sweep(buf, [b"b", b"c"])


@pytest.mark.parametrize("seed", range(4))
def test_standin_random_files_many_shards(seed):
    rng = random.Random(4200 + seed)
    ids = [b"b", b"q3", b"x" * 16]
    oset = orc.OSet.from_ids(ids)
    for _ in range(60):
        buf = rand_fasta(rng, rng.randrange(1, 12))
        rev = rng.random() < 0.5
        want = whole(buf, oset, rev)
        run = standin(buf, oset, rev)
        if len(buf) < 5:
            continue
        for _ in range(8):
            k = rng.randrange(1, 8)
            cuts = sorted(rng.sample(range(1, len(buf)), min(k, len(buf) - 1)))
            assert run_chain(run, len(buf), cuts, rng.choice([1, 2, 5, 17])) == want, (buf, cuts)


def test_standin_decision_in_a_later_shard():
    """the first records are header-only (they decide nothing); CRLF is decided two shards later"""
    buf = b"".join(b">h%d\n" % i for i in range(20)) + b">x\r\nAC\r\n" + b"".join(b">t%d\nGG\n" % i for i in range(20))
    ids = orc.OSet.from_ids([b"h3", b"t5"])
    want = whole(buf, ids, False)
    assert b"\r\n" in want[2]
    run = standin(buf, ids, False)
    for cuts in ([40, 80], [10, 60, 90, 120], list(range(16, len(buf), 16))):
        assert run_chain(run, len(buf), cuts, 8) == want
    # the shard that holds the deciding record reports it, the shards before report nothing
    a = buf.index(b">x")
    assert shard_clean(buf[: a - 1 + 10], a - 1, True, False, -1, ids, False)[6] == -1
    assert shard_clean(buf[a - 4:], len(buf) - a + 4, False, True, -1, ids, False)[6] == 1
    # le_own does not depend on le_before
    assert shard_clean(buf[a - 4:], len(buf) - a + 4, False, True, 0, ids, False)[6] == 1


def test_standin_errors_are_local_and_ordered():
    buf = b"".join(b">r%d\nACGT\n" % i for i in range(50)) + b">\nGG\n" + b"".join(b">s%d\nA\n" % i for i in range(50))
    ids = orc.OSet.from_ids([])
    want = whole(buf, ids, False)
    assert want[:2] == (po.E_HEADER, 50)
    run = standin(buf, ids, False)
    for cuts in ([100], [100, 300, 400], [350, 420]):
        assert run_chain(run, len(buf), cuts, 16) == want


def test_standin_halo_too_small():
    buf = b">a\n" + b"A" * 500 + b"\n>b\nC\n" + b">c\nG\n" * 100
    with pytest.raises(ShardFailure) as e:
        shard_clean(buf[:100], 50, True, False, -1, orc.OSet.from_ids([]), False)
    assert e.value.status == SGPU_ERR_HALO


# ----------------------------------------------------------------------------------------------------- gloo driver
class _Res:
    def __init__(self, t):
        self.status, _, self.written, self.other, self.reads_in, self.reads_out, self.le_own = t
        self.n_written, self.n_other = len(self.written), len(self.other)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _spawn(target, world, *args):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=target, args=(r, world, port, q) + args) for r in range(world)]
    for p in ps:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(world))
    for p in ps:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


def _clean_worker(rank, world, port, q, files, ids_list, reverse, halo):
    from scrubby_b200.dist import _clean_fasta_files_sharded

    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        ids = orc.OSet.from_ids(ids_list)
        shards = [plan_shards(len(f), world, halo)[rank] for f in files]
        calls, last = [], {}

        def call(f, le_before):
            sh = shards[f]
            calls.append((f, le_before))
            t = shard_clean(files[f][sh.start: sh.start + sh.buf_len], sh.own_len, sh.is_first, sh.is_last, le_before,
                            ids, reverse)
            if t[0]:
                raise ShardFailure(t[0], t[1])
            last[f] = _Res(t)
            return last[f]

        try:
            rs = _clean_fasta_files_sharded(call, shards, dist, "cpu", ShardFailure)
            q.put((rank, "ok", [(last[f].written if f in last else b"", last[f].other if f in last else b"",
                                 r.offset_written, r.total_written, r.reads_in, r.reads_out, r.crlf, r.one_pass)
                                for f, r in enumerate(rs)], calls))
        except ShardFailure as e:
            q.put((rank, "mine", (e.status, e.index), calls))
        except ShardError as e:
            q.put((rank, "other", (e.rank, e.status), calls))
    finally:
        dist.destroy_process_group()


def _check_clean(res, files, ids_list, reverse):
    ids = orc.OSet.from_ids(ids_list)
    for f, fa in enumerate(files):
        want = whole(fa, ids, reverse)
        assert want[0] == 0
        assert b"".join(r[2][f][0] for r in res) == want[2]
        assert b"".join(r[2][f][1] for r in res) == want[3]
        off = 0
        for r in res:
            w, o, offset, total, rin, rout, crlf, one_pass = r[2][f]
            assert (offset, total, rin, rout) == (off, len(want[2]), want[4], want[5])
            off += len(w)


@pytest.mark.parametrize("world", [2, 3])
def test_dist_fasta_lf_one_pass(world):
    """LF files (wrapped and not): every rank runs once, one exchange"""
    files = [synth.gen_fasta(300, 1, wrap=60).numpy().tobytes(), synth.gen_fasta(300, 2).numpy().tobytes()]
    ids = [b"syn.%d" % i for i in range(0, 300, 3)]
    for rev in (False, True):
        res = _spawn(_clean_worker, world, files, ids, rev, 256)
        _check_clean(res, files, ids, rev)
        assert all(r[1] == "ok" and all(x[7] for x in r[2]) for r in res)
        assert all(len(r[3]) == 2 for r in res)


@pytest.mark.parametrize("world", [2, 3])
def test_dist_fasta_crlf_decided_at_rank0(world):
    fa = synth.gen_fasta(300, 1, wrap=50, crlf=True).numpy().tobytes()
    ids = [b"syn.%d" % i for i in range(0, 300, 4)]
    res = _spawn(_clean_worker, world, [fa], ids, False, 256)
    _check_clean(res, [fa], ids, False)
    assert all(r[2][0][6] for r in res)  # crlf
    assert res[0][3] == [(0, -1)] and all(r[3] == [(0, 0), (0, 1)] for r in res[1:])  # rank 0 runs once


@pytest.mark.parametrize("world", [2, 3])
def test_dist_fasta_crlf_decided_at_a_later_rank(world):
    """header-only records fill rank 0; the deciding CRLF record sits in rank 1: rank 0 is right after one run, rank 1
    runs again undecided, the ranks after it with CRLF"""
    tail = synth.gen_fasta(200, 1, crlf=True).numpy().tobytes()
    head = b"".join(b">h%d\n" % i for i in range(int(1.3 * len(tail) / (world - 1) / 7)))
    fa = head + tail
    n = len(fa)
    sh = plan_shards(n, world, 256)
    assert sh[1].start < len(head) + 10 < sh[1].start + sh[1].own_len
    ids = [b"h7", b"syn.3", b"syn.150"]
    res = _spawn(_clean_worker, world, [fa], ids, False, 256)
    _check_clean(res, [fa], ids, False)
    assert res[0][3] == [(0, -1)] and res[1][3] == [(0, 0), (0, -1)]
    assert all(r[3] == [(0, 0), (0, 1)] for r in res[2:])


def test_dist_fasta_halo_error_ends_every_rank():
    fa = b">a\n" + b"A" * 4000 + b"\n" + b">b\nCC\n" * 50
    res = _spawn(_clean_worker, 2, [fa], [], False, 64)
    assert res[0][1] == "mine" and res[0][2][0] == SGPU_ERR_HALO
    assert res[1][1] == "other" and res[1][2] == (0, SGPU_ERR_HALO)


@pytest.mark.parametrize("world", [2, 3])
def test_dist_fasta_parse_error_ends_every_rank(world):
    """an empty id in the last rank's range: that rank raises with the record index in the whole file, every other
    rank a ShardError naming it"""
    recs = [b">r%d\nACGT\n" % i for i in range(300)]
    recs[280] = b">\nACGT\n"
    fa = b"".join(recs)
    assert whole(fa, orc.OSet.from_ids([]), False)[:2] == (po.E_HEADER, 280)
    res = _spawn(_clean_worker, world, [fa], [], False, 64)
    q = world - 1
    assert res[q][1] == "mine" and res[q][2] == (po.E_HEADER, 280)
    assert all(r[1] == "other" and r[2] == (q, po.E_HEADER) for r in res[:q])


class FastaIdsOps:
    """CPU stand-in for GpuOps' FASTA ids pass (TEST ONLY)"""

    def upload(self, b):
        return bytes(b)

    def new_set(self):
        return set()

    def set_ids(self, s):
        return sorted(s)

    def set_from_ids(self, id_list):
        return set(id_list)

    def fasta_ids_shard(self, probe, buf, sh: Shard, into):
        t = shard_clean(buf, sh.own_len, sh.is_first, sh.is_last, -1, orc.OSet.from_ids([]), False)
        if t[0]:
            raise ShardFailure(t[0], t[1])
        rec = picked = 0
        for _, rid, *_ in po.fasta_records(t[2]) if t[2] else []:
            k = po.get_id(rid)
            rec += 1
            if probe is None or k not in probe:
                picked += 1
                into.add(k)
        return rec, picked


def _diff_worker(rank, world, port, q, pairs, halo):
    from scrubby_b200.dist import diff_sharded

    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        r = diff_sharded(FastaIdsOps(), pairs, dist, halo=halo, fasta=True)
        q.put((rank, r.reads_in, r.reads_out, r.difference, r.diff_ids))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_dist_fasta_diff_matches_unsharded(world):
    fa1 = synth.gen_fasta(400, 1, wrap=60).numpy().tobytes()
    fa2 = synth.gen_fasta(400, 2, crlf=True).numpy().tobytes()
    ids = orc.OSet.from_ids([b"syn.%d" % i for i in range(0, 400, 3)])
    pairs = [(fa1, orc.clean_fastq(fa1, ids).written), (fa2, orc.clean_fastq(fa2, ids).written)]
    want = orc.diff(pairs)
    res = _spawn(_diff_worker, world, pairs, 128)
    for r in res:
        assert r[1:4] == tuple(want[:3])
        assert r[4] == want[3].sorted_ids()
