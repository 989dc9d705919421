"""The hash-partitioned diff on the B200: the route entry points (sgpu_{fastq,fasta}_ids_route_shard_dev) against the ids
entry points and the oracle, sgpu_idset_probe_lines_dev against a Python computation, the whole partitioned algebra on
virtual ranks of one device against sgpu_diff, and dist.diff_partitioned under NCCL (nccl_diff_partitioned_check.py)."""
import functools
import os
import random

import pytest
import torch

from oracle import oracle as orc
from oracle import pyoracle as po
from scrubby_b200 import api, synth
from scrubby_b200.dist import plan_shards

pytestmark = pytest.mark.gpu

M64 = (1 << 64) - 1


@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def _dev(b: bytes):
    d = torch.zeros(len(b) + 16, dtype=torch.uint8, device="cuda")
    if b:
        d[: len(b)] = torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
    return d


# ---- the owner function of include/scrubby_gpu.h, restated (idset.cuh key_image + route_owner)
def _mix64(x):
    x ^= x >> 32
    x = (x * 0xD6E8FEB86659FD93) & M64
    x ^= x >> 32
    x = (x * 0xD6E8FEB86659FD93) & M64
    return x ^ (x >> 32)


def _home(k: bytes) -> int:
    if len(k) <= 15:
        a = len(k) | (int.from_bytes(k[:7], "little") << 8)
        b = int.from_bytes(k[7:15], "little")
        return _mix64(a ^ _mix64((b + 0x9E3779B97F4A7C15) & M64))
    h = 0x9E3779B97F4A7C15 ^ ((len(k) * 0xD6E8FEB86659FD93) & M64)
    i = 0
    while i + 8 <= len(k):
        h = ((h ^ int.from_bytes(k[i: i + 8], "little")) * 0xFF51AFD7ED558CCD) & M64
        h ^= h >> 29
        i += 8
    h = _mix64(((h ^ int.from_bytes(k[i:], "little")) * 0xC4CEB9FE1A85EC53) & M64)
    return _mix64(0x80 | (h & ~0xFF & M64))


def owner(k: bytes, n_parts: int) -> int:
    h = _home(k) ^ 0x2545F4914F6CDD1D
    h ^= h >> 30
    h = (h * 0xBF58476D1CE4E5B9) & M64
    h ^= h >> 27
    h = (h * 0x94D049BB133111EB) & M64
    h ^= h >> 31
    return (h * n_parts) >> 64


# ---- route vs ids on the same shards
@functools.lru_cache(maxsize=8)
def _file_ids(buf: bytes):
    """the ids of a file's records in file order (the oracle's readers)"""
    return [po.get_id(rec[1]) for rec in po.fastq_records(buf)]


def _shard_calls(ctx, buf, a, own, blen, first, last, n_parts):
    """(ids entry point, route entry point) on one shard: ("ok", records, set ids) / ("ok", records, parts) or
    ("err", status, index)"""
    fasta = buf[:1] == b">"
    d = _dev(buf[a: a + blen])
    nb = buf[:a].count(b"\n")
    into = api.IdSet.empty(ctx)
    try:
        if fasta:
            rec, _ = api.fasta_ids_shard_dev(ctx, None, d, blen, own, first, last, into)
        else:
            rec, _ = api.fastq_ids_shard_dev(ctx, None, d, blen, own, nb, first, last, into)
        ids = ("ok", rec, into.sorted_ids())
    except api.ScrubbyGpuError as e:
        ids = ("err", e.status, e.index)
    try:
        if fasta:
            r = api.fasta_ids_route_shard_dev(ctx, d, blen, own, first, last, n_parts)
        else:
            r = api.fastq_ids_route_shard_dev(ctx, d, blen, own, nb, first, last, n_parts)
        flat = bytes(r.lines.cpu().numpy())
        parts, pos = [], 0
        for p in range(n_parts):
            chunk = flat[pos: pos + r.part_bytes[p]]
            pos += r.part_bytes[p]
            parts.append(chunk.split(b"\n")[:-1])
            assert len(parts[-1]) == r.part_lines[p] and (not chunk or chunk.endswith(b"\n"))
        assert pos == len(flat)
        route = ("ok", r.reads_in, parts)
    except api.ScrubbyGpuError as e:
        route = ("err", e.status, e.index)
    return ids, route


def _check_route(ctx, buf, shards, n_parts, seen):
    """every shard: route and ids agree on status / error record / records; the partitions, concatenated over the
    shards, are the file's ids split by owner in file order; `seen` (id -> partition) must stay consistent"""
    got = [[] for _ in range(n_parts)]
    for a, own, blen, first, last in shards:
        if own == 0:
            continue
        ids, route = _shard_calls(ctx, buf, a, own, blen, first, last, n_parts)
        assert ids[0] == route[0] and ids[1] == route[1], (ids[:2], route[:2], a, own, blen)
        if ids[0] == "err":
            assert ids[2] == route[2]
            return ids
        union = sorted(set(k for part in route[2] for k in part))
        assert union == ids[2]
        for p, part in enumerate(route[2]):
            got[p] += part
    want = _file_ids(buf)
    for p in range(n_parts):
        for k in got[p]:
            assert seen.setdefault((n_parts, k), p) == p, k
    for p in range(n_parts):
        assert got[p] == [k for k in want if seen[(n_parts, k)] == p]
    if n_parts == 1:
        assert got[0] == want
    return None


def _cut_shards(n, cut, halo):
    last = cut + halo >= n
    b = n if last else cut
    out = [(0, b, n if last else b + halo, True, last)]
    if not last:
        out.append((b, n - b, n - b, False, True))
    return out


def _small_cases():
    fq = synth.gen_fastq(12, 1, read_len=12).numpy().tobytes()
    crlf = fq.replace(b"\n", b"\r\n")
    plus_id = b"".join(b"@q%d extra\nACGTA\n+q%d\nIIIII\n" % (i, i) for i in range(10))
    no_final_nl = fq[:-1]
    ill = synth.gen_fastq_illumina(6, 1, read_len=8).numpy().tobytes()
    fa_wrap = synth.gen_fasta(10, 1, wrap=7, read_len=20).numpy().tobytes()
    fa_crlf = synth.gen_fasta(10, 2, crlf=True, read_len=12).numpy().tobytes()
    return {"canonical": fq, "crlf": crlf, "plus_id": plus_id, "no_final_newline": no_final_nl, "illumina": ill,
            "fasta_wrapped": fa_wrap, "fasta_crlf": fa_crlf}


@pytest.mark.parametrize("case", ["canonical", "crlf", "plus_id", "no_final_newline", "illumina", "fasta_wrapped",
                                  "fasta_crlf"])
def test_route_every_cut(ctx, case):
    buf = _small_cases()[case]
    seen = {}
    for n_parts in (1, 2, 3, 8):
        for halo in (4, 4096):
            for cut in range(1, len(buf)):
                # a 4-byte halo is short for most cuts: both entry points then report SGPU_ERR_HALO at the same record
                err = _check_route(ctx, buf, _cut_shards(len(buf), cut, halo), n_parts, seen)
                assert err is None or (halo == 4 and err[1] == 21), (cut, halo, err)
        for k, p in seen.items():
            if k[0] == n_parts:
                assert p == owner(k[1], n_parts), k  # the owner function stated in the header


def test_route_same_owner_across_files_and_formats(ctx):
    """the same ids in FASTQ, FASTA and CRLF files and at every shard count land in the same partition"""
    seen = {}
    n = 3000
    for buf in (synth.gen_fastq(n, 1, read_len=30).numpy().tobytes(), synth.gen_fastq(n, 2, read_len=30).numpy().tobytes(),
                synth.gen_fasta(n, 1, wrap=11, read_len=30).numpy().tobytes(),
                synth.gen_fastq(n, 1, read_len=30).numpy().tobytes().replace(b"\n", b"\r\n")):
        for world in (1, 3, 7):
            shards = [(s.start, s.own_len, s.buf_len, s.is_first, s.is_last) for s in plan_shards(len(buf), world, 512)]
            assert _check_route(ctx, buf, shards, 8, seen) is None
    assert len({k for k in seen}) == n


def test_route_errors_match_ids(ctx):
    """malformed input, a short halo and a first FASTQ shard of FASTA: the route entry points return the status and
    record index of the ids entry points"""
    fq = bytearray(synth.gen_fastq(200, 1, read_len=20).numpy().tobytes())
    pos = fq.index(b"\n@syn.150")
    bad_start = bytes(fq[: pos + 1]) + b"X" + bytes(fq[pos + 2:])
    bad_sep = bytes(fq[: pos + 1]) + bytes(fq[pos + 1:]).replace(b"\n+\n", b"\nx\n", 1)
    truncated = bytes(fq[:-30])
    longrec = bytes(fq[:pos + 1]) + b"@long\n" + b"A" * 5000 + b"\n+\n" + b"I" * 5000 + b"\n" + bytes(fq[pos + 1:])
    fa = synth.gen_fasta(50, 1).numpy().tobytes()
    seen = {}
    for buf in (bad_start, bad_sep, truncated):
        for cut in (0, len(buf) // 3, len(buf) - 100):
            shards = _cut_shards(len(buf), cut, 256) if cut else [(0, len(buf), len(buf), True, True)]
            assert _check_route(ctx, buf, shards, 3, seen) is not None
    # a record longer than the halo: SGPU_ERR_HALO from both
    ids, route = _shard_calls(ctx, longrec, 0, pos + 3, pos + 300, True, False, 4)
    assert ids == route and ids[:2] == ("err", 21)
    # a FASTA file cut into a FASTQ shard entry point: SGPU_ERR_FASTA_UNSUPPORTED from both
    d = _dev(fa)
    for fn in (lambda: api.fastq_ids_shard_dev(ctx, None, d, len(fa), len(fa) // 2, 0, True, False, None),
               lambda: api.fastq_ids_route_shard_dev(ctx, d, len(fa), len(fa) // 2, 0, True, False, 2)):
        with pytest.raises(api.ScrubbyGpuError) as e:
            fn()
        assert e.value.status == 15


@pytest.mark.parametrize("kind", ["fastq", "illumina", "fasta"])
def test_route_million_records(ctx, kind):
    n = 1_000_000
    if kind == "fastq":
        buf = synth.gen_fastq(n, 1).numpy().tobytes()
    elif kind == "illumina":
        buf = synth.gen_fastq_illumina(n, 1).numpy().tobytes()
    else:
        buf = synth.gen_fasta(n, 1, wrap=60).numpy().tobytes()
    seen = {}
    for n_parts in (3, 8):
        shards = [(s.start, s.own_len, s.buf_len, s.is_first, s.is_last) for s in plan_shards(len(buf), 3, 1 << 20)]
        assert _check_route(ctx, buf, shards, n_parts, seen) is None
    sample = random.Random(5).sample(sorted(k for k in seen if k[0] == 8), 20000)
    assert all(seen[k] == owner(k[1], 8) for k in sample)


def test_route_balance_ten_million_ids(ctx):
    """each of 8 partitions holds 1/8 of 10 M distinct ids within 1 %"""
    n = 10_000_000
    d = synth.gen_fastq(n, 1, device="cuda", read_len=16)
    nbytes = d.numel()
    buf = torch.zeros(nbytes + 16, dtype=torch.uint8, device="cuda")
    buf[:nbytes] = d
    del d
    r = api.fastq_ids_route_shard_dev(ctx, buf, nbytes, nbytes, 0, True, True, 8)
    assert r.reads_in == n and sum(r.part_lines) == n
    for c in r.part_lines:
        assert abs(c - n / 8) <= 0.01 * n / 8, r.part_lines


# ---- probe lines
def test_probe_lines(ctx):
    short = [b"a", b"b1", b"syn.7", b"x" * 15]
    long_ = [b"A00123:0456:H7ABCDEFG:1:1101:%05d:10000" % i for i in range(5)] + [b"y" * 16, b"z" * 300]
    member = set(short[::2] + long_[::2])
    probe = api.IdSet.from_ids(ctx, sorted(member))
    lines = short + long_ + short + [b"fresh", b"fresh", long_[1]]
    raw = b"".join(k + b"\n" for k in lines)
    for p, m in ((probe, member), (None, set())):
        into = api.IdSet.empty(ctx)
        got = api.idset_probe_lines_dev(ctx, p, _dev(raw), len(raw), into)
        absent = [k for k in lines if k not in m]
        assert got == (len(lines), len(absent))
        assert into.sorted_ids() == sorted(set(absent))
    # into NULL: counted only; an empty buffer: nothing
    assert api.idset_probe_lines_dev(ctx, probe, _dev(raw), len(raw), None) == (len(lines), len(lines) - sum(
        k in member for k in lines))
    into = api.IdSet.empty(ctx)
    assert api.idset_probe_lines_dev(ctx, probe, _dev(b""), 0, into) == (0, 0) and len(into) == 0
    # many lines (the bulk insert path) with duplicates
    many = [b"r%d" % (i % 70000) for i in range(200000)] + [b"long_read_name_%030d" % i for i in range(50000)]
    raw = b"".join(k + b"\n" for k in many)
    probe = api.IdSet.from_ids(ctx, [b"r%d" % i for i in range(0, 70000, 2)])
    into = api.IdSet.empty(ctx)
    got = api.idset_probe_lines_dev(ctx, probe, _dev(raw), len(raw), into)
    absent = [k for k in many if not (k.startswith(b"r") and int(k[1:]) % 2 == 0)]
    assert got == (len(many), len(absent)) and into.sorted_ids() == sorted(set(absent))


# ---- virtual ranks: the whole partitioned algebra on one device, without collectives
def _virtual_ranks(ctx, pairs, world, halo=1 << 16):
    """each "rank" routes its plan_shards range; destination r receives the parts for r in rank order; O_r, D_r,
    counters, merged sorted dumps -- what diff_partitioned computes with real collectives"""
    import heapq

    fasta = pairs[0][0][:1] == b">"

    def route(buf):
        recv = [[] for _ in range(world)]
        rec = 0
        for sh in plan_shards(len(buf), world, halo):
            if not sh.own_len:
                continue
            d = _dev(buf[sh.start: sh.start + sh.buf_len])
            if fasta:
                r = api.fasta_ids_route_shard_dev(ctx, d, sh.buf_len, sh.own_len, sh.is_first, sh.is_last, world)
            else:
                r = api.fastq_ids_route_shard_dev(ctx, d, sh.buf_len, sh.own_len, buf[: sh.start].count(b"\n"),
                                                  sh.is_first, sh.is_last, world)
            pos = 0
            for q in range(world):
                recv[q].append(r.lines[pos: pos + r.part_bytes[q]])
                pos += r.part_bytes[q]
            rec += r.reads_in
        return [torch.cat(x) if x else torch.empty(0, dtype=torch.uint8, device="cuda") for x in recv], rec

    d_sets = [api.IdSet.empty(ctx) for _ in range(world)]
    rin = rout = diff = 0
    for fin, fout in pairs:
        recv_o, rec_o = route(fout)
        o_sets = [api.IdSet.from_txt(ctx, t) if t.numel() else api.IdSet.empty(ctx) for t in recv_o]
        recv_i, _ = route(fin)
        for q in range(world):
            n_lines, absent = api.idset_probe_lines_dev(ctx, o_sets[q], recv_i[q], recv_i[q].numel(), d_sets[q])
            rin += n_lines
            diff += absent
        rout += rec_o
        for s in o_sets:
            s.free()
    dumps = [s.sorted_ids() for s in d_sets]
    for q in range(world):
        assert all(owner(k, world) == q for k in dumps[q][:200])
    return rin, rout, diff, list(heapq.merge(*dumps))


@pytest.mark.parametrize("kind", ["fastq", "fasta", "long_ids"])
def test_virtual_ranks_equal_diff(ctx, kind):
    n = 300_000
    gen = {"fastq": lambda m: synth.gen_fastq(n, m, read_len=60),
           "fasta": lambda m: synth.gen_fasta(n, m, wrap=50, read_len=60),
           "long_ids": lambda m: synth.gen_fastq_illumina(n, m, read_len=60)}[kind]
    files = [gen(m).numpy().tobytes() for m in (1, 2)]
    ids = _file_ids(files[0])[::3] if kind == "long_ids" else [b"syn.%d" % i for i in range(0, n, 3)]
    gs = api.IdSet.from_ids(ctx, ids)
    pairs = [(f, api.clean_fastq(ctx, gs, f).written) for f in files]
    want = api.diff(ctx, pairs)
    want = (want[0], want[1], want[2], want[3].sorted_ids())
    assert 0 < want[2] < want[0]
    for world in (2, 4, 8):
        assert _virtual_ranks(ctx, pairs, world) == want, world


def test_nccl_diff_partitioned():
    """dist.diff_partitioned under NCCL on min(device count, 8) GPUs, world 1 included (nccl_diff_partitioned_check.py)"""
    import socket
    import subprocess
    import sys

    n = min(torch.cuda.device_count(), 8)
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(root, "tests", "nccl_diff_partitioned_check.py")], capture_output=True, text=True,
                       timeout=900, cwd=root)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "nccl_diff_partitioned_check ok" in r.stdout and "MISMATCH" not in r.stdout
